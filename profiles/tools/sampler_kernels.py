"""Per-kernel times of the sampler (draw, bucket, emit and flag passes; the on-chip walk runs inside the bucket launch)
and of the whole of a cfg-A step
(bench.py's default line: 592 pairs of N = 5000 at 95 % outliers), from torch.profiler with CUDA activities, in a run of
its own.  Prints one JSON line: per sampler kernel the launches and milliseconds per step, and the whole step's kernel
time, so the sampler's share can be read off.

    python profiles/tools/sampler_kernels.py [--batch 592] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

KERNELS = ["sample_draws_kernel", "sample_bucket_kernel", "sample_emit_kernel", "sample_flag_kernel"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=592)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    import psulvsb_b200  # noqa: F401
    from psulvsb_b200 import capi

    pairs = bench.make_pairs(0, args.batch)
    seeds = [bench.pair_seed(0, i) for i in range(args.batch)]
    probs = [capi.HostProblem(p["src"], p["dst"]) for p in pairs]
    params = capi.default_params(**bench.PARAM_KW)
    h = capi.Handle(0)
    h.upload(probs)
    for _ in range(2):  # warm-up: module loads, arenas
        h.solve_resident(params, seeds)
    torch.cuda.synchronize()
    steps = 3
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            h.solve_resident(params, seeds)
        torch.cuda.synchronize()
    per = {k: {"launches": 0, "us": 0.0} for k in KERNELS}
    all_us = 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        all_us += ev.device_time
        for k in KERNELS:
            if k in ev.name:
                per[k]["launches"] += 1
                per[k]["us"] += ev.device_time
    out = {"batch": args.batch, "steps": steps,
           "gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                                  "--format=csv,noheader"], capture_output=True, text=True).stdout.strip(),
           "all_kernels_ms_per_step": round(all_us / 1e3 / steps, 3)}
    sampler_ms = 0.0
    for k, v in per.items():
        ms_step = v["us"] / 1e3 / steps
        sampler_ms += ms_step
        out[k] = {"launches_per_step": v["launches"] / steps, "ms_per_step": round(ms_step, 4),
                  "us_per_launch": round(v["us"] / max(v["launches"], 1), 2)}
    out["sampler_ms_per_step"] = round(sampler_ms, 3)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
