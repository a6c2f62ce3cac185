"""Per-kernel times of the passes that move the reduced set (compaction, the sampler's emit and flag passes) on the
cfg-A workload of bench.py (592 pairs of N = 5000 at 95 % outliers, two lock-step chunks of 296), from torch.profiler
with CUDA activities, in a run of its own.  Bytes come from shapes: the compaction writes every edge once, so
sum(n_reduced) x bytes per edge; the flag pass reads at most the whole list per launch.

    python profiles/tools/edge_format_kernels.py [--debug edge_wide=1] [--out FILE]

--debug sets psulvsb_debug_set switches (edge_wide=1: 8-byte edges although 4-byte ones fit).  Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

KERNELS = ["compact_edges_kernel", "sample_flag_kernel", "sample_emit_kernel", "sample_bucket_kernel",
           "sample_draws_kernel", "engine_round_start_kernel"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=592)
    ap.add_argument("--debug", default="")
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    import psulvsb_b200  # noqa: F401
    from psulvsb_b200 import capi

    for kv in filter(None, args.debug.split(",")):
        k, v = kv.split("=")
        capi.debug_set(k, float(v))
    pairs = bench.make_pairs(0, args.batch)
    seeds = [bench.pair_seed(0, i) for i in range(args.batch)]
    probs = [capi.HostProblem(p["src"], p["dst"]) for p in pairs]
    params = capi.default_params(**bench.PARAM_KW)
    h = capi.Handle(0)
    h.upload(probs)
    for _ in range(2):  # warm-up: module loads, arenas
        sols = h.solve_resident(params, seeds)
    torch.cuda.synchronize()
    steps = 3
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            sols = h.solve_resident(params, seeds)
        torch.cuda.synchronize()
    per = {k: {"launches": 0, "us": 0.0, "names": set()} for k in KERNELS}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        for k in KERNELS:
            if k in ev.name:
                per[k]["launches"] += 1
                per[k]["us"] += ev.device_time
                per[k]["names"].add(ev.name.split("(")[0])
    n_red = sum(int(s.n_reduced) for s in sols)
    wide = "edge_wide=1" in args.debug.replace(" ", "")
    narrow_names = any("EdgeNarrow" in n for v in per.values() for n in v["names"])
    eb = 4 if narrow_names else 8
    out = {"batch": args.batch, "steps": steps, "debug": args.debug, "edge_bytes": eb, "forced_wide": wide,
           "sum_n_reduced_per_step": n_red,
           "gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                                 capture_output=True, text=True).stdout.strip()}
    for k, v in per.items():
        ms_step = v["us"] / 1e3 / steps
        rec = {"launches_per_step": v["launches"] / steps, "ms_per_step": round(ms_step, 4),
               "us_per_launch": round(v["us"] / max(v["launches"], 1), 2), "names": sorted(v["names"])}
        if k == "compact_edges_kernel" and ms_step > 0:
            rec["bytes_written_per_step"] = n_red * eb
            rec["write_TBps"] = round(n_red * eb / (ms_step * 1e-3) / 1e12, 3)
        if k == "sample_flag_kernel":
            rec["list_bytes_per_step"] = n_red * eb  # one round's launches read at most this much together
        out[k] = rec
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
