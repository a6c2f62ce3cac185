#!/usr/bin/env python
"""bench_stages.py -- kernel-level roofline measurements of the two FP32-pipe-bound stages on their
large configurations (BASELINE.json configs[2] and configs[4]); NOT the contract benchmark
(that is bench.py), these are the explanatory numbers DESIGN.md quotes.

  --case k1 : consistency mask, N correspondences (default 100 000, 99 % outliers), rows sharded
              across ranks with triangular balancing; only the per-row popcounts are all-gathered.
  --case k4 : hypothesis scoring sweep, H hypotheses x N correspondences (default 2^20 x 50 000),
              hypotheses sharded across ranks; global best = one 8-byte NCCL max-allreduce.

Timing: CUDA events on torch's current stream (the stage entry points are launched on it), W >= 3
warm-up launches, max over ranks.  One JSON line per case on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", default="k1", choices=["k1", "k4"])
    ap.add_argument("--n", type=int, default=0)
    ap.add_argument("--hyp", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--debug", action="append", default=[], metavar="NAME=VALUE",
                    help="psulvsb_debug_set switch (equivalent code paths, e.g. edge_wide=1); repeatable")
    args = ap.parse_args()

    import torch
    import torch.distributed as dist

    import psulvsb_b200  # noqa: F401
    from psulvsb_b200 import capi, sharding, stages, synth

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    L = capi.lib()
    for kv in args.debug:
        name, _, value = kv.partition("=")
        capi.debug_set(name, float(value))
    sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    def timed(fn):
        for _ in range(max(args.warmup, 3)):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        ev[0].record()
        for i in range(args.steps):
            fn()
            ev[i + 1].record()
        torch.cuda.synchronize()
        ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
        return sharding.max_over_ranks(float(np.mean(ms)), "cuda"), sharding.max_over_ranks(float(np.min(ms)), "cuda")

    def sm_clock():
        import subprocess
        try:
            out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=clocks.sm,clocks.max.sm",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True).stdout
            a, b = [float(x) for x in out.strip().split(",")]
            return a, b
        except Exception:
            return None, None

    if args.case == "k1":
        n = args.n or 100_000
        pair = synth.make_pair(n, 0.99, 4242, side=30.0)
        beta = 0.1
        (cs, cd), bound = stages.centre_and_bound(pair["src"], pair["dst"])
        d_src, d_dst = stages.to_device_points(pair["src"]), stages.to_device_points(pair["dst"])
        f_src, f_dst = stages.pack_points(d_src, cs), stages.pack_points(d_dst, cd)
        stride = ((n + 31) // 32 + 3) // 4 * 4
        ranges = [sharding.triangular_row_range(n, r, world) for r in range(world)]
        rb, re = ranges[rank]
        mask = torch.empty((re - rb, stride), dtype=torch.int32, device="cuda")  # this rank's rows only
        counts = torch.zeros(n, dtype=torch.int32, device="cuda")
        border = torch.zeros(1, dtype=torch.int64, device="cuda")
        mask_base = mask.data_ptr() - rb * stride * 4  # row i lives at base + i * stride words

        def run():
            capi.check(L.psulvsb_consistency_mask_rows(torch.cuda.current_stream().cuda_stream, f_src.data_ptr(),
                                                       f_dst.data_ptr(), d_src.data_ptr(), d_dst.data_ptr(), n, rb, re,
                                                       beta, bound, mask_base, stride, counts.data_ptr(),
                                                       border.data_ptr()))

        ms_mean, ms_min = timed(run)
        clk = sm_clock()
        border.zero_()
        run()
        torch.cuda.synchronize()
        allc = sharding.allgather_row_counts(counts, n, ranges)
        n_red = int(allc.to(torch.int64).sum().item())
        pairs_total = n * (n - 1) // 2
        if rank == 0:
            f = clk[0] or 1965.0
            peak = world * sms * 128 * f * 1e6 / 1e9
            ach = pairs_total * 16 / (ms_mean / 1e3) / 1e9
            mask_bytes = sum((e - b) * stride * 4 for b, e in ranges)
            print(json.dumps({
                "case": "k1 consistency mask", "n": n, "n_gpus": world, "pairs": pairs_total, "n_reduced": n_red,
                "borderline_pairs_rank0": int(border.item()), "ms_mean": ms_mean, "ms_min": ms_min,
                "pairs_per_s": pairs_total / (ms_mean / 1e3),
                "roofline": {"bound": "fp32-pipe", "achieved": ach, "peak": peak, "frac": ach / peak,
                             "unit": "Gslot/s (16 FP32-pipe issue slots per unordered pair)",
                             "peak_source": f"{world} x {sms} SMs x 128 lanes x {f:.0f} MHz (nvidia-smi during the run)"},
                "hbm_mask_write": {"bytes_written_incl_memset": 2 * mask_bytes,
                                   "achieved_gbs": 2 * mask_bytes / world / (ms_mean / 1e3) / 1e9,
                                   "peak_gbs": peaks.get("hbm_gbs", 6650.0)},
                "sharding": "triangular row blocks, all-gather of per-row popcounts only"}), flush=True)
    else:
        n = args.n or 50_000
        H = args.hyp
        pair = synth.make_pair(n, 0.95, 777)
        (cs, cd), bound = stages.centre_and_bound(pair["src"], pair["dst"])
        d_src, d_dst = stages.to_device_points(pair["src"]), stages.to_device_points(pair["dst"])
        f_src, f_dst = stages.pack_points(d_src, cs), stages.pack_points(d_dst, cd)
        hb, he = sharding.shard_range(H, rank, world)
        g = torch.Generator(device="cuda").manual_seed(99)  # same stream of hypotheses on every rank, sliced
        # random rotations near and far from the truth (q -> R), translations around the truth
        q = torch.randn((H, 4), generator=g, device="cuda", dtype=torch.float64)
        q = q / q.norm(dim=1, keepdim=True)
        w, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
        R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y + z * w), 2 * (x * z - y * w),
                         2 * (x * y - z * w), 1 - 2 * (x * x + z * z), 2 * (y * z + x * w),
                         2 * (x * z + y * w), 2 * (y * z - x * w), 1 - 2 * (x * x + y * y)], dim=1)  # column-major
        t = torch.randn((H, 3), generator=g, device="cuda", dtype=torch.float64)
        hyp = torch.cat([R, t], dim=1)
        truth = torch.from_numpy(np.concatenate([pair["R"].ravel(order="F"), pair["t"]])).cuda()
        hyp[H // 3] = truth  # one hypothesis is the ground truth: the argmax must find it
        hyp_local = hyp[hb:he].contiguous()
        tau = 0.04
        counts = torch.zeros(he - hb, dtype=torch.int32, device="cuda")
        best = torch.zeros(1, dtype=torch.int64, device="cuda")
        border = torch.zeros(1, dtype=torch.int64, device="cuda")
        csa = (__import__("ctypes").c_double * 3)(*[float(v) for v in cs])
        cda = (__import__("ctypes").c_double * 3)(*[float(v) for v in cd])

        def run():
            best.zero_()
            capi.check(L.psulvsb_score_batch(torch.cuda.current_stream().cuda_stream, f_src.data_ptr(), f_dst.data_ptr(),
                                             d_src.data_ptr(), d_dst.data_ptr(), n, hyp_local.data_ptr(), he - hb, hb,
                                             1.0, tau, bound, csa, cda, counts.data_ptr(), best.data_ptr(),
                                             border.data_ptr()))
            sharding.allreduce_best(best)  # 8 bytes over NVLink: the only collective of the sweep

        ms_mean, ms_min = timed(run)
        clk = sm_clock()
        cnt, hid = sharding.unpack_best(int(best.item()))
        if rank == 0:
            f = clk[0] or 1965.0
            units = H * n
            peak = world * sms * 128 * f * 1e6 / 1e9
            ach = units * 16 / (ms_mean / 1e3) / 1e9
            print(json.dumps({
                "case": "k4 hypothesis scoring sweep", "n": n, "hypotheses": H, "n_gpus": world, "units": units,
                "ms_mean": ms_mean, "ms_min": ms_min, "scores_per_s": units / (ms_mean / 1e3),
                "best": {"count": cnt, "hypothesis": hid, "expected_hypothesis": H // 3},
                "roofline": {"bound": "fp32-pipe", "achieved": ach, "peak": peak, "frac": ach / peak,
                             "unit": "Gslot/s (16 FP32-pipe issue slots per (hypothesis, point))",
                             "peak_source": f"{world} x {sms} SMs x 128 lanes x {f:.0f} MHz (nvidia-smi during the run)"},
                "hbm_hypothesis_stream_gbs": H * 96 / world / (ms_mean / 1e3) / 1e9,
                "sharding": "hypotheses sliced across ranks, one 8-byte max-allreduce of (count<<32 | ~id)"}),
                flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
