"""Times the ICP refinement (csrc/k9_icp.cu) on one GPU.  Workload: the seeded synthetic surface (synth.make_surface)
at N = 50 000 and 500 000 points as the target, the source a noisy copy (sigma = 0.1 mean spacings) rotated by 2
degrees and shifted by 1 % of the extent, d = 3 mean spacings, point-to-point and point-to-plane (radius normals of
the target, r = 4 spacings), from the identity.  The relative criteria are 0, so every call runs exactly 30 iterations.
CUDA events around back-to-back calls after a warm-up, at least `--min-seconds` of timed work per line; the device
name, power limit and SM clock are read in the same run.

Per line it also reports:
  * the mean candidates a query visits at the final transform (the 27 cells, each bucket once), from the grid's bucket
    sizes recomputed on the host with the kernel's hash, and the candidate-record bytes (32 each) the correspondence
    pass gathers per iteration;
  * per-kernel device time from torch.profiler (a separate, untimed pass), and the gather rate of k9_icp_correspond;
  * an early-converging call (criteria 1e-6, max_iterations 30) against one capped at the iterations it took: the
    difference is what the launches after convergence cost.

    python profiles/tools/icp_bench.py [--out profiles/r3_icp_bench.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import psulvsb_b200  # noqa: E402,F401
from psulvsb_b200 import capi, features, icp, stages, synth  # noqa: E402

ITERS = 30
M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def smi(query):
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=" + query, "--format=csv,noheader,nounits", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return ""


def timed(fn, min_seconds):
    import torch

    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    reps = 1
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= 1000.0 * min_seconds:
            return ms / reps, reps
        reps = max(reps * 2, int(reps * 1.2 * 1000.0 * min_seconds / max(ms, 1e-3)))


def bucket_of(cx, cy, cz, mask):
    """grid.cuh's hash on int64 cell arrays (uint64 arithmetic wraps as in the kernel)."""
    with np.errstate(over="ignore"):
        k = (cx.view(np.uint64) * np.uint64(0x9E3779B97F4A7C15)) ^ (cy.view(np.uint64) * np.uint64(0xC2B2AE3D27D4EB4F)) \
            ^ (cz.view(np.uint64) * np.uint64(0x165667B19E3779F9))
        k ^= k >> np.uint64(31)
        k *= np.uint64(0xBF58476D1CE4E5B9)
        k ^= k >> np.uint64(29)
    return (k & np.uint64(mask)).astype(np.int64)


def mean_candidates(src_t, tgt, d, valid=None):
    """Mean records a query at src_t (3 x n, transformed) visits: sum of its distinct buckets' sizes."""
    pts = tgt if valid is None else tgt[:, valid]
    nb = 1
    while nb < tgt.shape[1]:
        nb <<= 1
    inv_h = 1.0 / (d * (1.0 + 1e-6))
    corner = tgt.min(axis=1)
    cell = lambda P: np.floor((P - corner[:, None]) * inv_h).astype(np.int64)  # noqa: E731
    ct = cell(pts)
    size = np.bincount(bucket_of(ct[0], ct[1], ct[2], nb - 1), minlength=nb)
    cs = cell(src_t)
    buckets = np.stack([bucket_of(cs[0] + dx, cs[1] + dy, cs[2] + dz, nb - 1)
                        for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)])
    buckets.sort(axis=0)
    first = np.ones_like(buckets, dtype=bool)
    first[1:] = buckets[1:] != buckets[:-1]
    return float((size[buckets] * first).sum(axis=0).mean())


def kernel_times(fn, reps=5):
    """Device time per call of each kernel name (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        name = e.key
        for k in ("k9_icp_correspond", "k9_icp_cross", "k9_icp_step", "k9_icp_bounds", "k9_icp_grid", "k8_scan",
                  "k8_grid_scatter"):
            if k in name:
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                out[k] = out.get(k, 0.0) + t / 1000.0 / reps
                break
    return out


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_icp_bench.json"))
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--sizes", default="50000,500000")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("icp_bench: no CUDA device (nothing is measured without one)")
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": smi("power.limit"),
           "sm_clock_max_mhz": smi("clocks.max.sm"), "sms": torch.cuda.get_device_properties(0).multi_processor_count,
           "iterations": ITERS, "lines": []}
    L = capi.lib()
    for n in [int(x) for x in args.sizes.split(",")]:
        tgt = synth.make_surface(n, 1)
        sp = 2.0 / np.sqrt(n)                                   # mean spacing of n uniform points on [0, 2]^2 (about)
        rng = np.random.default_rng(2)
        a = np.deg2rad(2.0)
        Rm = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
        shift = 0.01 * np.linalg.norm(np.ptp(tgt, axis=1)) * np.array([0.6, -0.5, 0.6])
        src = Rm @ tgt + shift[:, None] + rng.normal(0, 0.1 * sp, tgt.shape)
        d = 3.0 * sp
        ds, dt = stages.to_device_points(src), stages.to_device_points(tgt)
        _, dn = features.fpfh_device(dt, 4 * sp, 8 * sp)
        normals = dn.cpu().numpy().T
        work = torch.empty(L.psulvsb_icp_workspace_bytes(n, n), dtype=torch.uint8, device="cuda")
        out = torch.empty(C.sizeof(capi.IcpResult), dtype=torch.uint8, device="cuda")
        R0 = (C.c_double * 9)(1, 0, 0, 0, 1, 0, 0, 0, 1)
        t0 = (C.c_double * 3)(0, 0, 0)
        for p2l in (False, True):
            def call(p):
                capi.check(L.psulvsb_icp(stages._stream(), ds.data_ptr(), n, dt.data_ptr(), n, dn.data_ptr(),
                                         C.byref(p), R0, t0, work.data_ptr(), out.data_ptr(), None, None))

            def params(rel, iters):
                p = capi.IcpParams()
                L.psulvsb_icp_default_params(C.byref(p))
                p.max_correspondence_distance, p.point_to_plane = d, int(p2l)
                p.relative_fitness = p.relative_rmse = rel
                p.max_iterations = iters
                return p

            fixed = params(0.0, ITERS)
            ms, reps = timed(lambda: call(fixed), args.min_seconds)
            r = icp.icp_device(ds, dt, np.eye(3), np.zeros(3), d, d_target_normals=dn, point_to_plane=p2l,
                               relative_fitness=0, relative_rmse=0, max_iterations=ITERS)
            valid = np.isfinite(normals).all(axis=0) if p2l else None
            cand = mean_candidates(src if r.iterations == 0 else (r.R @ src + r.t[:, None]), tgt, d, valid)
            kt = kernel_times(lambda: call(fixed))
            corr_ms = kt.get("k9_icp_correspond", float("nan")) / (ITERS + 1)
            gather = cand * 32.0 * n
            # early convergence: the default criteria, max 30, against the same call capped where it stopped
            early = params(1e-6, ITERS)
            e = icp.icp_device(ds, dt, np.eye(3), np.zeros(3), d, d_target_normals=dn, point_to_plane=p2l,
                               max_iterations=ITERS)
            ms_early, _ = timed(lambda: call(early), args.min_seconds)
            capped = params(1e-6, e.iterations)
            ms_capped, _ = timed(lambda: call(capped), args.min_seconds)
            line = {"n": n, "mode": "point_to_plane" if p2l else "point_to_point", "d": d, "ms_per_call": ms,
                    "reps": reps, "ms_per_iteration": ms / ITERS, "status": r.status, "iterations_run": r.iterations,
                    "fitness": r.fitness, "mean_candidates_per_query": cand,
                    "candidate_bytes_per_iteration": gather, "kernel_ms_per_call": kt,
                    "correspond_ms_per_round": corr_ms,
                    "correspond_gather_GBps": gather / (corr_ms * 1e-3) / 1e9 if corr_ms == corr_ms else None,
                    "early": {"iterations": e.iterations, "status": e.status, "ms_max30": ms_early,
                              "ms_capped": ms_capped, "idle_launch_ms": ms_early - ms_capped,
                              "idle_launches": (ITERS - e.iterations) * (2 if p2l else 4)}}
            res["lines"].append(line)
            print(json.dumps(line), flush=True)
    res["sm_clock_during_mhz"] = smi("clocks.sm")
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "power_limit_w", "sm_clock_during_mhz")}))


if __name__ == "__main__":
    main()
