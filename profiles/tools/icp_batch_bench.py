"""Times batched ICP (psulvsb_icp_batch, csrc/k9_icp.cu) against a loop of single-pair psulvsb_icp calls on the same
inputs and the same stream, alternated in one run, on one GPU.

Workload: B pairs of the seeded synthetic surface (synth.make_surface; 8 base clouds), each target a distinct rigid
motion of its base, each source the base with noise (sigma = 0.1 mean spacings), refined from the truth moved by 2
degrees and 1 % of the extent; d = 3 mean spacings; point-to-plane uses the base's radius normals (r = 4 spacings)
rotated with the target.  The relative criteria are 0, so every pair runs exactly 30 iterations.  Lines: B = 64 and
592 pairs of 5 000 points and B = 16 pairs of 50 000, both modes.  Per line: pairs/s of the loop and of the batch,
ms per round (a call's 31 evaluations), and the launches (and memsets / copies) each issues.

With --parent-lib it also times the four single-pair lines of icp_bench.py (50 000 and 500 000 points, both modes)
through psulvsb_icp of that library (a build of the parent commit) and of this one, alternated, `--repeats` times
each: the batch-of-one route against the single-pair kernels it replaced.

CUDA events around back-to-back calls after a warm-up, at least `--min-seconds` of timed work per measurement; the
device name, power limit and SM clock are read in the same run.

    python profiles/tools/icp_batch_bench.py [--out profiles/r6_icp_batch_bench.json] [--parent-lib PATH]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import psulvsb_b200  # noqa: E402,F401
from icp_bench import smi, timed  # noqa: E402
from psulvsb_b200 import capi, features, stages, synth  # noqa: E402

ITERS = 30


def launches(p2l, B=1):
    """Operations one psulvsb_icp_batch call issues at 30 iterations (a psulvsb_icp call: B = 1 plus the same): pair
    table copy, bounds, count memset, count, scan, scatter, order, then per round correspond + step (and cross + step
    for point-to-point rounds with an update)."""
    rounds = 2 * (ITERS + 1) + (0 if p2l else 2 * ITERS)
    return 7 + rounds


def params(L, d, p2l):
    p = capi.IcpParams()
    L.psulvsb_icp_default_params(C.byref(p))
    p.max_correspondence_distance, p.point_to_plane = d, int(p2l)
    p.relative_fitness = p.relative_rmse = 0.0
    p.max_iterations = ITERS
    return p


def declare_icp(L):
    L.psulvsb_icp.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                              C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p]
    L.psulvsb_icp_workspace_bytes.argtypes = [C.c_int, C.c_int]
    L.psulvsb_icp_workspace_bytes.restype = C.c_ulonglong
    L.psulvsb_icp_default_params.argtypes = [C.c_void_p]
    L.psulvsb_last_error.restype = C.c_char_p
    return L


def make_batch(B, n, seed):
    """Device tensors of B pairs and their initial transforms; d."""
    import torch

    rng = np.random.default_rng(seed)
    bases = [synth.make_surface(n, s) for s in range(8)]
    sp = 2.0 / np.sqrt(n)                                   # mean spacing of n uniform points on [0, 2]^2 (about)
    nrm = [features.fpfh(P, 4 * sp, 8 * sp)[1] for P in bases]
    ds, dt, dn, R0s, t0s = [], [], [], [], []
    for b in range(B):
        P = bases[b % 8]
        R, _ = synth.random_rigid(rng)
        t = rng.normal(size=3)
        ax = rng.normal(size=3)
        ax /= np.linalg.norm(ax)
        K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
        a = np.deg2rad(2.0)
        R0 = (np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K) @ R
        t0 = t + 0.01 * np.linalg.norm(np.ptp(P, axis=1)) * rng.normal(size=3) / np.sqrt(3)
        ds.append(stages.to_device_points(P + rng.normal(0, 0.1 * sp, P.shape)))
        dt.append(stages.to_device_points(R @ P + t[:, None]))
        dn.append(stages.to_device_points(R @ nrm[b % 8]))
        R0s.append(R0)
        t0s.append(t0)
    torch.cuda.synchronize()
    return ds, dt, dn, R0s, t0s, 3.0 * sp


def batch_line(L, B, n, p2l, min_seconds, rounds):
    import torch

    ds, dt, dn, R0s, t0s, d = make_batch(B, n, 1000 * B + n)
    p = params(L, d, p2l)
    pairs = (capi.IcpPair * B)()
    Rc = [(C.c_double * 9)(*R.flatten(order="F")) for R in R0s]
    tc = [(C.c_double * 3)(*t) for t in t0s]
    for b in range(B):
        q = pairs[b]
        q.src, q.n_s, q.tgt, q.n_t, q.tgt_normals = ds[b].data_ptr(), n, dt[b].data_ptr(), n, dn[b].data_ptr()
        q.R0[:] = list(Rc[b])
        q.t0[:] = list(tc[b])
    work_b = torch.empty(L.psulvsb_icp_batch_workspace_bytes(pairs, B), dtype=torch.uint8, device="cuda")
    work_1 = torch.empty(L.psulvsb_icp_workspace_bytes(n, n), dtype=torch.uint8, device="cuda")
    res_b = torch.empty(B * C.sizeof(capi.IcpResult), dtype=torch.uint8, device="cuda")
    stream = stages._stream()

    def loop():
        for b in range(B):
            capi.check(L.psulvsb_icp(stream, ds[b].data_ptr(), n, dt[b].data_ptr(), n, dn[b].data_ptr(), C.byref(p),
                                     Rc[b], tc[b], work_1.data_ptr(),
                                     res_b.data_ptr() + b * C.sizeof(capi.IcpResult), None, None))

    def one():
        capi.check(L.psulvsb_icp_batch(stream, pairs, B, C.byref(p), work_b.data_ptr(), res_b.data_ptr(), None, None))

    # the two routes agree on every pair (bit for bit) before anything is timed
    loop()
    a = res_b.cpu().numpy().copy()
    one()
    assert np.array_equal(a, res_b.cpu().numpy()), "batch and per-pair results differ"
    res = (capi.IcpResult * B).from_buffer_copy(a.tobytes())
    ms_loop, ms_batch = [], []
    for _ in range(rounds):
        ms_loop.append(timed(loop, min_seconds)[0])
        ms_batch.append(timed(one, min_seconds)[0])
    ml, mb = float(np.median(ms_loop)), float(np.median(ms_batch))
    return {"B": B, "n": n, "mode": "point_to_plane" if p2l else "point_to_point", "d": d,
            "iterations": sorted({r.iterations for r in res}), "mean_fitness": float(np.mean([r.fitness for r in res])),
            "loop_ms": ms_loop, "batch_ms": ms_batch, "loop_pairs_per_s": B / (ml * 1e-3),
            "batch_pairs_per_s": B / (mb * 1e-3), "speedup": ml / mb, "loop_ms_per_round": ml / (ITERS + 1),
            "batch_ms_per_round": mb / (ITERS + 1), "loop_launches_per_call": B * launches(p2l),
            "batch_launches_per_call": launches(p2l)}


def single_lines(L, P, min_seconds, repeats):
    """icp_bench.py's four lines through psulvsb_icp of this build (L) and the parent's (P), alternated."""
    import torch

    out = []
    for n in (50000, 500000):
        tgt = synth.make_surface(n, 1)
        sp = 2.0 / np.sqrt(n)
        rng = np.random.default_rng(2)
        a = np.deg2rad(2.0)
        Rm = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
        shift = 0.01 * np.linalg.norm(np.ptp(tgt, axis=1)) * np.array([0.6, -0.5, 0.6])
        src = Rm @ tgt + shift[:, None] + rng.normal(0, 0.1 * sp, tgt.shape)
        d = 3.0 * sp
        ds, dt = stages.to_device_points(src), stages.to_device_points(tgt)
        _, dn = features.fpfh_device(dt, 4 * sp, 8 * sp)
        work = torch.empty(max(L.psulvsb_icp_workspace_bytes(n, n), P.psulvsb_icp_workspace_bytes(n, n)),
                           dtype=torch.uint8, device="cuda")
        res = {k: torch.empty(C.sizeof(capi.IcpResult), dtype=torch.uint8, device="cuda") for k in ("new", "parent")}
        R0 = (C.c_double * 9)(1, 0, 0, 0, 1, 0, 0, 0, 1)
        t0 = (C.c_double * 3)(0, 0, 0)
        for p2l in (False, True):
            p = params(L, d, p2l)

            def call(lib, key):
                rc = lib.psulvsb_icp(stages._stream(), ds.data_ptr(), n, dt.data_ptr(), n, dn.data_ptr(), C.byref(p),
                                     R0, t0, work.data_ptr(), res[key].data_ptr(), None, None)
                if rc:
                    raise RuntimeError(lib.psulvsb_last_error())

            call(L, "new")
            call(P, "parent")
            got = {k: capi.IcpResult.from_buffer_copy(v.cpu().numpy().tobytes()) for k, v in res.items()}
            same = all(np.array_equal(np.asarray(getattr(got["new"], f)), np.asarray(getattr(got["parent"], f)))
                       for f, _ in capi.IcpResult._fields_)           # field by field: the padding is not written
            ms = {"new": [], "parent": []}
            for _ in range(repeats):
                for key, lib in (("parent", P), ("new", L)):
                    ms[key].append(timed(lambda: call(lib, key), min_seconds)[0])
            mp, mn = float(np.mean(ms["parent"])), float(np.mean(ms["new"]))
            line = {"n": n, "mode": "point_to_plane" if p2l else "point_to_point", "results_identical": same,
                    "parent_ms": ms["parent"], "new_ms": ms["new"], "parent_mean_ms": mp, "new_mean_ms": mn,
                    "difference_pct": 100.0 * (mn - mp) / mp,
                    "parent_spread_pct": 100.0 * (max(ms["parent"]) - min(ms["parent"])) / mp,
                    "new_spread_pct": 100.0 * (max(ms["new"]) - min(ms["new"])) / mn}
            out.append(line)
            print(json.dumps(line), flush=True)
    return out


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_icp_batch_bench.json"))
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=2, help="alternations of loop and batch per line")
    ap.add_argument("--parent-lib", default=None, help="libpsulvsb_b200.so of the parent commit (single-pair lines)")
    ap.add_argument("--repeats", type=int, default=3, help="alternations of parent and new per single-pair line")
    ap.add_argument("--lines", default="64x5000,592x5000,16x50000")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("icp_batch_bench: no CUDA device (nothing is measured without one)")
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": smi("power.limit"),
           "sm_clock_max_mhz": smi("clocks.max.sm"), "sms": torch.cuda.get_device_properties(0).multi_processor_count,
           "iterations": ITERS, "batch_lines": [], "single_pair_lines": []}
    L = capi.lib()
    for spec in args.lines.split(","):
        B, n = (int(x) for x in spec.split("x"))
        for p2l in (False, True):
            line = batch_line(L, B, n, p2l, args.min_seconds, args.rounds)
            res["batch_lines"].append(line)
            print(json.dumps(line), flush=True)
    if args.parent_lib:
        P = declare_icp(C.CDLL(os.path.abspath(args.parent_lib)))
        res["single_pair_lines"] = single_lines(L, P, args.min_seconds, args.repeats)
    res["sm_clock_during_mhz"] = smi("clocks.sm")
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "power_limit_w", "sm_clock_during_mhz")}))


if __name__ == "__main__":
    main()
