"""Times generalized ICP (psulvsb_gicp / psulvsb_gicp_batch, csrc/k9_icp.cu) next to point-to-plane on the same inputs,
reports how the three modes converge, and checks single ICP calls against a build of the parent commit.

Workload (icp_bench.py's and icp_batch_bench.py's): the seeded synthetic surface (synth.make_surface), the source a
noisy copy (sigma = 0.1 mean spacings) moved by 2 degrees and 1 % of the extent, d = 3 mean spacings, radius normals
(r = 4 spacings) of both clouds.  Lines:
* single pairs, 50 000 and 500 000 points, 30 forced iterations (relative criteria 0): ms per call and per round of
  GICP and of point-to-plane, alternated `--rounds` times;
* batches, 592 x 5 000 and 16 x 50 000: pairs/s of one psulvsb_gicp_batch call and of one point-to-plane
  psulvsb_icp_batch call on the same pairs;
* convergence: per mode, default criteria (1e-6, 30 iterations), from starts of 2 and 5 degrees (1 % and 3 % of the
  extent): iterations, status, final rotation error (degrees) and translation error (fraction of the extent);
* with --parent-lib: icp_batch_bench.py's single-pair lines (psulvsb_icp, both ICP modes) through that library and
  this one, alternated, results compared field by field.

CUDA events around back-to-back calls after a warm-up, at least `--min-seconds` of timed work per measurement, medians
of the alternations; the device name, power limit and SM clock are read in the same run.

    python profiles/tools/gicp_bench.py [--out profiles/r8_gicp_bench.json] [--parent-lib PATH]
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
from icp_batch_bench import declare_icp, single_lines  # noqa: E402
from icp_bench import smi, timed  # noqa: E402
from psulvsb_b200 import capi, features, icp, stages, synth  # noqa: E402

ITERS = 30
EPS = 1e-3


def params(L, d, p2l, forced=True):
    p = capi.IcpParams()
    L.psulvsb_icp_default_params(C.byref(p))
    p.max_correspondence_distance, p.point_to_plane = d, int(p2l)
    if forced:
        p.relative_fitness = p.relative_rmse = 0.0
        p.max_iterations = ITERS
    return p


def moved(R, t, rng, deg, frac, ext):
    ax = rng.normal(size=3)
    ax /= np.linalg.norm(ax)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    a = np.deg2rad(deg)
    return (np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K) @ R, t + frac * ext * rng.normal(size=3) / np.sqrt(3)


def pair(n, seed, deg=2.0, frac=0.01):
    """Host clouds, radius normals, truth, start and d of one seeded pair."""
    rng = np.random.default_rng(seed)
    P = synth.make_surface(n, seed % 8)
    sp = 2.0 / np.sqrt(n)
    N = features.fpfh(P, 4 * sp, 8 * sp)[1]
    R, _ = synth.random_rigid(rng)
    t = rng.normal(size=3)
    ext = float(np.linalg.norm(np.ptp(P, axis=1)))
    R0, t0 = moved(R, t, rng, deg, frac, ext)
    src = P + rng.normal(0, 0.1 * sp, P.shape)
    return dict(src=src, tgt=R @ P + t[:, None], ns=N, nt=R @ N, R=R, t=t, R0=R0, t0=t0, d=3.0 * sp, ext=ext)


def single_line(L, n, min_seconds, rounds):
    import torch

    q = pair(n, 1)
    ds, dt = stages.to_device_points(q["src"]), stages.to_device_points(q["tgt"])
    dns, dnt = stages.to_device_points(q["ns"]), stages.to_device_points(q["nt"])
    work = torch.empty(L.psulvsb_icp_workspace_bytes(n, n), dtype=torch.uint8, device="cuda")
    res = torch.empty(C.sizeof(capi.IcpResult), dtype=torch.uint8, device="cuda")
    R0 = (C.c_double * 9)(*q["R0"].flatten(order="F"))
    t0 = (C.c_double * 3)(*q["t0"])
    stream = stages._stream()
    p2l, p2p = params(L, q["d"], True), params(L, q["d"], False)

    def plane():
        capi.check(L.psulvsb_icp(stream, ds.data_ptr(), n, dt.data_ptr(), n, dnt.data_ptr(), C.byref(p2l), R0, t0,
                                 work.data_ptr(), res.data_ptr(), None, None))

    def gicp():
        capi.check(L.psulvsb_gicp(stream, ds.data_ptr(), n, dns.data_ptr(), dt.data_ptr(), n, dnt.data_ptr(),
                                  C.byref(p2p), EPS, R0, t0, work.data_ptr(), res.data_ptr(), None, None))

    gicp()
    r = capi.IcpResult.from_buffer_copy(res.cpu().numpy().tobytes())
    ms = {"gicp": [], "point_to_plane": []}
    for _ in range(rounds):
        ms["point_to_plane"].append(timed(plane, min_seconds)[0])
        ms["gicp"].append(timed(gicp, min_seconds)[0])
    mg, mp = float(np.median(ms["gicp"])), float(np.median(ms["point_to_plane"]))
    return {"n": n, "d": q["d"], "iterations": r.iterations, "fitness": r.fitness, "gicp_ms": ms["gicp"],
            "point_to_plane_ms": ms["point_to_plane"], "gicp_ms_per_round": mg / (ITERS + 1),
            "point_to_plane_ms_per_round": mp / (ITERS + 1), "gicp_over_point_to_plane": mg / mp}


def batch_line(L, B, n, min_seconds, rounds):
    import torch

    qs = [pair(n, 100 * B + b % 8) for b in range(min(B, 8))]
    dev = [{k: stages.to_device_points(q[k]) for k in ("src", "tgt", "ns", "nt")} for q in qs]
    gp, ip = (capi.GicpPair * B)(), (capi.IcpPair * B)()
    for b in range(B):
        q, v = qs[b % len(qs)], dev[b % len(dev)]
        g, i = gp[b], ip[b]
        g.src = i.src = v["src"].data_ptr()
        g.tgt = i.tgt = v["tgt"].data_ptr()
        g.n_s = g.n_t = i.n_s = i.n_t = n
        g.src_normals = v["ns"].data_ptr()
        g.tgt_normals = i.tgt_normals = v["nt"].data_ptr()
        g.R0[:] = i.R0[:] = list(q["R0"].flatten(order="F"))
        g.t0[:] = i.t0[:] = list(q["t0"])
    d = qs[0]["d"]
    work = torch.empty(L.psulvsb_gicp_batch_workspace_bytes(gp, B), dtype=torch.uint8, device="cuda")
    res = torch.empty(B * C.sizeof(capi.IcpResult), dtype=torch.uint8, device="cuda")
    stream = stages._stream()
    p2l, p2p = params(L, d, True), params(L, d, False)

    def plane():
        capi.check(L.psulvsb_icp_batch(stream, ip, B, C.byref(p2l), work.data_ptr(), res.data_ptr(), None, None))

    def gicp():
        capi.check(L.psulvsb_gicp_batch(stream, gp, B, C.byref(p2p), EPS, work.data_ptr(), res.data_ptr(), None,
                                        None))

    gicp()
    r = (capi.IcpResult * B).from_buffer_copy(res.cpu().numpy().tobytes())
    ms = {"gicp": [], "point_to_plane": []}
    for _ in range(rounds):
        ms["point_to_plane"].append(timed(plane, min_seconds)[0])
        ms["gicp"].append(timed(gicp, min_seconds)[0])
    mg, mp = float(np.median(ms["gicp"])), float(np.median(ms["point_to_plane"]))
    return {"B": B, "n": n, "iterations": sorted({x.iterations for x in r}),
            "mean_fitness": float(np.mean([x.fitness for x in r])), "gicp_ms": ms["gicp"],
            "point_to_plane_ms": ms["point_to_plane"], "gicp_pairs_per_s": B / (mg * 1e-3),
            "point_to_plane_pairs_per_s": B / (mp * 1e-3), "gicp_over_point_to_plane": mg / mp}


def convergence(n, deg, frac, seeds):
    out = []
    for mode in ("point_to_point", "point_to_plane", "gicp"):
        rows = []
        for s in seeds:
            q = pair(n, s, deg, frac)
            if mode == "gicp":
                r = icp.gicp(q["src"], q["tgt"], q["ns"], q["nt"], q["R0"], q["t0"], q["d"], epsilon=EPS)
            else:
                r = icp.icp(q["src"], q["tgt"], q["R0"], q["t0"], q["d"], target_normals=q["nt"],
                            point_to_plane=mode == "point_to_plane")
            rows.append({"seed": s, "iterations": r.iterations, "status": r.status, "fitness": r.fitness,
                         "rotation_error_deg": float(np.degrees(synth.rotation_error(r.R, q["R"]))),
                         "translation_error_rel": float(np.linalg.norm(r.t - q["t"]) / q["ext"])})
        out.append({"n": n, "start_deg": deg, "start_shift_rel": frac, "mode": mode, "runs": rows,
                    "median_iterations": float(np.median([x["iterations"] for x in rows])),
                    "median_rotation_error_deg": float(np.median([x["rotation_error_deg"] for x in rows])),
                    "median_translation_error_rel": float(np.median([x["translation_error_rel"] for x in rows]))})
        print(json.dumps({k: v for k, v in out[-1].items() if k != "runs"}), flush=True)
    return out


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_gicp_bench.json"))
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of point-to-plane and GICP per line")
    ap.add_argument("--parent-lib", default=None, help="libpsulvsb_b200.so of the parent commit (ICP regression)")
    ap.add_argument("--repeats", type=int, default=3, help="alternations of parent and new per ICP line")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gicp_bench: no CUDA device (nothing is measured without one)")
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": smi("power.limit"),
           "sm_clock_max_mhz": smi("clocks.max.sm"), "iterations": ITERS, "epsilon": EPS, "single_lines": [],
           "batch_lines": [], "convergence": [], "icp_regression_lines": []}
    L = capi.lib()
    for n in (50000, 500000):
        line = single_line(L, n, args.min_seconds, args.rounds)
        res["single_lines"].append(line)
        print(json.dumps(line), flush=True)
    for B, n in ((592, 5000), (16, 50000)):
        line = batch_line(L, B, n, args.min_seconds, args.rounds)
        res["batch_lines"].append(line)
        print(json.dumps(line), flush=True)
    for deg, frac in ((2.0, 0.01), (5.0, 0.03)):
        res["convergence"] += convergence(50000, deg, frac, range(10, 15))
    if args.parent_lib:
        P = declare_icp(C.CDLL(os.path.abspath(args.parent_lib)))
        res["icp_regression_lines"] = single_lines(L, P, args.min_seconds, args.repeats)
    res["sm_clock_during_mhz"] = smi("clocks.sm")
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "power_limit_w", "sm_clock_during_mhz")}))


if __name__ == "__main__":
    main()
