"""Times the robust kernels of point-to-plane ICP and generalized ICP (psulvsb_icp_robust[_batch],
psulvsb_gicp_robust[_batch], csrc/k9_icp.cu) against the plain modes on the same inputs, checks their outputs in the
run, and tabulates their accuracy on a partial-overlap scene with clutter.

Workload: gicp_bench.py's seeded synthetic surface pairs (noise 0.1 mean spacings, 2 degrees and 1 % of the extent
from the truth, d = 3 mean spacings, radius normals), TukeyLoss(d / 3) for the robust calls.  Lines:
* single pairs, 50 000 and 500 000 points, 30 forced iterations (relative criteria 0): ms per call and per round of
  plain and robust point-to-plane and GICP, the four alternated `--rounds` times;
* batches, 592 x 5 000 and 16 x 50 000: pairs/s of the same four calls;
* checks: the L2 loss through psulvsb_icp_robust returns psulvsb_icp's result bytes, and the timed robust calls
  return the result of their first call;
* accuracy: five seeds of a 20 000-point surface seen with 60 % overlap, 20 % of the source replaced by uniform
  outliers in its bounding box, started 5 degrees and 3 % of the extent from the truth, default criteria: rotation
  error (degrees) and translation error (fraction of the extent) of L2 and each kernel, both objectives.

CUDA events around back-to-back calls after a warm-up, at least `--min-seconds` of timed work per measurement, medians
of the alternations; the device name, power limit and SM clock are read in the same run.

    python profiles/tools/robust_icp_bench.py [--out profiles/r13_robust_icp_bench.json]
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
from gicp_bench import EPS, ITERS, moved, pair, params  # noqa: E402
from icp_bench import smi, timed  # noqa: E402
from psulvsb_b200 import capi, features, icp, stages, synth  # noqa: E402

MODES = ("point_to_plane", "point_to_plane_robust", "gicp", "gicp_robust")


def tukey(d):
    return capi.RobustKernel(capi.LOSS_TUKEY, d / 3.0)


def alternate(fns, min_seconds, rounds):
    """{mode: [ms per call of each alternation]}, the modes timed in turn."""
    ms = {m: [] for m in fns}
    for _ in range(rounds):
        for m, fn in fns.items():
            ms[m].append(timed(fn, min_seconds)[0])
    return ms


def single_line(L, n, min_seconds, rounds):
    import torch

    q = pair(n, 1)
    ds, dt = stages.to_device_points(q["src"]), stages.to_device_points(q["tgt"])
    dns, dnt = stages.to_device_points(q["ns"]), stages.to_device_points(q["nt"])
    work = torch.empty(L.psulvsb_icp_workspace_bytes(n, n), dtype=torch.uint8, device="cuda")
    res = {m: torch.empty(C.sizeof(capi.IcpResult), dtype=torch.uint8, device="cuda") for m in MODES + ("l2",)}
    R0 = (C.c_double * 9)(*q["R0"].flatten(order="F"))
    t0 = (C.c_double * 3)(*q["t0"])
    stream = stages._stream()
    p2l, p2p = params(L, q["d"], True), params(L, q["d"], False)
    loss, l2 = tukey(q["d"]), capi.RobustKernel(capi.LOSS_L2, 1.0)
    a = (ds.data_ptr(), n, dt.data_ptr(), n, dnt.data_ptr(), C.byref(p2l))
    g = (ds.data_ptr(), n, dns.data_ptr(), dt.data_ptr(), n, dnt.data_ptr(), C.byref(p2p), EPS)
    tail = lambda m: (R0, t0, work.data_ptr(), res[m].data_ptr(), None, None)  # noqa: E731
    fns = {"point_to_plane": lambda: capi.check(L.psulvsb_icp(stream, *a, *tail("point_to_plane"))),
           "point_to_plane_robust": lambda: capi.check(L.psulvsb_icp_robust(stream, *a, C.byref(loss),
                                                                             *tail("point_to_plane_robust"))),
           "gicp": lambda: capi.check(L.psulvsb_gicp(stream, *g, *tail("gicp"))),
           "gicp_robust": lambda: capi.check(L.psulvsb_gicp_robust(stream, *g, C.byref(loss), *tail("gicp_robust")))}
    capi.check(L.psulvsb_icp_robust(stream, *a, C.byref(l2), *tail("l2")))
    for fn in fns.values():
        fn()
    first = {m: res[m].cpu().numpy().tobytes() for m in res}
    ms = alternate(fns, min_seconds, rounds)
    after = {m: res[m].cpu().numpy().tobytes() for m in MODES}
    out = {m: capi.IcpResult.from_buffer_copy(first[m]) for m in MODES}
    line = {"n": n, "d": q["d"], "loss": "TukeyLoss(d / 3)",
            "l2_robust_bytes_equal_point_to_plane": first["l2"] == first["point_to_plane"],
            "timed_results_equal_first": all(after[m] == first[m] for m in MODES)}
    for m in MODES:
        med = float(np.median(ms[m]))
        line[m] = {"ms": ms[m], "ms_per_round": med / (ITERS + 1), "iterations": out[m].iterations,
                   "fitness": out[m].fitness,
                   "rotation_error_deg": float(np.degrees(synth.rotation_error(
                       np.array(out[m].rotation[:]).reshape(3, 3, order="F"), q["R"])))}
    line["robust_over_plain"] = {"point_to_plane": float(np.median(ms["point_to_plane_robust"]) /
                                                         np.median(ms["point_to_plane"])),
                                 "gicp": float(np.median(ms["gicp_robust"]) / np.median(ms["gicp"]))}
    return line


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
    res = {m: torch.empty(B * C.sizeof(capi.IcpResult), dtype=torch.uint8, device="cuda") for m in MODES + ("l2",)}
    stream = stages._stream()
    p2l, p2p = params(L, d, True), params(L, d, False)
    loss, l2 = tukey(d), capi.RobustKernel(capi.LOSS_L2, 1.0)
    tail = lambda m: (work.data_ptr(), res[m].data_ptr(), None, None)  # noqa: E731
    fns = {"point_to_plane": lambda: capi.check(L.psulvsb_icp_batch(stream, ip, B, C.byref(p2l),
                                                                    *tail("point_to_plane"))),
           "point_to_plane_robust": lambda: capi.check(L.psulvsb_icp_robust_batch(
               stream, ip, B, C.byref(p2l), C.byref(loss), *tail("point_to_plane_robust"))),
           "gicp": lambda: capi.check(L.psulvsb_gicp_batch(stream, gp, B, C.byref(p2p), EPS, *tail("gicp"))),
           "gicp_robust": lambda: capi.check(L.psulvsb_gicp_robust_batch(stream, gp, B, C.byref(p2p), EPS,
                                                                         C.byref(loss), *tail("gicp_robust")))}
    capi.check(L.psulvsb_icp_robust_batch(stream, ip, B, C.byref(p2l), C.byref(l2), *tail("l2")))
    for fn in fns.values():
        fn()
    first = {m: res[m].cpu().numpy().tobytes() for m in res}
    ms = alternate(fns, min_seconds, rounds)
    after = {m: res[m].cpu().numpy().tobytes() for m in MODES}
    line = {"B": B, "n": n, "loss": "TukeyLoss(d / 3)",
            "l2_robust_bytes_equal_point_to_plane": first["l2"] == first["point_to_plane"],
            "timed_results_equal_first": all(after[m] == first[m] for m in MODES)}
    for m in MODES:
        r = (capi.IcpResult * B).from_buffer_copy(first[m])
        med = float(np.median(ms[m]))
        line[m] = {"ms": ms[m], "pairs_per_s": B / (med * 1e-3), "iterations": sorted({x.iterations for x in r}),
                   "mean_fitness": float(np.mean([x.fitness for x in r]))}
    line["robust_over_plain"] = {"point_to_plane": float(np.median(ms["point_to_plane_robust"]) /
                                                         np.median(ms["point_to_plane"])),
                                 "gicp": float(np.median(ms["gicp_robust"]) / np.median(ms["gicp"]))}
    return line


def cluttered_pair(seed, n=20000, overlap=0.6, outliers=0.2, deg=5.0, frac=0.03):
    """A surface seen with `overlap` of the target kept, `outliers` of the source uniform in its bounding box."""
    rng = np.random.default_rng(seed)
    P = synth.make_surface(n, seed % 8)
    sp = 2.0 / np.sqrt(n)
    R, _ = synth.random_rigid(rng)
    t = rng.normal(size=3)
    ext = float(np.linalg.norm(np.ptp(P, axis=1)))
    src = P + rng.normal(0, 0.1 * sp, P.shape)
    out = rng.random(n) < outliers
    lo, hi = P.min(axis=1), P.max(axis=1)
    src[:, out] = rng.uniform(lo[:, None], hi[:, None], (3, int(out.sum())))
    keep = P[0] <= np.quantile(P[0], overlap)
    tgt = R @ P[:, keep] + t[:, None] + rng.normal(0, 0.1 * sp, (3, int(keep.sum())))
    R0, t0 = moved(R, t, rng, deg, frac, ext)
    ns, nt = features.fpfh(src, 4 * sp, 8 * sp)[1], features.fpfh(tgt, 4 * sp, 8 * sp)[1]
    return dict(src=src, tgt=tgt, ns=ns, nt=nt, R=R, t=t, R0=R0, t0=t0, d=3.0 * sp, ext=ext, sp=sp)


def accuracy(seeds):
    rows = []
    for s in seeds:
        q = cluttered_pair(s)
        d = q["d"]
        kernels = {"L2": None, "L2Loss()": icp.L2Loss(), "HuberLoss(d/3)": icp.HuberLoss(d / 3),
                   "CauchyLoss(d/3)": icp.CauchyLoss(d / 3), "GMLoss((d/3)^2)": icp.GMLoss((d / 3) ** 2),
                   "TukeyLoss(d)": icp.TukeyLoss(d)}
        for obj in ("point_to_plane", "gicp"):
            for name, loss in kernels.items():
                if obj == "gicp":
                    r = icp.gicp(q["src"], q["tgt"], q["ns"], q["nt"], q["R0"], q["t0"], d, epsilon=EPS, loss=loss)
                else:
                    r = icp.icp(q["src"], q["tgt"], q["R0"], q["t0"], d, target_normals=q["nt"], point_to_plane=True,
                                loss=loss)
                rows.append({"seed": s, "objective": obj, "loss": name, "iterations": r.iterations,
                             "status": r.status, "fitness": r.fitness,
                             "rotation_error_deg": float(np.degrees(synth.rotation_error(r.R, q["R"]))),
                             "translation_error_rel": float(np.linalg.norm(r.t - q["t"]) / q["ext"])})
    table = []
    for obj in ("point_to_plane", "gicp"):
        for name in dict.fromkeys(r["loss"] for r in rows):
            sel = [r for r in rows if r["objective"] == obj and r["loss"] == name]
            table.append({"objective": obj, "loss": name,
                          "median_rotation_error_deg": float(np.median([r["rotation_error_deg"] for r in sel])),
                          "median_translation_error_rel": float(np.median([r["translation_error_rel"] for r in sel])),
                          "max_rotation_error_deg": float(np.max([r["rotation_error_deg"] for r in sel])),
                          "median_iterations": float(np.median([r["iterations"] for r in sel]))})
            print(json.dumps(table[-1]), flush=True)
    return {"scene": "synth.make_surface(20000), 60 % overlap, 20 % uniform source outliers, noise 0.1 spacings, "
                     "start 5 deg / 3 % of the extent, d = 3 spacings, radius normals (4 spacings), default criteria",
            "table": table, "runs": rows}


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r13_robust_icp_bench.json"))
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the four modes per line")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("robust_icp_bench: no CUDA device (nothing is measured without one)")
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": smi("power.limit"),
           "sm_clock_max_mhz": smi("clocks.max.sm"), "iterations": ITERS, "epsilon": EPS, "single_lines": [],
           "batch_lines": []}
    L = capi.lib()
    for n in (50000, 500000):
        line = single_line(L, n, args.min_seconds, args.rounds)
        res["single_lines"].append(line)
        print(json.dumps(line), flush=True)
    for B, n in ((592, 5000), (16, 50000)):
        line = batch_line(L, B, n, args.min_seconds, args.rounds)
        res["batch_lines"].append(line)
        print(json.dumps(line), flush=True)
    res["sm_clock_during_mhz"] = smi("clocks.sm")
    res["accuracy"] = accuracy(range(20, 25))
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    ok = all(x["l2_robust_bytes_equal_point_to_plane"] and x["timed_results_equal_first"]
             for x in res["single_lines"] + res["batch_lines"])
    res["checks_passed"] = ok
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "power_limit_w", "sm_clock_during_mhz", "checks_passed")}))
    if not ok:
        raise SystemExit("robust_icp_bench: an output check failed")


if __name__ == "__main__":
    main()
