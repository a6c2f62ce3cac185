"""Times the normals-alone stage (psulvsb_normals / psulvsb_normals_batch, csrc/k8_features.cu) against what users had
before it, and checks FPFH against a build of the parent commit.

Workload (features_bench.py's): the seeded synthetic surface (synth.make_surface), radii scaled with the spacing,
s = sqrt(5000 / n): r_n = 0.06 s, r_f = 0.1 s.  Lines:
* radius normals (max_nn = 0, radius r_n) against psulvsb_fpfh (r_n, r_f), 50 000 and 500 000 points;
* hybrid normals, max_nn = 30, radius 0.12 s (the share of neighbourhoods over 30 points is reported);
* psulvsb_estimate_normals (k = 20, the O(n^2) k-NN path) at 50 000 points;
* batches of 592 x 5 000 and 16 x 50 000 points, radius and hybrid: one psulvsb_normals_batch call against a loop of
  psulvsb_normals calls, with the kernels, copies and memsets of one call counted by torch.profiler;
* with --parent-lib: psulvsb_fpfh (50 000 and 500 000 points) and psulvsb_fpfh_batch (592 x 5 000) through that
  library and this one, alternated `--rounds` times, outputs compared bit for bit.

CUDA events around back-to-back calls after a warm-up, at least `--min-seconds` of timed work per measurement, medians
of `--rounds` alternations; the device name, power limit and SM clock are read in the same run.

    python profiles/tools/normals_bench.py [--out profiles/r9_normals_bench.json] [--parent-lib PATH]
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


def radii(n):
    s = (5000.0 / n) ** 0.5
    return 0.06 * s, 0.1 * s, 0.12 * s


def over(P, r, k):
    from scipy.spatial import cKDTree

    return float(np.mean(cKDTree(P.T).query_ball_point(P.T, r, return_length=True) > k))


def alternate(fns, rounds, min_seconds):
    """{name: [ms per call of each round]}: the functions timed in turn, `rounds` times."""
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            out[k].append(timed(fn, min_seconds)[0])
    return out


def med(xs):
    return float(np.median(xs))


def launches(fn):
    """Kernels, copies and memsets of one call of fn (torch.profiler, CUDA activities), warmed up first."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
    return {"kernels": sum(1 for x in names if "k8_" in x), "memcpy": sum(1 for x in names if "Memcpy" in x),
            "memset": sum(1 for x in names if "Memset" in x), "k8_names": sorted({x.split("<")[0].split("(")[0]
                                                                                   for x in names if "k8_" in x})}


def single_lines(rounds, min_seconds):
    import torch

    out = []
    for n in (50000, 500000):
        P = synth.make_surface(n, 1)
        d = stages.to_device_points(P)
        rn, rf, rh = radii(n)
        L = capi.lib()
        work = torch.empty(int(L.psulvsb_fpfh_workspace_bytes(n)), dtype=torch.uint8, device="cuda")
        fns = {"normals_radius": lambda: features.normals_device(d, rn, 0, work=work),
               "normals_hybrid30": lambda: features.normals_device(d, rh, 30, work=work),
               "fpfh": lambda: features.fpfh_device(d, rn, rf)}
        t = alternate(fns, rounds, min_seconds)
        same = torch.equal(features.normals_device(d, rn).isnan(), features.fpfh_device(d, rn, rn)[1].isnan()) and \
            bool(torch.equal(torch.nan_to_num(features.normals_device(d, rn), 9.0),
                             torch.nan_to_num(features.fpfh_device(d, rn, rn)[1], 9.0)))
        line = {"n": n, "normal_radius": rn, "feature_radius": rf, "hybrid_radius": rh,
                "hybrid_share_over_30": over(P, rh, 30), "ms": {k: med(v) for k, v in t.items()},
                "ms_rounds": t, "radius_over_fpfh": med(t["normals_radius"]) / med(t["fpfh"]),
                "hybrid30_over_radius": med(t["normals_hybrid30"]) / med(t["normals_radius"]),
                "radius_equals_fpfh_normals_rf_eq_rn": same,
                "workspace_bytes": {"normals": int(L.psulvsb_normals_workspace_bytes(n)),
                                    "fpfh": int(L.psulvsb_fpfh_workspace_bytes(n))}}
        if n == 50000:
            knn = torch.empty((n, 3), dtype=torch.float64, device="cuda")
            origin = (C.c_double * 3)(0.0, 0.0, 0.0)
            t = alternate({"estimate_normals_k20": lambda: capi.check(L.psulvsb_estimate_normals(
                stages._stream(), stages._dev(d), n, 20, origin, stages._dev(knn)))}, 1, min_seconds)
            line["ms"]["estimate_normals_k20"] = med(t["estimate_normals_k20"])
            line["estimate_k20_over_radius"] = line["ms"]["estimate_normals_k20"] / line["ms"]["normals_radius"]
        out.append(line)
        print(json.dumps({k: v for k, v in line.items() if k != "ms_rounds"}), flush=True)
    return out


def batch_lines(rounds, min_seconds):
    import torch

    out = []
    for B, n in ((592, 5000), (16, 50000)):
        d = [stages.to_device_points(synth.make_surface(n, 7000 + b)) for b in range(B)]
        rn, _, rh = radii(n)
        L = capi.lib()
        for mode, r, k in (("radius", rn, 0), ("hybrid30", rh, 30)):
            arr = features._clouds([stages._dev(p) for p in d], [n] * B, [(0.0, 0.0, 0.0)] * B)
            work = torch.empty(int(L.psulvsb_normals_batch_workspace_bytes(arr, B)), dtype=torch.uint8, device="cuda")
            one = torch.empty(int(L.psulvsb_normals_workspace_bytes(n)), dtype=torch.uint8, device="cuda")
            res = torch.empty((B * n, 3), dtype=torch.float64, device="cuda")
            singles = [res[b * n:(b + 1) * n] for b in range(B)]
            vp = (C.c_double * 3)(0.0, 0.0, 0.0)

            def batch():
                capi.check(L.psulvsb_normals_batch(stages._stream(), arr, B, r, k, stages._dev(work),
                                                   stages._dev(res)))

            def loop():
                for b in range(B):
                    capi.check(L.psulvsb_normals(stages._stream(), stages._dev(d[b]), n, r, k, vp, stages._dev(one),
                                                 stages._dev(singles[b])))

            loop()
            want = res.clone()
            batch()
            same = bool(torch.equal(torch.nan_to_num(res, 9.0), torch.nan_to_num(want, 9.0)))
            t = alternate({"batch": batch, "loop": loop}, rounds, min_seconds)
            line = {"B": B, "n": n, "mode": mode, "radius": r, "max_nn": k, "ms": {x: med(v) for x, v in t.items()},
                    "ms_rounds": t, "clouds_per_s": {x: B / med(v) * 1e3 for x, v in t.items()},
                    "loop_over_batch": med(t["loop"]) / med(t["batch"]), "batch_equals_loop": same,
                    "per_call_batch": launches(batch), "per_single_call": launches(
                        lambda: capi.check(L.psulvsb_normals(stages._stream(), stages._dev(d[0]), n, r, k, vp,
                                                             stages._dev(one), stages._dev(singles[0]))))}
            out.append(line)
            print(json.dumps({x: v for x, v in line.items() if x != "ms_rounds"}), flush=True)
    return out


def declare_fpfh(lib):
    vp, ull = C.c_void_p, C.c_ulonglong
    lib.psulvsb_fpfh_workspace_bytes.argtypes = [C.c_int]
    lib.psulvsb_fpfh_workspace_bytes.restype = ull
    lib.psulvsb_fpfh.argtypes = [vp, vp, C.c_int, C.c_double, C.c_double, C.POINTER(C.c_double), vp, vp, vp]
    lib.psulvsb_fpfh_batch_workspace_bytes.argtypes = [C.POINTER(capi.FpfhCloud), C.c_int]
    lib.psulvsb_fpfh_batch_workspace_bytes.restype = ull
    lib.psulvsb_fpfh_batch.argtypes = [vp, C.POINTER(capi.FpfhCloud), C.c_int, C.c_double, C.c_double, vp, vp, vp]
    return lib


def parent_lines(path, rounds, min_seconds):
    import torch

    libs = {"parent": declare_fpfh(C.CDLL(path)), "new": capi.lib()}
    out = []
    cases = [("fpfh", 1, 50000), ("fpfh", 1, 500000), ("fpfh_batch", 592, 5000)]
    for call, B, n in cases:
        d = [stages.to_device_points(synth.make_surface(n, 11 + b)) for b in range(B)]
        rn, rf, _ = radii(n)
        arr = features._clouds([stages._dev(p) for p in d], [n] * B, [(0.0, 0.0, 1.0)] * B)
        vp = (C.c_double * 3)(0.0, 0.0, 1.0)
        bufs = {}
        fns = {}
        for name, L in libs.items():
            ws = L.psulvsb_fpfh_batch_workspace_bytes(arr, B)
            work = torch.empty(int(ws), dtype=torch.uint8, device="cuda")
            feats = torch.empty((B * n, 33), dtype=torch.float32, device="cuda")
            nrm = torch.empty((B * n, 3), dtype=torch.float64, device="cuda")
            bufs[name] = (feats, nrm)
            if call == "fpfh":
                fns[name] = (lambda L=L, work=work, feats=feats, nrm=nrm: capi.check(L.psulvsb_fpfh(
                    stages._stream(), stages._dev(d[0]), n, rn, rf, vp, stages._dev(work), stages._dev(nrm),
                    stages._dev(feats))))
            else:
                fns[name] = (lambda L=L, work=work, feats=feats, nrm=nrm: capi.check(L.psulvsb_fpfh_batch(
                    stages._stream(), arr, B, rn, rf, stages._dev(work), stages._dev(nrm), stages._dev(feats))))
        for fn in fns.values():
            fn()
        torch.cuda.synchronize()
        same = all(torch.equal(torch.nan_to_num(bufs["parent"][i], 9.0), torch.nan_to_num(bufs["new"][i], 9.0))
                   for i in range(2))
        t = alternate(fns, rounds, min_seconds)
        line = {"call": call, "B": B, "n": n, "parent_ms": t["parent"], "new_ms": t["new"],
                "new_over_parent": med(t["new"]) / med(t["parent"]), "identical_outputs": same}
        out.append(line)
        print(json.dumps(line), flush=True)
    return out


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9_normals_bench.json"))
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--parent-lib", default=None, help="libpsulvsb_b200.so of the parent commit (FPFH regression)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("normals_bench: no CUDA device (nothing is measured without one)")
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": smi("power.limit"),
           "sm_clock_max_mhz": smi("clocks.max.sm")}
    res["single"] = single_lines(args.rounds, args.min_seconds)
    res["batch"] = batch_lines(args.rounds, args.min_seconds)
    if args.parent_lib:
        res["parent_vs_new"] = parent_lines(args.parent_lib, args.rounds, args.min_seconds)
    res["sm_clock_during_mhz"] = smi("clocks.sm")
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "power_limit_w", "sm_clock_during_mhz")}))


if __name__ == "__main__":
    main()
