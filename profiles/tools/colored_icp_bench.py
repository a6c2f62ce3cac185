"""Times colored ICP (psulvsb_colored_icp[_batch], csrc/k9_icp.cu) and its colour-gradient stage
(psulvsb_color_gradients_batch, csrc/k8_colors.cu) against point-to-plane ICP on the same inputs, and checks their
outputs in the run.

Workload: gicp_bench.py's seeded synthetic surface pairs (noise 0.1 mean spacings, 2 degrees and 1 % of the extent
from the truth, d = 3 mean spacings, radius normals), coloured by a smooth RGB field over the world coordinates
(period about a fifth of the extent), lambda_geometric 0.968, the L2 loss.  Lines:
* the gradient stage alone on the 50 000- and 500 000-point targets (radius 2 d, max_nn 30): ms per call;
* single pairs, 50 000 and 500 000 points, 30 forced iterations (relative criteria 0): ms per call and per round of
  point-to-plane ICP and colored ICP, alternated `--rounds` times; a colored call includes its gradient stage, so its
  per-round figure is (call - gradient stage) / 31 evaluations;
* batches, 592 x 5 000 and 16 x 50 000: pairs/s of the same two calls (default criteria);
* checks: colored ICP with lambda 1 returns point-to-plane's result bytes, and the timed calls return the result of
  their first call.

CUDA events around back-to-back calls after a warm-up, at least `--min-seconds` of timed work per measurement, medians
of the alternations; the device name, power limit and SM clock are read in the same run.

    python profiles/tools/colored_icp_bench.py [--out profiles/r14_colored_icp_bench.json]
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
from gicp_bench import ITERS, pair, params  # noqa: E402
from icp_bench import smi, timed  # noqa: E402
from psulvsb_b200 import capi, stages  # noqa: E402

LAMBDA = 0.968
MODES = ("point_to_plane", "colored")


def colours(X, ext):
    x, y, z = X / (0.2 * ext / np.pi)
    return np.clip(np.vstack([0.5 + 0.3 * np.sin(x) * np.cos(y), 0.5 + 0.3 * np.sin(y + 0.5 * z),
                              0.5 + 0.3 * np.cos(z - x)]), 0.0, 1.0)


def coloured_pair(n, seed):
    q = pair(n, seed)
    q["ct"] = colours(q["tgt"], q["ext"])
    q["cs"] = colours(q["R"] @ q["src"] + q["t"][:, None], q["ext"])
    return q


def alternate(fns, min_seconds, rounds):
    ms = {m: [] for m in fns}
    for _ in range(rounds):
        for m, fn in fns.items():
            ms[m].append(timed(fn, min_seconds)[0])
    return ms


def gradient_line(L, q, dv, min_seconds):
    import torch

    n = q["tgt"].shape[1]
    cl = (capi.ColorCloud * 1)(capi.ColorCloud(dv["tgt"].data_ptr(), n, dv["ct"].data_ptr(), dv["nt"].data_ptr()))
    work = torch.empty(L.psulvsb_color_gradients_batch_workspace_bytes(cl, 1), dtype=torch.uint8, device="cuda")
    out = torch.empty((n, 3), dtype=torch.float64, device="cuda")
    stream = stages._stream()
    fn = lambda: capi.check(L.psulvsb_color_gradients_batch(stream, cl, 1, 2.0 * q["d"], 30, work.data_ptr(),  # noqa
                                                            out.data_ptr()))
    fn()
    first = out.cpu().numpy().tobytes()
    ms, reps = timed(fn, min_seconds)
    return {"n": n, "radius": 2.0 * q["d"], "max_nn": 30, "ms": ms, "reps": reps,
            "timed_results_equal_first": out.cpu().numpy().tobytes() == first}


def single_line(L, n, min_seconds, rounds):
    import torch

    q = coloured_pair(n, 1)
    dv = {k: stages.to_device_points(q[k]) for k in ("src", "tgt", "nt", "cs", "ct")}
    grad = gradient_line(L, q, dv, min_seconds)
    work = torch.empty(L.psulvsb_colored_icp_workspace_bytes(n, n), dtype=torch.uint8, device="cuda")
    # zeroed: the byte comparisons then see the same (unwritten) padding after the last field
    res = {m: torch.zeros(C.sizeof(capi.IcpResult), dtype=torch.uint8, device="cuda") for m in MODES + ("lambda1",)}
    R0 = (C.c_double * 9)(*q["R0"].flatten(order="F"))
    t0 = (C.c_double * 3)(*q["t0"])
    stream = stages._stream()
    p2l, p2p = params(L, q["d"], True), params(L, q["d"], False)
    a = (dv["src"].data_ptr(), n, dv["tgt"].data_ptr(), n, dv["nt"].data_ptr(), C.byref(p2l))
    c = (dv["src"].data_ptr(), n, dv["cs"].data_ptr(), dv["tgt"].data_ptr(), n, dv["ct"].data_ptr(),
         dv["nt"].data_ptr(), C.byref(p2p))
    tail = lambda m: (R0, t0, work.data_ptr(), res[m].data_ptr(), None, None)  # noqa: E731
    fns = {"point_to_plane": lambda: capi.check(L.psulvsb_icp(stream, *a, *tail("point_to_plane"))),
           "colored": lambda: capi.check(L.psulvsb_colored_icp(stream, *c, LAMBDA, None, *tail("colored")))}
    capi.check(L.psulvsb_colored_icp(stream, *c, 1.0, None, *tail("lambda1")))
    for fn in fns.values():
        fn()
    first = {m: res[m].cpu().numpy().tobytes() for m in res}
    ms = alternate(fns, min_seconds, rounds)
    after = {m: res[m].cpu().numpy().tobytes() for m in MODES}
    line = {"n": n, "d": q["d"], "lambda_geometric": LAMBDA, "gradient_stage": grad,
            "lambda1_bytes_equal_point_to_plane": first["lambda1"] == first["point_to_plane"],
            "timed_results_equal_first": all(after[m] == first[m] for m in MODES) and grad["timed_results_equal_first"]}
    for m in MODES:
        r = capi.IcpResult.from_buffer_copy(first[m])
        med = float(np.median(ms[m]))
        rounds_ms = (med - (grad["ms"] if m == "colored" else 0.0)) / (ITERS + 1)
        line[m] = {"ms": ms[m], "ms_per_round": rounds_ms, "iterations": r.iterations, "fitness": r.fitness}
    line["colored_over_point_to_plane_per_round"] = line["colored"]["ms_per_round"] / \
        line["point_to_plane"]["ms_per_round"]
    return line


def batch_line(L, B, n, min_seconds, rounds):
    import torch

    qs = [coloured_pair(n, 100 * B + b % 8) for b in range(min(B, 8))]
    dev = [{k: stages.to_device_points(q[k]) for k in ("src", "tgt", "nt", "cs", "ct")} for q in qs]
    cp, ip = (capi.ColoredIcpPair * B)(), (capi.IcpPair * B)()
    for b in range(B):
        q, v = qs[b % len(qs)], dev[b % len(dev)]
        g, i = cp[b], ip[b]
        g.src = i.src = v["src"].data_ptr()
        g.tgt = i.tgt = v["tgt"].data_ptr()
        g.n_s = g.n_t = i.n_s = i.n_t = n
        g.src_colors, g.tgt_colors = v["cs"].data_ptr(), v["ct"].data_ptr()
        g.tgt_normals = i.tgt_normals = v["nt"].data_ptr()
        g.R0[:] = i.R0[:] = list(q["R0"].flatten(order="F"))
        g.t0[:] = i.t0[:] = list(q["t0"])
    d = qs[0]["d"]
    work = torch.empty(L.psulvsb_colored_icp_batch_workspace_bytes(cp, B), dtype=torch.uint8, device="cuda")
    res = {m: torch.zeros(B * C.sizeof(capi.IcpResult), dtype=torch.uint8, device="cuda") for m in MODES + ("lambda1",)}
    stream = stages._stream()
    p2l, p2p = params(L, d, True, forced=False), params(L, d, False, forced=False)
    tail = lambda m: (work.data_ptr(), res[m].data_ptr(), None, None)  # noqa: E731
    fns = {"point_to_plane": lambda: capi.check(L.psulvsb_icp_batch(stream, ip, B, C.byref(p2l),
                                                                    *tail("point_to_plane"))),
           "colored": lambda: capi.check(L.psulvsb_colored_icp_batch(stream, cp, B, C.byref(p2p), LAMBDA, None,
                                                                     *tail("colored")))}
    capi.check(L.psulvsb_colored_icp_batch(stream, cp, B, C.byref(p2p), 1.0, None, *tail("lambda1")))
    for fn in fns.values():
        fn()
    first = {m: res[m].cpu().numpy().tobytes() for m in res}
    ms = alternate(fns, min_seconds, rounds)
    after = {m: res[m].cpu().numpy().tobytes() for m in MODES}
    line = {"B": B, "n": n, "lambda_geometric": LAMBDA,
            "lambda1_bytes_equal_point_to_plane": first["lambda1"] == first["point_to_plane"],
            "timed_results_equal_first": all(after[m] == first[m] for m in MODES)}
    for m in MODES:
        r = (capi.IcpResult * B).from_buffer_copy(first[m])
        med = float(np.median(ms[m]))
        line[m] = {"ms": ms[m], "pairs_per_s": B / (med * 1e-3), "iterations": sorted({x.iterations for x in r}),
                   "mean_fitness": float(np.mean([x.fitness for x in r]))}
    return line


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r14_colored_icp_bench.json"))
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two modes per line")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("colored_icp_bench: no CUDA device (nothing is measured without one)")
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": smi("power.limit"),
           "sm_clock_max_mhz": smi("clocks.max.sm"), "iterations": ITERS, "single_lines": [], "batch_lines": []}
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
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    ok = all(x["lambda1_bytes_equal_point_to_plane"] and x["timed_results_equal_first"]
             for x in res["single_lines"] + res["batch_lines"])
    res["checks_passed"] = ok
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "power_limit_w", "sm_clock_during_mhz", "checks_passed")}))
    if not ok:
        raise SystemExit("colored_icp_bench: an output check failed")


if __name__ == "__main__":
    main()
