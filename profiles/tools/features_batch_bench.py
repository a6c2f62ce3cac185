"""Times the batched correspondence stage (psulvsb_fpfh_batch + psulvsb_match_batch) against a loop of single calls on
one GPU, alternated, on seeded synthetic surfaces (synth.make_surface, radii scaled with the spacing as in
features_bench.py): B pairs of N points, FPFH of both clouds plus the crosscheck matcher (and one line with the tuple
test).  Then the raw-cloud chain for 592 pairs, batch against loop: fpfh_batch -> match_batch -> solve_batch ->
icp_batch, with the time per stage.  With --parent-lib, the single-call lines of features_bench.py through the parent
build's library and this one, alternated, with a check that the results are identical.  Device name, power limit and SM
clock are read in the same run.

    python profiles/tools/features_batch_bench.py [--parent-lib path/to/libpsulvsb_b200.so] [--out ...]
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

UNIT_SLOTS = 66
# launches of one batched call, from run_fpfh / run_match (kernels, plus the table copy and the memsets)
FPFH_OPS = 9           # table copy, memset, 7 kernels
MATCH_CROSS_OPS = 7    # table copy, key memset, NN, finish, flags, scan, place


def smi(query):
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=" + query, "--format=csv,noheader,nounits", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return ""


def wall(fn, reps):
    import torch

    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) / reps * 1e3


def workload(B, n, seed):
    rng = np.random.default_rng(seed)
    s = (5000.0 / n) ** 0.5
    d_clouds = []
    for b in range(B):
        P = synth.make_surface(n, 1000 * seed + b)
        R, _ = synth.random_rigid(rng)
        Q = R @ P + rng.normal(0, 0.002 * s, P.shape)
        d_clouds += [stages.to_device_points(P), stages.to_device_points(Q)]
    return d_clouds, 0.06 * s, 0.1 * s


def loop_call(d_clouds, rn, rf, tuple_test):
    out = []
    for b in range(len(d_clouds) // 2):
        fs, _ = features.fpfh_device(d_clouds[2 * b], rn, rf)
        ft, _ = features.fpfh_device(d_clouds[2 * b + 1], rn, rf)
        src, tgt = d_clouds[2 * b].cpu().numpy().T, d_clouds[2 * b + 1].cpu().numpy().T
        out.append(features.match(src, tgt, fs.cpu().numpy(), ft.cpu().numpy(), crosscheck=True, tuple_test=tuple_test,
                                  seed=b))
    return out


def batch_call(d_clouds, rn, rf, tuple_test, work):
    feats, _, views = features.fpfh_batch_device(d_clouds, rn, rf, work=work[0])
    pairs, counts, offs = features.match_batch_device(d_clouds[0::2], d_clouds[1::2], [v[0] for v in views[0::2]],
                                                      [v[0] for v in views[1::2]], crosscheck=True,
                                                      tuple_test=tuple_test, seed=0, work=work[1])
    return pairs, counts, offs


def nn_time(d_clouds, rn, rf):
    """CUDA-event time of one crosscheck psulvsb_match_batch on the batch's descriptors (the NN and the list kernels; the
    NN is not timed apart), and the descriptor distances it evaluates."""
    import torch

    _, _, views = features.fpfh_batch_device(d_clouds, rn, rf)
    fs, ft = [v[0] for v in views[0::2]], [v[0] for v in views[1::2]]
    work = torch.empty(max(1, capi.lib().psulvsb_match_batch_workspace_bytes(
        features._match_pairs([(None, None, None, None)] * len(fs), [(f.shape[0], g.shape[0]) for f, g in zip(fs, ft)],
                              [0] * len(fs)), len(fs), 1, 0)), dtype=torch.uint8, device="cuda")
    fn = lambda: features.match_batch_device(d_clouds[0::2], d_clouds[1::2], fs, ft, crosscheck=True, work=work)  # noqa
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(10):
        fn()
    b.record()
    b.synchronize()
    ms = a.elapsed_time(b) / 10
    return ms, sum(f.shape[0] * g.shape[0] for f, g in zip(fs, ft))


def loop_vs_batch(B, n, tuple_test, rounds):
    import torch

    d_clouds, rn, rf = workload(B, n, 3)
    L = capi.lib()
    arr = features._clouds([None] * len(d_clouds), [n] * len(d_clouds), [(0.0, 0.0, 0.0)] * len(d_clouds))
    marr = features._match_pairs([(None, None, None, None)] * B, [(n, n)] * B, [0] * B)
    work = (torch.empty(L.psulvsb_fpfh_batch_workspace_bytes(arr, len(d_clouds)), dtype=torch.uint8, device="cuda"),
            torch.empty(L.psulvsb_match_batch_workspace_bytes(marr, B, 1, int(tuple_test)), dtype=torch.uint8,
                        device="cuda"))
    want = loop_call(d_clouds, rn, rf, tuple_test)
    pairs, counts, offs = batch_call(d_clouds, rn, rf, tuple_test, work)
    pairs, counts = pairs.cpu().numpy(), counts.cpu().numpy()
    identical = all(np.array_equal(pairs[offs[b]:offs[b] + counts[b]], want[b]) for b in range(B))
    reps_loop = max(1, 8 // B)
    t_loop, t_batch = [], []
    for _ in range(rounds):
        t_loop.append(wall(lambda: loop_call(d_clouds, rn, rf, tuple_test), reps_loop))
        t_batch.append(wall(lambda: batch_call(d_clouds, rn, rf, tuple_test, work), 3))
    ml, mb = float(np.median(t_loop)), float(np.median(t_batch))
    line = {"pairs": B, "n": n, "tuple_test": tuple_test, "loop_ms": t_loop, "batch_ms": t_batch,
            "loop_pairs_per_s": B / ml * 1e3, "batch_pairs_per_s": B / mb * 1e3, "speedup": ml / mb,
            "identical": identical, "launches_batch_fpfh": FPFH_OPS,
            "launches_batch_match": MATCH_CROSS_OPS if not tuple_test else "7 + 2 per tuple round",
            "launches_loop": f"{B} x (2 x {FPFH_OPS - 1} FPFH + match_host)"}
    if not tuple_test:
        # the crosscheck match alone (NN plus the list kernels): its distances over the NN's roofline bound the NN's share
        line["match_batch_ms"], line["distances"] = nn_time(d_clouds, rn, rf)
    print(json.dumps(line), flush=True)
    return line


def chain(B, rounds):
    """fpfh_batch -> match_batch -> solve_batch -> icp_batch (host entry points), against the loop of single calls."""
    rng = np.random.default_rng(7)
    srcs, tgts, vps = [], [], []
    for b in range(B):
        P = synth.make_surface(5000, 7000 + b)
        R, _ = synth.random_rigid(rng)
        t = rng.uniform(-0.5, 0.5, 3)
        srcs.append(P)
        tgts.append(R @ P + t[:, None] + rng.normal(0, 0.002, P.shape))
        vps.append(tuple(t))
    rn, rf = 0.06, 0.1
    kw = dict(noise_bound=0.01, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005, wallclock_cap_s=0.0,
              seed=1)
    h = capi.Handle(0)

    def stages_batch():
        t = [time.perf_counter()]
        f = features.fpfh_batch(srcs + tgts, rn, rf, viewpoints=[(0.0, 0.0, 0.0)] * B + vps)
        t.append(time.perf_counter())
        m = features.match_batch(srcs, tgts, [x[0] for x in f[:B]], [x[0] for x in f[B:]], crosscheck=True)
        t.append(time.perf_counter())
        sols = h.solve_batch(capi.default_params(**kw), [capi.HostProblem(s[:, k[:, 0]], g[:, k[:, 1]])
                                                         for s, g, k in zip(srcs, tgts, m)])
        t.append(time.perf_counter())
        icp.icp_batch(srcs, tgts, np.array([s.R for s in sols]), np.array([s.t for s in sols]), 0.05)
        t.append(time.perf_counter())
        return np.diff(t) * 1e3, m

    def stages_loop():
        t = [time.perf_counter()]
        fs = [features.fpfh(s, rn, rf)[0] for s in srcs]
        ft = [features.fpfh(g, rn, rf, viewpoint=v)[0] for g, v in zip(tgts, vps)]
        t.append(time.perf_counter())
        m = [features.match(s, g, a, b, crosscheck=True) for s, g, a, b in zip(srcs, tgts, fs, ft)]
        t.append(time.perf_counter())
        return np.diff(t) * 1e3, m

    stages_batch()
    stages_loop()
    tb, tl, same = [], [], True
    for _ in range(rounds):
        a, mb = stages_batch()
        b, ml = stages_loop()
        tb.append(a.tolist())
        tl.append(b.tolist())
        same = same and all(np.array_equal(x, y) for x, y in zip(mb, ml))
    med_b, med_l = np.median(tb, axis=0), np.median(tl, axis=0)
    line = {"pairs": B, "n": 5000, "batch_stage_ms": {"fpfh_batch": med_b[0], "match_batch": med_b[1],
                                                       "solve_batch": med_b[2], "icp_batch": med_b[3]},
            "loop_stage_ms": {"fpfh_loop": med_l[0], "match_loop": med_l[1]},
            "correspondence_stage_speedup": float(med_l.sum() / med_b[:2].sum()), "identical_correspondences": same,
            "all_ms_batch": tb, "all_ms_loop": tl}
    print(json.dumps(line), flush=True)
    return line


def parent_compare(path, rounds, min_reps=20):
    """The single-call lines of features_bench.py through the parent build and this one, alternated (host wall clock
    around `reps` calls ending in a synchronise); results compared bit for bit."""
    import torch

    libs = {"parent": C.CDLL(path), "new": capi.lib()}
    for L in libs.values():
        L.psulvsb_fpfh_workspace_bytes.restype = C.c_ulonglong
        L.psulvsb_fpfh_workspace_bytes.argtypes = [C.c_int]
        L.psulvsb_fpfh.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p]
        L.psulvsb_feature_nn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.psulvsb_match_host.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                         C.c_int, C.c_double, C.c_uint64, C.c_void_p, C.c_longlong,
                                         C.POINTER(C.c_longlong)]
    lines = []
    for n in (5000, 50000):
        P = synth.make_surface(n, 1)
        s = (5000.0 / n) ** 0.5
        rn, rf = 0.06 * s, 0.1 * s
        d = stages.to_device_points(P)
        R, _ = synth.random_rigid(np.random.default_rng(2))
        Q = R @ P
        dq = stages.to_device_points(Q)
        work = torch.empty(max(int(L.psulvsb_fpfh_workspace_bytes(n)) for L in libs.values()), dtype=torch.uint8,
                           device="cuda")
        out = {k: (torch.empty((n, 33), dtype=torch.float32, device="cuda"),
                   torch.empty((n, 33), dtype=torch.float32, device="cuda")) for k in libs}
        nn = {k: (torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, dtype=torch.int32, device="cuda"))
              for k in libs}
        pairs = {k: np.zeros((n, 2), dtype=np.int32) for k in libs}
        Pf, Qf = np.asfortranarray(P), np.asfortranarray(Q)

        def fpfh(k):
            L = libs[k]
            L.psulvsb_fpfh(None, d.data_ptr(), n, rn, rf, None, work.data_ptr(), None, out[k][0].data_ptr())
            L.psulvsb_fpfh(None, dq.data_ptr(), n, rn, rf, None, work.data_ptr(), None, out[k][1].data_ptr())

        def nnf(k):
            libs[k].psulvsb_feature_nn(None, out[k][0].data_ptr(), n, out[k][1].data_ptr(), n, nn[k][0].data_ptr(),
                                       nn[k][1].data_ptr())

        fs_h = {k: out[k][0] for k in libs}
        cnt = {k: C.c_longlong(0) for k in libs}

        def match(k):
            a, b = fs_h[k][0], fs_h[k][1]
            libs[k].psulvsb_match_host(Pf.ctypes.data, n, Qf.ctypes.data, n, a.ctypes.data, b.ctypes.data, 1, 0, 0.95,
                                       0, pairs[k].ctypes.data, n, C.byref(cnt[k]))

        for k in libs:
            fpfh(k)
        torch.cuda.synchronize()
        fs_h = {k: (out[k][0].cpu().numpy(), out[k][1].cpu().numpy()) for k in libs}
        for name, fn, reps in (("fpfh_x2", fpfh, min_reps), ("nn", nnf, min_reps), ("match_host", match, 5)):
            times = {k: [] for k in libs}
            for _ in range(rounds):
                for k in libs:
                    fn(k)
                    times[k].append(wall(lambda: fn(k), reps))
            torch.cuda.synchronize()
            if name == "fpfh_x2":
                same = all(torch.equal(out["parent"][i], out["new"][i]) for i in range(2))
            elif name == "nn":
                same = all(torch.equal(nn["parent"][i], nn["new"][i]) for i in range(2))
            else:
                same = cnt["parent"].value == cnt["new"].value and np.array_equal(pairs["parent"], pairs["new"])
            med = {k: float(np.median(v)) for k, v in times.items()}
            line = {"n": n, "call": name, "parent_ms": times["parent"], "new_ms": times["new"],
                    "new_over_parent": med["new"] / med["parent"],
                    "spread_parent": (max(times["parent"]) - min(times["parent"])) / med["parent"],
                    "spread_new": (max(times["new"]) - min(times["new"])) / med["new"], "identical": bool(same)}
            print(json.dumps(line), flush=True)
            lines.append(line)
    return lines


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_features_batch_bench.json"))
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small sizes only (a rehearsal of the script)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("features_batch_bench: no CUDA device (nothing is measured without one)")
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": smi("power.limit"),
           "sm_clock_max_mhz": smi("clocks.max.sm"), "sms": torch.cuda.get_device_properties(0).multi_processor_count}
    sizes = [(4, 1000, False)] if args.quick else [(64, 5000, False), (592, 5000, False), (16, 50000, False),
                                                   (64, 5000, True)]
    res["loop_vs_batch"] = [loop_vs_batch(B, n, t, args.rounds) for B, n, t in sizes]
    # the SM clock under load (an idle card reports a lower one): the roofline of the 66-slot unit cost at that clock
    clock = smi("clocks.sm")
    f_mhz = float(clock) if clock else float(res["sm_clock_max_mhz"] or 1965)
    roof = res["sms"] * 128 * f_mhz * 1e6 / UNIT_SLOTS
    res["nn_roofline_distances_per_s"] = roof
    for line in res["loop_vs_batch"]:
        if "match_batch_ms" in line:
            line["nn_of_roofline_upper_bound"] = line["distances"] / line["match_batch_ms"] * 1e3 / roof
    res["chain"] = chain(8 if args.quick else 592, args.rounds)
    if args.parent_lib:
        res["parent_vs_new"] = parent_compare(args.parent_lib, args.rounds)
    res["sm_clock_during_mhz"] = smi("clocks.sm")
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "power_limit_w", "sm_clock_during_mhz")}))


if __name__ == "__main__":
    main()
