"""Times the device-buffer upload of the batch solver (psulvsb_batch_upload_device, Handle.upload_device) against the
host upload (psulvsb_batch_upload / psulvsb_solve_batch) on the same arrays.  Lines:
* upload alone, followed by a device synchronisation: cfg-A inputs (592 x 5 000 correspondences, 95 % outliers) and
  cfg-B inputs (1 x 100 000, 99 %);
* upload plus solve_resident on the same two workloads;
* the raw-scan chain voxel_down_sample_batch_device -> fpfh_batch_device -> match_batch_device, then the solve from the
  matches: the host hop (pairs and voxels to the host, numpy gathers, HostProblem, solve_batch) against the device path
  (the B match counts to the host, DeviceProblem.from_matches, solve_batch_device), at 592 pairs of 5 000 points and at
  16 pairs of 200 000 points of the seeded surface.

A host clock around work that ends in a device synchronisation; every measurement is the median of `--reps` calls after
a warm-up, and every line the median of `--rounds` alternations of the two paths.  The solutions of the two paths are
compared field by field within the run.  The device name, power limit and SM clock are read in the same run.

    python profiles/tools/device_upload_bench.py [--out profiles/r12_device_upload_bench.json]
"""
import argparse
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
from icp_bench import smi  # noqa: E402
from psulvsb_b200 import capi, features, synth  # noqa: E402

PKW = dict(noise_bound=0.05, cbar2=1.0, estimate_scaling=0, rotation_max_iterations=100, rotation_gnc_factor=1.4,
           rotation_cost_threshold=0.005, wallclock_cap_s=0.0)


def identical(a, b):
    for x, y in zip(a, b):
        for name, _ in x._fields_:
            u, v = getattr(x, name), getattr(y, name)
            if np.array(u, dtype=np.float64).tobytes() != np.array(v, dtype=np.float64).tobytes():
                return False
    return len(a) == len(b)


def clock_ms(fn, reps):
    import torch

    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out))


def alternate(fns, rounds, reps):
    res = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            res[k].append(clock_ms(fn, reps))
    return {k: {"median_ms": float(np.median(v)), "rounds_ms": v} for k, v in res.items()}


def to_device(hp):
    import torch

    return capi.DeviceProblem(torch.from_numpy(np.ascontiguousarray(hp.src.T)).cuda(),
                              torch.from_numpy(np.ascontiguousarray(hp.dst.T)).cuda())


def upload_lines(h, name, host, rounds, reps):
    import torch

    dev = [to_device(p) for p in host]
    params = capi.default_params(seed=11, **PKW)
    ref = h.solve_batch(params, host)
    h.upload_device(dev)
    same = identical(ref, h.solve_resident(params))
    h.upload(host)
    same = same and identical(ref, h.solve_resident(params))
    up = alternate({"host": lambda: h.upload(host), "device": lambda: h.upload_device(dev)}, rounds, reps)
    # the C calls alone, on problem arrays built once (no Python per problem)
    L, arr_h, arr_d = capi.lib(), h._problem_array(host), h._problem_array(dev)
    stream = torch.cuda.current_stream().cuda_stream
    c_up = alternate({"host": lambda: capi.check(L.psulvsb_batch_upload(h._h, arr_h, len(host))),
                      "device": lambda: capi.check(L.psulvsb_batch_upload_device(h._h, stream, arr_d, len(dev)))},
                     rounds, reps)
    # device time of one device upload: the kernel and the copies, from torch.profiler
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        h.upload_device(dev)
        torch.cuda.synchronize()
    dev_us = {}
    for e in prof.key_averages():
        t = getattr(e, "self_device_time_total", 0.0) or 0.0
        if t > 0:
            key = "engine_upload_device_kernel" if "engine_upload_device_kernel" in e.key else e.key
            dev_us[key] = dev_us.get(key, 0.0) + float(t)

    def host_solve():
        h.upload(host)
        h.solve_resident(params)

    def dev_solve():
        h.upload_device(dev)
        h.solve_resident(params)

    solve = alternate({"host": host_solve, "device": dev_solve}, rounds, reps)
    mb = sum(p.nbytes for p in host) / 1e6
    return {"workload": name, "B": len(host), "bytes_MB": mb, "solutions_identical": bool(same), "upload": up,
            "upload_c_call_only": c_up, "device_upload_device_us": dev_us, "upload_plus_solve_resident": solve}


def chain_line(h, B, n, v, rounds, reps):
    import torch

    srcs, tgts = [], []
    for b in range(B):
        src = synth.make_surface(n, 60 + b)
        R, _ = synth.random_rigid(np.random.default_rng(80 + b))
        tgts.append((R @ src + np.array([0.4, -0.3, 0.2])[:, None])[:, np.random.default_rng(90 + b).permutation(n)])
        srcs.append(src)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a.T)).cuda()  # noqa: E731
    d_clouds = [d(a) for a in srcs + tgts]
    params = capi.default_params(seed=1, **dict(PKW, noise_bound=1.5 * v))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    vox, counts, offsets = features.voxel_down_sample_batch_device(d_clouds, v)
    counts = counts.cpu().numpy()
    down = [vox[int(o):int(o) + int(c)] for o, c in zip(offsets, counts)]
    _, _, views = features.fpfh_batch_device(down, 2.0 * v, 5.0 * v)
    pairs, mcounts, moff = features.match_batch_device(down[:B], down[B:], [f for f, _ in views[:B]],
                                                       [f for f, _ in views[B:]], crosscheck=True)
    torch.cuda.synchronize()
    front_ms = (time.perf_counter() - t0) * 1e3

    def host_hop():
        mc = mcounts.cpu().numpy()
        hv = [a.cpu().numpy().T for a in down]
        pr = pairs.cpu().numpy()
        probs = [capi.HostProblem(hv[b][:, pr[int(moff[b]):int(moff[b]) + int(mc[b]), 0]],
                                  hv[B + b][:, pr[int(moff[b]):int(moff[b]) + int(mc[b]), 1]]) for b in range(B)]
        return h.solve_batch(params, probs)

    def device_path():
        mc = mcounts.cpu().numpy()
        dev = [capi.DeviceProblem.from_matches(down[b], down[B + b], pairs[int(moff[b]):int(moff[b]) + int(mc[b])])
               for b in range(B)]
        return h.solve_batch_device(params, dev)

    same = identical(host_hop(), device_path())
    t = alternate({"host_hop": host_hop, "device": device_path}, rounds, reps)
    return {"workload": f"raw chain, {B} pairs of {n} points of the seeded surface, voxel {v}", "B": B, "n": n,
            "voxels_per_cloud_mean": float(np.mean(counts)),
            "matches_per_pair_mean": float(mcounts.double().mean().item()),
            "voxel_fpfh_match_ms_once": front_ms, "solve_from_matches": t, "solutions_identical": bool(same)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r12_device_upload_bench.json"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-chain", action="store_true")
    args = ap.parse_args()
    import torch

    if capi.lib().psulvsb_device_count() < 1:
        raise SystemExit("no CUDA device")
    out = {"device": smi("name"), "power_limit_W": smi("power.limit"), "sm_clock_MHz": smi("clocks.sm"),
           "sm_clock_max_MHz": smi("clocks.max.sm"), "timing": "host clock around calls that end in a device "
           "synchronisation; median of reps per round, median of rounds of alternation", "lines": []}
    h = capi.Handle(0)
    cfg_a = [capi.HostProblem(p["src"], p["dst"]) for p in
             (synth.make_pair(5000, 0.95, 1_000_000 + i) for i in range(592))]
    out["lines"].append(upload_lines(h, "cfg-A inputs: 592 x 5000 correspondences, 95% outliers", cfg_a, args.rounds,
                                     args.reps))
    print(json.dumps(out["lines"][-1]), flush=True)
    del cfg_a
    pb = synth.make_pair(100_000, 0.99, 4242, side=30.0)
    out["lines"].append(upload_lines(h, "cfg-B inputs: 1 x 100000 correspondences, 99% outliers",
                                     [capi.HostProblem(pb["src"], pb["dst"])], args.rounds, args.reps))
    print(json.dumps(out["lines"][-1]), flush=True)
    if not args.skip_chain:
        for B, n in ((592, 5000), (16, 200_000)):
            out["lines"].append(chain_line(h, B, n, 0.04, args.rounds, max(1, args.reps // 2)))
            print(json.dumps(out["lines"][-1]), flush=True)
    out["sm_clock_after_MHz"] = smi("clocks.sm")
    h.close()
    torch.cuda.synchronize()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
