"""Times the voxel filter (psulvsb_voxel_down_sample / _batch, csrc/k8_voxel.cu) and the raw-scan chain it opens.

Workload: the seeded synthetic surface (synth.make_surface, area about 4.6 over [0, 2]^2).  Lines:
* single calls at 50 000 and 500 000 points with voxel sizes for about 4, 64 and 1 000 points per voxel (the last is
  the coarse case where the in-bucket ranking and the first-of-voxel test, O(sum m^2), show); the achieved points per
  voxel are reported;
* 592 x 5 000 and 16 x 50 000 (about 16 points per voxel) in one batched call against a loop of single calls, outputs
  compared bit for bit in the run;
* the kernels, copies and memsets of one call, counted by torch.profiler;
* the device chain voxel_down_sample_batch -> fpfh_batch -> match_batch -> solve_batch -> icp_batch for 16 pairs of
  200 000 points (FPFH and matching on the voxels, ICP on the dense clouds), each stage timed between synchronisations,
  and FPFH plus the matcher on the same dense clouds without downsampling, at that one fixed size (no search for the
  largest size that fits);
* the numpy restatement (tests/voxel_restatement.py) on the host, at the single-call sizes.

CUDA events around back-to-back calls after a warm-up, at least `--min-seconds` of timed work per measurement, medians
of `--rounds` alternations; the device name, power limit and SM clock are read in the same run.

    python profiles/tools/voxel_bench.py [--out profiles/r10_voxel_bench.json]
"""
import argparse
import ctypes as C
import json
import os
import re
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import psulvsb_b200  # noqa: E402,F401
from icp_bench import smi, timed  # noqa: E402
from psulvsb_b200 import capi, features, icp, stages, synth  # noqa: E402
from tests import voxel_restatement as VR  # noqa: E402

AREA = 4.6


def voxel_for(n, per_voxel):
    return (per_voxel * AREA / n) ** 0.5


def med(xs):
    return float(np.median(xs))


def alternate(fns, rounds, min_seconds):
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            out[k].append(timed(fn, min_seconds)[0])
    return out


def count_launches(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
    kern = [x for x in names if "Memcpy" not in x and "Memset" not in x]
    return {"kernels": len(kern), "memcpy": sum(1 for x in names if "Memcpy" in x),
            "memset": sum(1 for x in names if "Memset" in x),
            "kernel_names": sorted({m.group(0) for x in kern for m in [re.search(r"k8_[a-z0-9_]+", x)] if m})}


class Single:
    """psulvsb_voxel_down_sample on preallocated device buffers."""

    def __init__(self, P, v):
        import torch

        self.L = capi.lib()
        self.n = P.shape[1]
        self.v = v
        self.d = stages.to_device_points(P)
        self.work = torch.empty(max(1, self.L.psulvsb_voxel_down_sample_workspace_bytes(self.n)), dtype=torch.uint8,
                                device="cuda")
        self.out = torch.empty((self.n, 3), dtype=torch.float64, device="cuda")
        self.cnt = torch.empty(1, dtype=torch.int32, device="cuda")

    def __call__(self):
        capi.check(self.L.psulvsb_voxel_down_sample(stages._stream(), self.d.data_ptr(), self.n, self.v,
                                                    self.work.data_ptr(), self.out.data_ptr(), self.cnt.data_ptr()))

    def result(self):
        return self.out[:int(self.cnt.item())].cpu().numpy()


class Batch:
    def __init__(self, clouds, v):
        import torch

        self.L = capi.lib()
        self.v = v
        self.d = [stages.to_device_points(P) for P in clouds]
        self.sizes = [P.shape[1] for P in clouds]
        self.arr = features._clouds([t.data_ptr() for t in self.d], self.sizes, [(0.0, 0.0, 0.0)] * len(clouds))
        self.B = len(clouds)
        self.work = torch.empty(max(1, self.L.psulvsb_voxel_down_sample_batch_workspace_bytes(self.arr, self.B)),
                                dtype=torch.uint8, device="cuda")
        self.out = torch.empty((sum(self.sizes), 3), dtype=torch.float64, device="cuda")
        self.cnt = torch.empty(self.B, dtype=torch.int32, device="cuda")

    def __call__(self):
        capi.check(self.L.psulvsb_voxel_down_sample_batch(stages._stream(), self.arr, self.B, self.v,
                                                          self.work.data_ptr(), self.out.data_ptr(),
                                                          self.cnt.data_ptr()))

    def results(self):
        out, cnt = self.out.cpu().numpy(), self.cnt.cpu().numpy()
        offs = np.concatenate([[0], np.cumsum(self.sizes)])
        return [out[offs[c]:offs[c] + cnt[c]] for c in range(self.B)]


def single_lines(rounds, min_seconds):
    out = []
    for n in (50000, 500000):
        P = synth.make_surface(n, 7)
        for k in (4, 64, 1000):
            v = voxel_for(n, k)
            s = Single(P, v)
            t = alternate({"call": s}, rounds, min_seconds)["call"]
            got = s.result()
            t0 = time.perf_counter()
            want = VR.voxel_down_sample(P, v)
            t_np = (time.perf_counter() - t0) * 1e3
            assert np.array_equal(got, want.T), (n, k)
            out.append({"n": n, "target_points_per_voxel": k, "voxel_size": v, "voxels": int(got.shape[0]),
                        "points_per_voxel": n / got.shape[0], "max_voxels_per_bucket": VR.voxels_per_bucket(P, v),
                        "ms": med(t), "ms_rounds": t, "numpy_restatement_ms": t_np, "equals_restatement": True})
            print(json.dumps(out[-1]), flush=True)
    return out


def batch_lines(rounds, min_seconds):
    out = []
    for B, n in ((592, 5000), (16, 50000)):
        clouds = [synth.make_surface(n, b) for b in range(B)]
        v = voxel_for(n, 16)
        bat = Batch(clouds, v)
        singles = [Single(P, v) for P in clouds]

        def loop():
            for s in singles:
                s()

        t = alternate({"batch": bat, "loop": loop}, rounds, min_seconds)
        got = bat.results()
        same = all(np.array_equal(g, s.result()) for g, s in zip(got, singles))
        assert same
        out.append({"B": B, "n": n, "voxel_size": v, "voxels": int(sum(g.shape[0] for g in got)),
                    "batch_ms": med(t["batch"]), "loop_ms": med(t["loop"]), "speedup": med(t["loop"]) / med(t["batch"]),
                    "batch_ms_rounds": t["batch"], "loop_ms_rounds": t["loop"], "identical_to_single_calls": same,
                    "launches_batch_call": count_launches(bat), "launches_single_call": count_launches(singles[0])})
        print(json.dumps(out[-1]), flush=True)
    return out


def chain_line(reps):
    """16 pairs of 200 000 points; FPFH radii 2 v and 5 v on the voxels, ICP on the dense clouds (d = v)."""
    import torch

    B, n, v = 16, 200000, 0.04
    src = synth.make_surface(n, 31)
    tgts, truth = [], []
    for b in range(B):
        R, _ = synth.random_rigid(np.random.default_rng(100 + b))
        t = np.array([0.4, -0.3, 0.2])
        tgts.append((R @ src + t[:, None])[:, np.random.default_rng(200 + b).permutation(n)])
        truth.append((R, t))
    d_src = stages.to_device_points(src)
    d_tgt = [stages.to_device_points(T) for T in tgts]
    kw = dict(noise_bound=1.5 * v, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005, wallclock_cap_s=0.0,
              seed=1)
    handle = capi.Handle(0)

    def stage(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return r, (time.perf_counter() - t0) * 1e3

    def run():
        times = {}
        (allv, counts, offs), times["voxel_down_sample_batch"] = stage(
            lambda: features.voxel_down_sample_batch_device([d_src] + d_tgt, v))
        cnt = counts.cpu().numpy()
        vox = [allv[int(o):int(o) + int(c)] for o, c in zip(offs, cnt)]
        (fe, _, views), times["fpfh_batch"] = stage(lambda: features.fpfh_batch_device(vox, 2.0 * v, 5.0 * v))
        fs = views[0][0]
        (pairs, pc, po), times["match_batch"] = stage(lambda: features.match_batch_device(
            [vox[0]] * B, vox[1:], [fs] * B, [f for f, _ in views[1:]], crosscheck=True))
        pc, po = pc.cpu().numpy(), po
        pr = pairs.cpu().numpy()
        s_h = vox[0].cpu().numpy().T
        problems = []
        for b in range(B):
            m = pr[int(po[b]):int(po[b]) + int(pc[b])]
            problems.append(capi.HostProblem(s_h[:, m[:, 0]], vox[b + 1].cpu().numpy().T[:, m[:, 1]]))
        sols, times["solve_batch"] = stage(lambda: handle.solve_batch(capi.default_params(**kw), problems))
        res, times["icp_batch"] = stage(lambda: icp.icp_batch_device([d_src] * B, d_tgt, np.array([s.R for s in sols]),
                                                                    np.array([s.t for s in sols]), v,
                                                                    max_iterations=60))
        err = [(synth.rotation_error(o.R, R), float(np.linalg.norm(o.t - t))) for o, (R, t) in zip(res, truth)]
        return times, cnt, pc, err

    run()
    runs = [run() for _ in range(reps)]
    stages_ms = {k: med([r[0][k] for r in runs]) for k in runs[0][0]}
    total = sum(stages_ms.values())
    times, cnt, pc, err = runs[-1]
    line = {"B": B, "n": n, "voxel_size": v, "voxels_per_cloud": [int(c) for c in cnt],
            "correspondences": [int(c) for c in pc], "stage_ms": stages_ms, "total_ms": total,
            "voxel_share": stages_ms["voxel_down_sample_batch"] / total,
            "max_rotation_error_rad": max(e[0] for e in err), "max_translation_error": max(e[1] for e in err),
            "note": "stages timed between synchronisations; the match stage's counts and the solver's problems go "
                    "through the host"}
    print(json.dumps(line), flush=True)
    # FPFH and the matcher on the same 16 x 200 000 dense clouds, without downsampling (radii scaled to the spacing)
    s = (5000.0 / n) ** 0.5
    (fe, _, views), t_f = stage(lambda: features.fpfh_batch_device([d_src] + d_tgt, 0.06 * s, 0.1 * s))
    fs = views[0][0]
    mfn = lambda: features.match_batch_device([d_src] * B, d_tgt, [fs] * B, [f for f, _ in views[1:]],  # noqa: E731
                                              crosscheck=True)
    stage(mfn)
    _, t_m = stage(mfn)
    line["dense_without_downsampling"] = {"fpfh_batch_ms": t_f, "match_batch_ms": t_m, "B": B, "n": n}
    print(json.dumps(line["dense_without_downsampling"]), flush=True)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_voxel_bench.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--chain-reps", type=int, default=3)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("voxel_bench.py measures on the GPU; no CUDA device")
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": smi("power.limit"),
           "sm_clock_mhz": smi("clocks.sm"), "sm_clock_max_mhz": smi("clocks.max.sm"),
           "method": f"CUDA events, >= {a.min_seconds} s of back-to-back calls per measurement after warm-up, medians "
                     f"of {a.rounds} alternations"}
    print(json.dumps(res), flush=True)
    res["single"] = single_lines(a.rounds, a.min_seconds)
    res["batch"] = batch_lines(a.rounds, a.min_seconds)
    res["chain"] = chain_line(a.chain_reps)
    res["sm_clock_mhz_end"] = smi("clocks.sm")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
