"""Times the colour-carrying voxel filter (psulvsb_voxel_down_sample_colors*, csrc/k8_voxel_colors.cu) and multi-scale
colored ICP (icp.multiscale_colored_icp_batch_device).

Lines:
* the colour filter against the plain one, alternated, at 50 000 and 500 000 points of the seeded synthetic surface
  with voxel sizes for about 3.5, 45 and 650 points per voxel, and for 592 x 5 000 and 16 x 50 000 in one batched call;
  the points and counts are checked equal to the plain call's and the colours to tests/voxel_colors_restatement.py's,
  bit for bit, in the run;
* with --parent-lib, the plain filter of the parent build against this build, alternated in one process at the same
  single-call sizes, outputs compared bit for bit;
* the pyramid (3 scales, v, v/2, v/4; 50, 30 and 14 iterations as Open3D's tutorial) against colored ICP at the finest
  voxel size alone and on the dense clouds (target normals radius 2 v/4, 30 points; d = v/4), from one common start
  (the truth moved 2.5 fine voxels along z), for one pair of 500 000 points and 16 pairs of 200 000 points of the
  coloured patch of tests/multiscale_colored_icp_restatement.py: the time of each stage per scale (filter, normals,
  colored ICP; each between synchronisations), the total of the library call, iterations and final errors.

CUDA events around back-to-back calls after a warm-up (filter lines), host clocks around synchronised work (pyramid
lines); medians over `--rounds` alternations; the device name, power limit and SM clock are read in the same run.

    python profiles/tools/multiscale_colored_icp_bench.py [--out profiles/r15_multiscale_colored_icp_bench.json]
        [--parent-lib PATH/libpsulvsb_b200.so]
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
from psulvsb_b200 import capi, features, icp, stages, synth  # noqa: E402
from tests import multiscale_colored_icp_restatement as MR  # noqa: E402
from tests import voxel_colors_restatement as VCR  # noqa: E402

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


class Filter:
    """One batched call of the plain (colors None) or the colour filter on preallocated device buffers; lib: the
    library to call (this build by default)."""

    def __init__(self, clouds, cols, v, lib=None, colors=True):
        import torch

        self.L = lib or capi.lib()
        self.v, self.colors, self.B = v, colors, len(clouds)
        self.d = [stages.to_device_points(P) for P in clouds]
        self.dc = [stages.to_device_points(K) for K in cols]
        self.sizes = [P.shape[1] for P in clouds]
        if colors:
            self.arr = features._color_clouds([(p.data_ptr(), c.data_ptr(), None) for p, c in zip(self.d, self.dc)],
                                              self.sizes)
            nb = self.L.psulvsb_voxel_down_sample_colors_batch_workspace_bytes(self.arr, self.B)
        else:
            self.arr = features._clouds([p.data_ptr() for p in self.d], self.sizes, [(0.0, 0.0, 0.0)] * self.B)
            nb = self.L.psulvsb_voxel_down_sample_batch_workspace_bytes(self.arr, self.B)
        N = sum(self.sizes)
        self.work = torch.empty(max(1, nb), dtype=torch.uint8, device="cuda")
        self.out = torch.empty((N, 3), dtype=torch.float64, device="cuda")
        self.oc = torch.empty((N, 3), dtype=torch.float64, device="cuda")
        self.cnt = torch.empty(self.B, dtype=torch.int32, device="cuda")

    def __call__(self):
        if self.colors:
            capi.check(self.L.psulvsb_voxel_down_sample_colors_batch(
                stages._stream(), self.arr, self.B, self.v, self.work.data_ptr(), self.out.data_ptr(),
                self.oc.data_ptr(), self.cnt.data_ptr()))
        else:
            capi.check(self.L.psulvsb_voxel_down_sample_batch(stages._stream(), self.arr, self.B, self.v,
                                                              self.work.data_ptr(), self.out.data_ptr(),
                                                              self.cnt.data_ptr()))

    def results(self):
        out, oc, cnt = self.out.cpu().numpy(), self.oc.cpu().numpy(), self.cnt.cpu().numpy()
        offs = np.concatenate([[0], np.cumsum(self.sizes)])
        return [(out[offs[c]:offs[c] + cnt[c]].T, oc[offs[c]:offs[c] + cnt[c]].T) for c in range(self.B)]


def colours(P, seed):
    return np.random.default_rng(seed).uniform(0.0, 1.0, P.shape)


def filter_lines(rounds, min_seconds):
    out = []
    shapes = [(1, 50000, k) for k in (3.5, 45, 650)] + [(1, 500000, k) for k in (3.5, 45, 650)] + \
        [(592, 5000, 16), (16, 50000, 16)]
    for B, n, k in shapes:
        clouds = [synth.make_surface(n, 7 + b) for b in range(B)]
        cols = [colours(P, b) for b, P in enumerate(clouds)]
        v = voxel_for(n, k)
        col, plain = Filter(clouds, cols, v), Filter(clouds, cols, v, colors=False)
        t = alternate({"colors": col, "plain": plain}, rounds, min_seconds)
        got, ref = col.results(), plain.results()
        assert all(np.array_equal(g[0], r[0]) for g, r in zip(got, ref))
        for c in range(0, B, max(1, B // 8)):
            wv, wc = VCR.voxel_down_sample_colors(clouds[c], cols[c], v)
            assert np.array_equal(got[c][0], wv) and np.array_equal(got[c][1], wc), (B, n, k, c)
        vox = sum(g[0].shape[1] for g in got)
        out.append({"B": B, "n": n, "target_points_per_voxel": k, "voxel_size": v, "voxels": int(vox),
                    "points_per_voxel": B * n / vox, "colors_ms": med(t["colors"]), "plain_ms": med(t["plain"]),
                    "ratio": med(t["colors"]) / med(t["plain"]), "colors_ms_rounds": t["colors"],
                    "plain_ms_rounds": t["plain"], "points_equal_plain": True, "colours_equal_restatement": True})
        print(json.dumps(out[-1]), flush=True)
    return out


def parent_lines(path, rounds, min_seconds):
    P = C.CDLL(path)
    P.psulvsb_voxel_down_sample_batch_workspace_bytes.argtypes = [C.POINTER(capi.FpfhCloud), C.c_int]
    P.psulvsb_voxel_down_sample_batch_workspace_bytes.restype = C.c_ulonglong
    P.psulvsb_voxel_down_sample_batch.argtypes = [C.c_void_p, C.POINTER(capi.FpfhCloud), C.c_int, C.c_double,
                                                  C.c_void_p, C.c_void_p, C.c_void_p]
    out = []
    for B, n, k in [(1, 50000, k) for k in (3.5, 45, 650)] + [(1, 500000, k) for k in (3.5, 45, 650)] + \
            [(592, 5000, 16)]:
        clouds = [synth.make_surface(n, 7 + b) for b in range(B)]
        v = voxel_for(n, k)
        new, old = Filter(clouds, clouds, v, colors=False), Filter(clouds, clouds, v, lib=P, colors=False)
        t = alternate({"parent": old, "new": new}, rounds, min_seconds)
        same = all(np.array_equal(a[0], b[0]) for a, b in zip(new.results(), old.results()))
        assert same
        out.append({"B": B, "n": n, "target_points_per_voxel": k, "parent_ms": med(t["parent"]),
                    "new_ms": med(t["new"]), "ratio": med(t["new"]) / med(t["parent"]),
                    "parent_ms_rounds": t["parent"], "new_ms_rounds": t["new"], "identical_outputs": same})
        print(json.dumps(out[-1]), flush=True)
    return out


def sync_ms(fn):
    import torch

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, (time.perf_counter() - t0) * 1e3


def pyramid_stages(d, R0, t0, scales, its):
    """multiscale_colored_icp_batch_device's loop with each stage timed between synchronisations."""
    B = len(d[0])
    R, t, rows, res = R0, t0, [], None
    for v, k in zip(scales, its):
        (vox, col, counts, offsets), tf = sync_ms(lambda: features.voxel_down_sample_batch_device(
            d[0] + d[1], v, colors=d[2] + d[3]))
        m = counts.cpu().numpy()
        vv = [vox[o:o + c] for o, c in zip(offsets, m)]
        cv = [col[o:o + c] for o, c in zip(offsets, m)]
        (_, nrm), tn = sync_ms(lambda: features.normals_batch_device(vv[B:], 2.0 * v, 30))
        res, ti = sync_ms(lambda: icp.colored_icp_batch_device(vv[:B], vv[B:], cv[:B], cv[B:], nrm, R, t, v,
                                                              max_iterations=k))
        R, t = np.array([r.R for r in res]), np.array([r.t for r in res])
        rows.append({"voxel_size": v, "voxels_src": int(m[:B].sum()), "voxels_tgt": int(m[B:].sum()),
                     "filter_ms": tf, "normals_ms": tn, "colored_icp_ms": ti,
                     "iterations": [r.iterations for r in res]})
    return rows, res


def errors(res, truth, fine):
    e = [MR.pose_errors(r.R, r.t, Rt, tt) for r, (Rt, tt) in zip(res, truth)]
    return {"max_deg": max(a for a, _ in e), "max_fine_spacings": max(b for _, b in e) / fine,
            "median_deg": med([a for a, _ in e]), "median_fine_spacings": med([b for _, b in e]) / fine,
            "n_correspondences": [r.n_correspondences for r in res], "status": [r.status for r in res]}


def pyramid_lines(reps):
    out = []
    for B, n, v in ((1, 500000, 0.04), (16, 200000, 0.06)):
        scales, its = (v, v / 2, v / 4), (50, 30, 14)
        fine = scales[-1]
        pairs = []
        for b in range(B):
            P, Q, Cs, Ct, Rt, tt, _, _ = MR.scene(seed=b, n=n)
            pairs.append((P, Q, Cs, Ct, Rt, tt))
        truth = [(p[4], p[5]) for p in pairs]
        R0 = np.array([np.eye(3)] * B)
        t0 = np.array([p[5] + np.array([0.0, 0.0, 2.5 * fine]) for p in pairs])
        d = [[stages.to_device_points(p[k]) for p in pairs] for k in range(4)]
        call = lambda: icp.multiscale_colored_icp_batch_device(*d, R0, t0, scales, max_iterations=its)  # noqa: E731
        call()
        totals = [sync_ms(call)[1] for _ in range(reps)]
        res = call()
        stage_runs = [pyramid_stages(d, R0, t0, scales, its) for _ in range(reps)]
        rows = stage_runs[-1][0]
        for s, row in enumerate(rows):
            for key in ("filter_ms", "normals_ms", "colored_icp_ms"):
                row[key] = med([r[0][s][key] for r in stage_runs])
        assert all(np.array_equal(a.R, b.R) for a, b in zip(res[-1], stage_runs[-1][1]))
        # colored ICP at the finest voxel size alone
        single = lambda: icp.multiscale_colored_icp_batch_device(*d, R0, t0, (fine,), max_iterations=50)  # noqa: E731
        single()
        t_single = [sync_ms(single)[1] for _ in range(reps)]
        r_single = single()[0]
        # colored ICP on the dense clouds (target normals radius 2 fine, 30 points)
        (_, dn), t_dn = sync_ms(lambda: features.normals_batch_device(d[1], 2.0 * fine, 30))

        def dense():
            return icp.colored_icp_batch_device(d[0], d[1], d[2], d[3], dn, R0, t0, fine, max_iterations=50)

        dense()
        t_dense = [sync_ms(dense)[1] for _ in range(reps)]
        r_dense = dense()
        out.append({"B": B, "n": n, "voxel_sizes": list(scales), "max_iterations": list(its),
                    "start": "truth moved 2.5 fine voxels along z",
                    "pyramid": {"total_ms": med(totals), "total_ms_runs": totals, "scales": rows,
                                "iterations": [[r.iterations for r in rs] for rs in res],
                                "errors": errors(res[-1], truth, fine)},
                    "finest_scale_alone": {"total_ms": med(t_single), "iterations": [r.iterations for r in r_single],
                                           "errors": errors(r_single, truth, fine)},
                    "dense": {"normals_ms": t_dn, "colored_icp_ms": med(t_dense),
                              "iterations": [r.iterations for r in r_dense], "errors": errors(r_dense, truth, fine)}})
        print(json.dumps(out[-1]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r15_multiscale_colored_icp_bench.json"))
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--min-seconds", type=float, default=0.3)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if capi.lib().psulvsb_device_count() < 1:
        raise SystemExit("no CUDA device: nothing is measured")
    rec = {"device": smi("name"), "power_limit_w": smi("power.limit"), "sm_clock_max_mhz": smi("clocks.max.sm"),
           "rounds": args.rounds, "min_seconds": args.min_seconds}
    print(json.dumps(rec), flush=True)
    rec["filter"] = filter_lines(args.rounds, args.min_seconds)
    if args.parent_lib:
        rec["plain_filter_parent_vs_new"] = parent_lines(args.parent_lib, args.rounds, args.min_seconds)
    rec["pyramid"] = pyramid_lines(args.reps)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
