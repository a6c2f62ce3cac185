"""The ICP refinement on the GPU against the numpy restatement (oracle/icp.py): step-locked on every trace record,
determinism, edge shapes, and registration from raw clouds end to end (Python and the C++ example)."""
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial import cKDTree

import psulvsb_b200  # noqa: F401
from oracle import icp as OI
from psulvsb_b200 import capi, features, icp, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bunny():
    return np.load(os.path.join(ROOT, "tests", "golden", "bunny_res3.npz"))["vertices"].astype(np.float64) * 10


def extent(P):
    return float(np.linalg.norm(np.ptp(P, axis=1)))


def spacing(P):
    return float(cKDTree(P.T).query(P.T, k=2)[0][:, 1].mean())


def perturbed(R, t, rng, angle_deg, shift):
    axis = rng.normal(size=3)
    axis /= np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    a = np.deg2rad(angle_deg)
    return (np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K) @ R, t + shift * rng.normal(size=3) / np.sqrt(3)


def scene(P, seed):
    """Source: P with noise (sigma = 0.002 extent) and 10 % of its points replaced by outliers without a counterpart;
    target: the transformed cloud cropped to about 70 % overlap.  Returns src, tgt, R, t, T0 = the truth moved by 2
    degrees and 1 % of the extent, and d = 3 mean spacings."""
    rng = np.random.default_rng(seed)
    ext = extent(P)
    R, _ = synth.random_rigid(rng)
    t = rng.normal(size=3) * 0.3 * ext
    src = P + rng.normal(0, 0.002 * ext, P.shape)
    out = rng.random(P.shape[1]) < 0.1
    lo, hi = P.min(axis=1), P.max(axis=1)
    src[:, out] = rng.uniform(lo[:, None], hi[:, None], (3, int(out.sum())))
    keep = P[0] <= np.quantile(P[0], 0.7)
    tgt = R @ P[:, keep] + t[:, None]
    R0, t0 = perturbed(R, t, rng, 2.0, 0.01 * ext)
    return src, tgt, R, t, R0, t0, 3.0 * spacing(P)


def check_step_locked(src, tgt, d, out, *, normals=None, point_to_plane=False, max_iterations=30,
                      relative_fitness=1e-6, relative_rmse=1e-6):
    """Every trace record k against the restatement evaluated at the GPU's T_k; the stop rule applied to the trace."""
    tr = out.trace
    K = len(tr["fitness"])
    assert K == out.iterations + 1
    # t_u = mu_q - R_u mu_p carries R_u's last bits times the clouds' distance from the origin
    scale = max(extent(tgt), np.abs(tgt).max(initial=0.0), 1e-300)
    keep = OI.candidate_mask(tgt, normals if point_to_plane else None)
    tree = cKDTree(tgt[:, keep].T) if keep.any() else None
    prev = None
    for k in range(K):
        chk = OI.step_check(src, tgt, d, tr["R"][k], tr["t"][k], normals=normals, point_to_plane=point_to_plane,
                            tree=tree)
        assert tr["n_correspondences"][k] == chk["n_corr"], k
        assert tr["fitness"][k] == chk["fitness"], k
        assert abs(tr["inlier_rmse"][k] - chk["inlier_rmse"]) <= 1e-12 * chk["inlier_rmse"], k
        cur = (tr["fitness"][k], tr["inlier_rmse"][k])
        status = OI.stop(k, prev, cur, max_iterations, relative_fitness, relative_rmse)
        if k < K - 1:
            assert status is None and chk["next"] is not None, k
            Rn, tn = chk["next"]
            assert np.abs(tr["R"][k + 1] - Rn).max() <= 1e-10, (k, np.abs(tr["R"][k + 1] - Rn).max())
            assert np.abs(tr["t"][k + 1] - tn).max() <= 1e-10 * scale, (k, np.abs(tr["t"][k + 1] - tn).max())
        else:
            if status is None:
                assert chk["next"] is None
                status = OI.NO_UPDATE
            assert out.status == status
            assert np.array_equal(out.correspondences, chk["corr"])
            assert np.array_equal(out.R, tr["R"][k]) and np.array_equal(out.t, tr["t"][k])
            assert out.fitness == cur[0] and out.inlier_rmse == cur[1] and out.n_correspondences == chk["n_corr"]
        prev = cur


def radius_normals(Q, rn):
    return features.fpfh(Q, rn, 2 * rn)[1]


CLOUDS = {"bunny": lambda b: b, "surface": lambda b: synth.make_surface(50_000, 4)}


@pytest.mark.parametrize("cloud", ["bunny", "surface"])
@pytest.mark.parametrize("point_to_plane", [False, True])
def test_step_locked_vs_restatement(bunny, cloud, point_to_plane):
    P = CLOUDS[cloud](bunny)
    src, tgt, R, t, R0, t0, d = scene(P, 21 if cloud == "bunny" else 22)
    N = radius_normals(tgt, 4 * spacing(P)) if point_to_plane else None
    out = icp.icp(src, tgt, R0, t0, d, target_normals=N, point_to_plane=point_to_plane, trace=True)
    check_step_locked(src, tgt, d, out, normals=N, point_to_plane=point_to_plane)
    assert out.iterations >= 2 and out.fitness > 0.4        # at most 0.9 x 0.7: outliers and the crop
    if point_to_plane:
        assert np.isfinite(N[:, out.correspondences[out.correspondences >= 0]]).all()
    # the correspondences of the intermediate records: a shorter call reproduces the trace's prefix bit for bit
    for k in (0, 1):
        part = icp.icp(src, tgt, R0, t0, d, target_normals=N, point_to_plane=point_to_plane, max_iterations=k,
                       trace=True)
        assert np.array_equal(part.trace["R"], out.trace["R"][:k + 1])
        assert np.array_equal(part.trace["t"], out.trace["t"][:k + 1])
        want, _ = OI.correspond(OI.transform(src, part.R, part.t), tgt, d, N if point_to_plane else None)
        assert np.array_equal(part.correspondences, want) and part.status == OI.MAX_ITERATIONS


def test_determinism_host_device_and_dirty_workspace(bunny):
    import torch

    from psulvsb_b200 import stages

    src, tgt, R, t, R0, t0, d = scene(bunny, 31)
    N = radius_normals(tgt, 0.1)
    for p2l in (False, True):
        kw = dict(target_normals=N, point_to_plane=p2l, trace=True, relative_fitness=0, relative_rmse=0,
                  max_iterations=12)
        a, b = icp.icp(src, tgt, R0, t0, d, **kw), icp.icp(src, tgt, R0, t0, d, **kw)
        assert np.array_equal(a.R, b.R) and np.array_equal(a.t, b.t) and a.inlier_rmse == b.inlier_rmse
        assert np.array_equal(a.correspondences, b.correspondences)
        assert all(np.array_equal(a.trace[k], b.trace[k]) for k in a.trace)
        ds, dt, dn = stages.to_device_points(src), stages.to_device_points(tgt), stages.to_device_points(N)
        side = torch.cuda.Stream()
        nbytes = capi.lib().psulvsb_icp_workspace_bytes(src.shape[1], tgt.shape[1])
        work = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, device="cuda")
        for _ in range(2):                          # the second call finds the first one's leftovers
            with torch.cuda.stream(side):
                c = icp.icp_device(ds, dt, R0, t0, d, d_target_normals=dn, point_to_plane=p2l, trace=True,
                                   relative_fitness=0, relative_rmse=0, max_iterations=12, work=work)
            side.synchronize()
            assert np.array_equal(c.R, a.R) and np.array_equal(c.t, a.t) and c.fitness == a.fitness
            assert np.array_equal(c.correspondences.cpu().numpy(), a.correspondences)
            assert all(np.array_equal(c.trace[k], a.trace[k]) for k in a.trace)
        assert a.status == OI.MAX_ITERATIONS and a.iterations == 12


def test_empty_and_tiny_clouds(bunny):
    R0, t0 = synth.random_rigid(np.random.default_rng(3))[0], np.array([0.1, 0.2, 0.3])
    P = bunny[:, :50]
    for s, q in ((P[:, :0], P), (P, P[:, :0]), (P[:, :0], P[:, :0])):
        out = icp.icp(s, q, R0, t0, 0.1, trace=True)
        assert out.status == OI.NO_UPDATE and out.iterations == 0 and out.fitness == 0.0 and out.n_correspondences == 0
        assert np.array_equal(out.R, R0) and np.array_equal(out.t, t0) and len(out.trace["fitness"]) == 1
        assert (out.correspondences == -1).all() and out.correspondences.size == s.shape[1]
    Q = R0 @ P + t0[:, None]
    for n in (1, 2):
        out = icp.icp(P[:, :n], Q, R0, t0, 0.1, trace=True)
        assert out.status == OI.NO_UPDATE and out.iterations == 0 and out.n_correspondences == n
        assert out.correspondences.tolist() == list(range(n))
    out = icp.icp(P, Q, R0, t0, 0.1, max_iterations=0, trace=True)
    assert out.status == OI.MAX_ITERATIONS and out.iterations == 0 and out.fitness == 1.0
    assert np.array_equal(out.trace["R"][0], R0) and np.array_equal(out.trace["t"][0], t0)


@pytest.mark.parametrize("point_to_plane", [False, True])
def test_whole_target_in_a_handful_of_cells(bunny, point_to_plane):
    P = bunny[:, ::4]
    src, tgt, R, t, R0, t0, _ = scene(P, 41)
    d = extent(P)                                     # h ~ the extent: the target spans a few cells
    N = radius_normals(tgt, 0.15) if point_to_plane else None
    out = icp.icp(src, tgt, R0, t0, d, target_normals=N, point_to_plane=point_to_plane, max_iterations=5, trace=True)
    check_step_locked(src, tgt, d, out, normals=N, point_to_plane=point_to_plane, max_iterations=5)


def test_far_from_the_origin(bunny):
    P = bunny[:, ::2]
    src, tgt, R, t, R0, t0, d = scene(P, 51)
    off = 1e6 * d * np.array([1.0, -0.7, 0.4])
    src, tgt = src + off[:, None], tgt + off[:, None]
    t0 = t0 + off - R0 @ off                            # the same motion expressed around the offset
    out = icp.icp(src, tgt, R0, t0, d, max_iterations=8, trace=True)
    check_step_locked(src, tgt, d, out, max_iterations=8)
    # every pair within d is found: brute force at the final T
    Pp = OI.transform(src, out.R, out.t)
    D = ((tgt[0][None] - Pp[0][:, None]) ** 2 + (tgt[1][None] - Pp[1][:, None]) ** 2) + (tgt[2][None] - Pp[2][:, None]) ** 2
    has = (D <= d * d).any(axis=1)
    assert np.array_equal(out.correspondences >= 0, has) and out.n_correspondences > 0.3 * src.shape[1]


@pytest.mark.parametrize("nt", [1, 3, 5, 9, 17])
def test_hash_colliding_buckets(nt):
    """A target of a few points has 1 to 32 buckets: the 27 cells of a query collide, and every bucket is visited
    once."""
    rng = np.random.default_rng(nt)
    tgt = rng.uniform(0, 1, (3, nt))
    src = np.concatenate([tgt + rng.normal(0, 0.05, tgt.shape), rng.uniform(-0.5, 1.5, (3, 400))], axis=1)
    out = icp.icp(src, tgt, np.eye(3), np.zeros(3), 0.3, max_iterations=0, trace=True)
    want, d2 = OI.correspond(src, tgt, 0.3)
    assert np.array_equal(out.correspondences, want)
    n, fit, rmse = OI.evaluate(want, d2)
    assert out.n_correspondences == n and out.fitness == fit and abs(out.inlier_rmse - rmse) <= 1e-12 * rmse


def test_point_to_plane_with_nan_radius_normals():
    P = synth.make_surface(20_000, 6)
    rng = np.random.default_rng(7)
    iso = rng.uniform(3.0, 4.0, (3, 200))               # isolated target points: fewer than 3 neighbours, NaN normals
    src, tgt, R, t, R0, t0, d = scene(P, 61)
    tgt = np.concatenate([tgt, R @ iso + t[:, None]], axis=1)
    src = np.concatenate([src, iso + rng.normal(0, 1e-3, iso.shape)], axis=1)
    N = radius_normals(tgt, 4 * spacing(P))
    bad = ~np.isfinite(N).all(axis=0)
    assert bad[-200:].all()
    out = icp.icp(src, tgt, R0, t0, d, target_normals=N, point_to_plane=True, trace=True)
    check_step_locked(src, tgt, d, out, normals=N, point_to_plane=True)
    c = out.correspondences
    assert not bad[c[c >= 0]].any()
    assert (c[-200:] == -1).all()                        # their only counterparts have NaN normals


def registration(bunny, noise, seed):
    """bunny -> FPFH -> match -> solve; the solve's R, t and the clouds."""
    R, _ = synth.random_rigid(np.random.default_rng(seed))
    t = np.array([0.4, -0.3, 0.2])
    n = bunny.shape[1]
    perm = np.random.default_rng(seed + 1).permutation(n)
    tgt = (R @ bunny + t[:, None])[:, perm]
    ext = extent(bunny)
    if noise:
        tgt = tgt + np.random.default_rng(seed + 2).normal(0, noise * ext, tgt.shape)
    fs, _ = features.fpfh(bunny, 0.08, 0.15)
    ft, _ = features.fpfh(tgt, 0.08, 0.15, viewpoint=t)
    pairs = features.match(bunny, tgt, fs, ft, crosscheck=True)
    kw = dict(noise_bound=0.01 * ext, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005,
              wallclock_cap_s=0.0, seed=1)
    sol, _ = capi.Handle(0).solve(capi.default_params(**kw), capi.HostProblem(bunny[:, pairs[:, 0]],
                                                                              tgt[:, pairs[:, 1]]))
    assert sol.valid
    return R, t, tgt, sol.R, sol.t, ext


def test_end_to_end_bunny_noise_free(bunny):
    R, t, tgt, Rs, ts, ext = registration(bunny, 0.0, 12)
    d = 3.0 * spacing(bunny)                            # three mean point spacings
    out = icp.icp(bunny, tgt, Rs, ts, d, max_iterations=100, relative_fitness=1e-12, relative_rmse=1e-12)
    print("solve", synth.rotation_error(Rs, R), np.linalg.norm(ts - t), "icp", synth.rotation_error(out.R, R),
          np.linalg.norm(out.t - t), out.fitness, out.iterations, out.status, "d", d)
    assert synth.rotation_error(out.R, R) <= 1e-6
    assert np.linalg.norm(out.t - t) <= 1e-6 * ext
    assert out.fitness == 1.0


def test_end_to_end_bunny_with_noise(bunny):
    R, t, tgt, Rs, ts, ext = registration(bunny, 0.002, 14)
    d = 3.0 * spacing(bunny)
    out = icp.icp(bunny, tgt, Rs, ts, d)
    print("solve", synth.rotation_error(Rs, R), np.linalg.norm(ts - t), "icp", synth.rotation_error(out.R, R),
          np.linalg.norm(out.t - t), out.fitness, out.iterations, out.status)
    assert synth.rotation_error(out.R, R) <= synth.rotation_error(Rs, R)
    assert np.linalg.norm(out.t - t) <= np.linalg.norm(ts - t)


def test_example_binary_refines_with_icp(tmp_path):
    from tests.test_cpp_facade import write_bunny_ply

    exe = str(tmp_path / "psulvsb_fpfh")
    libdir = os.path.dirname(capi.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
                           "-I", os.path.join(ROOT, "tests", "shim"), os.path.join(ROOT, "examples", "psulvsb_fpfh.cc"),
                           "-o", exe, "-L", libdir, "-l:libpsulvsb_b200.so", "-Wl,-rpath," + libdir])
    ply = str(tmp_path / "bunny.ply")
    write_bunny_ply(ply)
    base = subprocess.run([exe, ply, "10", "0.08", "0.15"], capture_output=True, text=True, timeout=300)
    r = subprocess.run([exe, ply, "10", "0.08", "0.15", "0", "1", "0.15"], capture_output=True, text=True, timeout=300)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
    first, second = r.stdout.splitlines()
    assert first == base.stdout.strip()                # the first line is today's output
    assert second.startswith("icp: fitness=")
    rot = float(first.split("rotation_error_deg=")[1].split()[0])
    rot_icp = float(second.split("rotation_error_deg=")[1].split()[0])
    assert rot_icp < rot, r.stdout
