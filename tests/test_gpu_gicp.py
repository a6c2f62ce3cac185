"""Generalized ICP on the GPU against the numpy restatement (tests/gicp_restatement.py): step-locked on every trace
record with k-NN and radius normals, edge normals, the sign and epsilon rules, edge shapes, determinism, batches, and
registration from raw clouds end to end."""
import os

import numpy as np
import pytest
from scipy.spatial import cKDTree

import psulvsb_b200  # noqa: F401
from oracle import icp as OI
from psulvsb_b200 import capi, features, icp, synth
from psulvsb_b200 import io as pio
from tests import gicp_restatement as G
from tests.test_gpu_icp import extent, registration, scene, spacing

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bunny():
    return np.load(os.path.join(ROOT, "tests", "golden", "bunny_res3.npz"))["vertices"].astype(np.float64) * 10


def check_step_locked(src, tgt, Ns, Nt, d, out, *, epsilon=1e-3, max_iterations=30, relative_fitness=1e-6,
                      relative_rmse=1e-6):
    """Every trace record k against the restatement evaluated at the GPU's T_k (test_gpu_icp.check_step_locked's
    tolerances); the stop rule applied to the trace."""
    tr = out.trace
    K = len(tr["fitness"])
    assert K == out.iterations + 1
    scale = max(extent(tgt), np.abs(tgt).max(initial=0.0), 1e-300)
    tree = cKDTree(tgt.T) if tgt.shape[1] else None
    prev = None
    for k in range(K):
        chk = G.step_check(src, tgt, Ns, Nt, d, tr["R"][k], tr["t"][k], epsilon, tree)
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


def same(a, b):
    return (np.array_equal(a.R, b.R) and np.array_equal(a.t, b.t) and a.fitness == b.fitness and
            a.inlier_rmse == b.inlier_rmse and a.status == b.status and a.iterations == b.iterations and
            np.array_equal(np.asarray(a.correspondences), np.asarray(b.correspondences)) and
            (a.trace is None) == (b.trace is None) and
            (a.trace is None or all(np.array_equal(a.trace[k], b.trace[k]) for k in a.trace)))


CLOUDS = {"bunny": lambda b: b, "surface": lambda b: synth.make_surface(50_000, 4)}


@pytest.mark.parametrize("cloud", ["bunny", "surface"])
@pytest.mark.parametrize("normals", ["knn", "radius"])
def test_step_locked_vs_restatement(bunny, cloud, normals):
    P = CLOUDS[cloud](bunny)
    src, tgt, R, t, R0, t0, d = scene(P, 21 if cloud == "bunny" else 22)
    if normals == "knn":
        Ns, Nt = pio.estimate_normals(src, 20), pio.estimate_normals(tgt, 20)
    else:
        rn = 4 * spacing(P)
        Ns, Nt = radius_normals(src, rn), radius_normals(tgt, rn)
    out = icp.gicp(src, tgt, Ns, Nt, R0, t0, d, trace=True)
    check_step_locked(src, tgt, Ns, Nt, d, out)
    assert out.iterations >= 2 and out.fitness > 0.4
    for k in (0, 1):                 # a shorter call reproduces the trace's prefix bit for bit
        part = icp.gicp(src, tgt, Ns, Nt, R0, t0, d, max_iterations=k, trace=True)
        assert np.array_equal(part.trace["R"], out.trace["R"][:k + 1])
        assert np.array_equal(part.trace["t"], out.trace["t"][:k + 1])
        want, _ = OI.correspond(OI.transform(src, part.R, part.t), tgt, d)
        assert np.array_equal(part.correspondences, want) and part.status == OI.MAX_ITERATIONS


def test_nan_radius_normals_on_both_sides_and_zero_normals():
    P = synth.make_surface(20_000, 6)
    rng = np.random.default_rng(7)
    iso = rng.uniform(3.0, 4.0, (3, 200))              # isolated points: fewer than 3 neighbours, NaN radius normals
    src, tgt, R, t, R0, t0, d = scene(P, 61)
    tgt = np.concatenate([tgt, R @ iso + t[:, None]], axis=1)
    src = np.concatenate([src, iso + rng.normal(0, 1e-3, iso.shape)], axis=1)
    rn = 4 * spacing(P)
    Ns, Nt = radius_normals(src, rn), radius_normals(tgt, rn)
    assert not np.isfinite(Ns[:, -200:]).any() and not np.isfinite(Nt[:, -200:]).any()
    out = icp.gicp(src, tgt, Ns, Nt, R0, t0, d, trace=True)
    check_step_locked(src, tgt, Ns, Nt, d, out)
    c = out.correspondences
    assert (c[-200:] >= 0).mean() > 0.9                 # they stay candidates (point-to-plane drops them)
    Ns0, Nt0 = Ns.copy(), Nt.copy()
    Ns0[:, ::7] = 0.0
    Nt0[:, 3::5] = 0.0
    out0 = icp.gicp(src, tgt, Ns0, Nt0, R0, t0, d, trace=True)
    check_step_locked(src, tgt, Ns0, Nt0, d, out0)


def test_normal_signs_do_not_matter_and_epsilon(bunny):
    src, tgt, R, t, R0, t0, d = scene(bunny, 23)
    Ns, Nt = pio.estimate_normals(src, 20), pio.estimate_normals(tgt, 20)
    rng = np.random.default_rng(1)
    fs, ft = np.where(rng.random(src.shape[1]) < 0.5, -1.0, 1.0), np.where(rng.random(tgt.shape[1]) < 0.5, -1.0, 1.0)
    kw = dict(trace=True, max_iterations=10, relative_fitness=0, relative_rmse=0)
    a = icp.gicp(src, tgt, Ns, Nt, R0, t0, d, **kw)
    b = icp.gicp(src, tgt, Ns * fs, Nt * ft, R0, t0, d, **kw)
    assert same(a, b)
    # both ends of epsilon's range: the linearised point-to-point step and nearly flat covariances
    for eps in (1.0, 1e-6):
        out = icp.gicp(src, tgt, Ns, Nt, R0, t0, d, epsilon=eps, trace=True)
        check_step_locked(src, tgt, Ns, Nt, d, out, epsilon=eps)
        assert out.iterations >= 2


def test_empty_tiny_and_zero_criteria(bunny):
    R0, t0 = synth.random_rigid(np.random.default_rng(3))[0], np.array([0.1, 0.2, 0.3])
    P = bunny[:, :50]
    N = np.tile(np.array([[0.0], [0.0], [1.0]]), (1, 50))
    for s, q in ((P[:, :0], P), (P, P[:, :0]), (P[:, :0], P[:, :0])):
        out = icp.gicp(s, q, N[:, :s.shape[1]], N[:, :q.shape[1]], R0, t0, 0.1, trace=True)
        assert out.status == OI.NO_UPDATE and out.iterations == 0 and out.fitness == 0.0 and out.n_correspondences == 0
        assert np.array_equal(out.R, R0) and np.array_equal(out.t, t0) and len(out.trace["fitness"]) == 1
        assert (out.correspondences == -1).all() and out.correspondences.size == s.shape[1]
    Q = R0 @ P + t0[:, None]
    for n in (1, 2):                                    # fewer than 3 correspondences: no update
        out = icp.gicp(P[:, :n], Q, N[:, :n], N, R0, t0, 0.1, trace=True)
        assert out.status == OI.NO_UPDATE and out.iterations == 0 and out.n_correspondences == n
        assert out.correspondences.tolist() == list(range(n))
    out = icp.gicp(P, Q, N, N, R0, t0, 0.1, max_iterations=0, trace=True)
    assert out.status == OI.MAX_ITERATIONS and out.iterations == 0 and out.fitness == 1.0
    src, tgt, R, t, R0, t0, d = scene(bunny[:, ::2], 24)
    Ns, Nt = pio.estimate_normals(src, 20), pio.estimate_normals(tgt, 20)
    out = icp.gicp(src, tgt, Ns, Nt, R0, t0, d, max_iterations=6, relative_fitness=0, relative_rmse=0, trace=True)
    assert out.status == OI.MAX_ITERATIONS and out.iterations == 6
    check_step_locked(src, tgt, Ns, Nt, d, out, max_iterations=6, relative_fitness=0, relative_rmse=0)


def test_far_from_the_origin(bunny):
    """300 d (about 30 extents) from the origin.  Open3D's Jacobian linearises the rotation about the origin, so the
    system's condition grows with (distance / extent)^2: from about 1e4 d on, the order of the sums alone moves the
    update by more than d and the loop diverges in numpy as on the GPU (DESIGN.md section 11, "Generalized ICP")."""
    P = bunny[:, ::2]
    src, tgt, R, t, R0, t0, d = scene(P, 51)
    Ns, Nt = pio.estimate_normals(src, 20), pio.estimate_normals(tgt, 20)
    off = 300 * d * np.array([1.0, -0.7, 0.4])
    src, tgt = src + off[:, None], tgt + off[:, None]
    t0 = t0 + off - R0 @ off
    out = icp.gicp(src, tgt, Ns, Nt, R0, t0, d, max_iterations=8, trace=True)
    check_step_locked(src, tgt, Ns, Nt, d, out, max_iterations=8)
    assert out.n_correspondences > 0.3 * src.shape[1]


@pytest.mark.parametrize("nt", [1, 3, 5, 9, 17])
def test_hash_colliding_buckets(nt):
    rng = np.random.default_rng(nt)
    tgt = rng.uniform(0, 1, (3, nt))
    src = np.concatenate([tgt + rng.normal(0, 0.05, tgt.shape), rng.uniform(-0.5, 1.5, (3, 400))], axis=1)
    Ns, Nt = rng.normal(size=src.shape), rng.normal(size=tgt.shape)
    out = icp.gicp(src, tgt, Ns, Nt, np.eye(3), np.zeros(3), 0.3, max_iterations=3, trace=True)
    check_step_locked(src, tgt, Ns, Nt, 0.3, out, max_iterations=3)


def test_determinism_host_device_and_dirty_workspace(bunny):
    import torch

    from psulvsb_b200 import stages

    src, tgt, R, t, R0, t0, d = scene(bunny, 31)
    Ns, Nt = radius_normals(src, 0.1), radius_normals(tgt, 0.1)
    kw = dict(trace=True, relative_fitness=0, relative_rmse=0, max_iterations=12)
    a, b = icp.gicp(src, tgt, Ns, Nt, R0, t0, d, **kw), icp.gicp(src, tgt, Ns, Nt, R0, t0, d, **kw)
    assert same(a, b)
    ds, dt = stages.to_device_points(src), stages.to_device_points(tgt)
    dns, dnt = stages.to_device_points(Ns), stages.to_device_points(Nt)
    side = torch.cuda.Stream()
    nbytes = capi.lib().psulvsb_icp_workspace_bytes(src.shape[1], tgt.shape[1])
    work = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    for _ in range(2):                              # the second call finds the first one's leftovers
        with torch.cuda.stream(side):
            c = icp.gicp_device(ds, dt, dns, dnt, R0, t0, d, work=work, **kw)
        side.synchronize()
        c.correspondences = c.correspondences.cpu().numpy()
        assert same(c, a)
    assert a.status == OI.MAX_ITERATIONS and a.iterations == 12


def mixed_batch(bunny):
    """(src, tgt, Ns, Nt, R0, t0) of an empty, tiny, far-away and 50k pair, and d."""
    items = []
    rng = np.random.default_rng(5)
    P = bunny[:, :40]
    N = rng.normal(size=P.shape)
    items.append((P[:, :0], P, N[:, :0], N, np.eye(3), np.zeros(3)))
    items.append((P, P[:, :0], N, N[:, :0], np.eye(3), np.zeros(3)))
    items.append((P[:, :2], P, N[:, :2], N, np.eye(3), np.zeros(3)))
    src, tgt, R, t, R0, t0, d = scene(bunny[:, ::2], 51)
    off = 1e6 * d * np.array([1.0, -0.7, 0.4])
    items.append((src + off[:, None], tgt + off[:, None], pio.estimate_normals(src, 20), pio.estimate_normals(tgt, 20),
                  R0, t0 + off - R0 @ off))
    S = synth.make_surface(50_000, 4)
    src, tgt, R, t, R0, t0, d50 = scene(S, 22)
    rn = 4 * spacing(S)
    items.append((src, tgt, radius_normals(src, rn), radius_normals(tgt, rn), R0, t0))
    return items, d


def test_mixed_batch_is_bit_identical_to_single_calls(bunny):
    import torch

    from psulvsb_b200 import stages

    items, d = mixed_batch(bunny)
    kw = dict(trace=True, max_iterations=15)
    want = [icp.gicp(s, q, ns, nt, R0, t0, d, **kw) for s, q, ns, nt, R0, t0 in items]
    got = icp.gicp_batch(*zip(*[it[:4] for it in items]), np.array([it[4] for it in items]),
                         np.array([it[5] for it in items]), d, **kw)
    assert all(same(g, w) for g, w in zip(got, want))
    perm = np.random.default_rng(2).permutation(len(items))
    again = icp.gicp_batch(*zip(*[items[k][:4] for k in perm]), np.array([items[k][4] for k in perm]),
                           np.array([items[k][5] for k in perm]), d, **kw)
    assert all(same(g, want[k]) for k, g in zip(perm, again))
    dev = lambda a: stages.to_device_points(a) if a.shape[1] else torch.empty((0, 3), dtype=torch.float64,  # noqa
                                                                              device="cuda")
    work = torch.full((int(2e8),), 0xFF, dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        res = icp.gicp_batch_device(*[[dev(it[j]) for it in items] for j in range(4)],
                                    np.array([it[4] for it in items]), np.array([it[5] for it in items]), d,
                                    work=work, **kw)
    side.synchronize()
    for r, w in zip(res, want):
        r.correspondences = r.correspondences.cpu().numpy()
        assert same(r, w)
    assert want[0].status == want[1].status == want[2].status == OI.NO_UPDATE
    assert want[4].iterations >= 2


def test_592_pairs_of_5000_points():
    rng = np.random.default_rng(0)
    srcs, tgts, nss, nts, R0s, t0s = [], [], [], [], [], []
    sp = 2.0 / np.sqrt(5000)
    for b in range(592):
        S = synth.make_surface(5000, b % 37)
        R, _ = synth.random_rigid(rng)
        t = rng.normal(size=3)
        Ns = radius_normals(S, 4 * sp) if b < 37 else nss[b % 37]
        srcs.append(S + rng.normal(0, 0.1 * sp, S.shape))
        tgts.append(R @ S + t[:, None])
        nss.append(Ns)
        nts.append(R @ Ns)
        a = np.deg2rad(2.0)
        R0s.append(R @ (np.cos(a) * np.eye(3) + np.sin(a) * np.array([[0, -1, 0], [1, 0, 0], [0, 0, 0]]) +
                        (1 - np.cos(a)) * np.diag([0, 0, 1.0])))
        t0s.append(t + 0.01 * rng.normal(size=3))
    d = 3 * sp
    got = icp.gicp_batch(srcs, tgts, nss, nts, np.array(R0s), np.array(t0s), d)
    for b in (0, 1, 295, 591):
        want = icp.gicp(srcs[b], tgts[b], nss[b], nts[b], R0s[b], t0s[b], d)
        assert same(got[b], want), b
    assert np.mean([g.fitness for g in got]) > 0.95


def test_fpfh_match_solve_gicp_batch_end_to_end(bunny):
    """The raw-cloud chain in four batched calls, the FPFH radius normals going straight into gicp_batch."""
    ext = extent(bunny)
    tgts, vps, truth = [], [], []
    for seed, noise in ((12, 0.0), (14, 0.002)):
        R, _ = synth.random_rigid(np.random.default_rng(seed))
        t = np.array([0.4, -0.3, 0.2])
        perm = np.random.default_rng(seed + 1).permutation(bunny.shape[1])
        tgt = (R @ bunny + t[:, None])[:, perm]
        if noise:
            tgt = tgt + np.random.default_rng(seed + 2).normal(0, noise * ext, tgt.shape)
        tgts.append(tgt)
        vps.append(tuple(t))
        truth.append((R, t))
    out = features.fpfh_batch([bunny] + tgts, 0.08, 0.15, viewpoints=[(0.0, 0.0, 0.0)] + vps)
    matches = features.match_batch([bunny] * 2, tgts, [out[0][0]] * 2, [f for f, _ in out[1:]], crosscheck=True)
    problems = [capi.HostProblem(bunny[:, m[:, 0]], tgt[:, m[:, 1]]) for m, tgt in zip(matches, tgts)]
    kw = dict(noise_bound=0.01 * ext, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005,
              wallclock_cap_s=0.0, seed=1)
    sols = capi.Handle(0).solve_batch(capi.default_params(**kw), problems)
    assert all(s.valid for s in sols)
    d = 3.0 * spacing(bunny)
    res = icp.gicp_batch([bunny] * 2, tgts, [out[0][1]] * 2, [n for _, n in out[1:]], np.array([s.R for s in sols]),
                         np.array([s.t for s in sols]), d)
    for o, s, (R, t) in zip(res, sols, truth):
        print("solve", synth.rotation_error(s.R, R), "gicp", synth.rotation_error(o.R, R), o.fitness, o.iterations)
        assert synth.rotation_error(o.R, R) <= synth.rotation_error(s.R, R)
        assert np.linalg.norm(o.t - t) <= np.linalg.norm(s.t - t)
    for k in range(2):
        alone = icp.gicp(bunny, tgts[k], out[0][1], out[k + 1][1], sols[k].R, sols[k].t, d)
        assert same(alone, res[k])


def test_end_to_end_bunny_noise_free(bunny):
    R, t, tgt, Rs, ts, ext = registration(bunny, 0.0, 12)
    d = 3.0 * spacing(bunny)
    Ns, Nt = radius_normals(bunny, 0.08), radius_normals(tgt, 0.08)
    out = icp.gicp(bunny, tgt, Ns, Nt, Rs, ts, d, max_iterations=100, relative_fitness=1e-12, relative_rmse=1e-12)
    print("solve", synth.rotation_error(Rs, R), "gicp", synth.rotation_error(out.R, R), np.linalg.norm(out.t - t),
          out.fitness, out.iterations, out.status)
    assert synth.rotation_error(out.R, R) <= 1e-6
    assert np.linalg.norm(out.t - t) <= 1e-6 * ext
    assert out.fitness == 1.0


def test_end_to_end_bunny_with_noise(bunny):
    R, t, tgt, Rs, ts, ext = registration(bunny, 0.002, 14)
    d = 3.0 * spacing(bunny)
    Ns, Nt = pio.estimate_normals(bunny, 20), pio.estimate_normals(tgt, 20)
    out = icp.gicp(bunny, tgt, Ns, Nt, Rs, ts, d)
    print("solve", synth.rotation_error(Rs, R), "gicp", synth.rotation_error(out.R, R), out.fitness, out.iterations)
    assert synth.rotation_error(out.R, R) <= synth.rotation_error(Rs, R)
    assert np.linalg.norm(out.t - t) <= np.linalg.norm(ts - t)
