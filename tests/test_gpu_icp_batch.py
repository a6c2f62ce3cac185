"""The batched ICP refinement on the GPU: every pair of a batch against the same pair refined alone (bit for bit, both
modes, edge pairs included), pairs that stop at different rounds, order / host / stream / workspace independence, a
batch of 592 pairs, and the solve_batch -> icp_batch chain from raw clouds."""
import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from oracle import icp as OI
from psulvsb_b200 import capi, features, icp, stages, synth
from tests.test_gpu_icp import bunny, check_step_locked, extent, perturbed, radius_normals, scene, spacing  # noqa: F401

pytestmark = pytest.mark.gpu


def same(a, b):
    """Two IcpResults are equal field by field (bit for bit), correspondences and trace included."""
    ca = a.correspondences.cpu().numpy() if hasattr(a.correspondences, "cpu") else a.correspondences
    cb = b.correspondences.cpu().numpy() if hasattr(b.correspondences, "cpu") else b.correspondences
    ok = (np.array_equal(a.R, b.R) and np.array_equal(a.t, b.t) and a.fitness == b.fitness
          and a.inlier_rmse == b.inlier_rmse and a.n_correspondences == b.n_correspondences
          and a.iterations == b.iterations and a.status == b.status and np.array_equal(ca, cb))
    if a.trace is not None or b.trace is not None:
        ok = ok and all(np.array_equal(a.trace[k], b.trace[k]) for k in a.trace)
    return ok


def single(pair, d, p2l, **kw):
    """The pair refined alone.  psulvsb_icp_host wants a normals pointer for point-to-plane even without target points
    (the batch takes NULL there): an empty target gets an empty normal array."""
    src, tgt, R0, t0, N = pair
    if p2l and N is None:
        N = np.zeros((3, 0))
    return icp.icp(src, tgt, R0, t0, d, target_normals=N if p2l else None, point_to_plane=p2l, **kw)


def batch(pairs, d, p2l, **kw):
    return icp.icp_batch([p[0] for p in pairs], [p[1] for p in pairs], np.array([p[2] for p in pairs]),
                         np.array([p[3] for p in pairs]), d,
                         target_normals=[p[4] for p in pairs] if p2l else None, point_to_plane=p2l, **kw)


@pytest.fixture(scope="module")
def mixed(bunny):
    """One batch of edge pairs sharing d = 3 mean bunny spacings: (src, tgt, R0, t0, normals) each, and the names."""
    d = 3.0 * spacing(bunny)
    rn = 4 * spacing(bunny)
    out, names = [], []

    def add(name, src, tgt, R0, t0, N):
        out.append((src, tgt, R0, t0, N))
        names.append(name)

    for seed in (21, 22, 23):
        src, tgt, R, t, R0, t0, _ = scene(bunny, seed)
        add(f"bunny{seed}", src, tgt, R0, t0, radius_normals(tgt, rn))
    src, tgt, R, t, R0, t0, _ = scene(bunny, 24)
    m = 128 * (src.shape[1] // 128)
    add("ns_multiple_of_128", src[:, :m], tgt, R0, t0, radius_normals(tgt, rn))
    S = synth.make_surface(50_000, 4)
    src, tgt, R, t, R0, t0, _ = scene(S, 22)
    add("surface50k", src, tgt, R0, t0, radius_normals(tgt, 4 * spacing(S)))
    R0, t0 = synth.random_rigid(np.random.default_rng(3))[0], np.array([0.1, 0.2, 0.3])
    Q = R0 @ bunny + t0[:, None]
    add("one_point_source", bunny[:, :1], Q, R0, t0, radius_normals(Q, rn))
    add("empty_source", bunny[:, :0], Q, R0, t0, radius_normals(Q, rn))
    add("empty_target", bunny[:, :50], Q[:, :0], R0, t0, None)
    small = bunny[:, ::4] * (d / extent(bunny))                  # the whole target spans a handful of cells
    src, tgt, R, t, R0, t0, _ = scene(small, 41)
    add("few_cells", src, tgt, R0, t0, radius_normals(tgt, 4 * spacing(small)))
    P = bunny[:, ::2]
    src, tgt, R, t, R0, t0, _ = scene(P, 51)
    off = 1e6 * d * np.array([1.0, -0.7, 0.4])
    src, tgt = src + off[:, None], tgt + off[:, None]
    add("far_from_origin", src, tgt, R0, t0 + off - R0 @ off, radius_normals(tgt, rn))
    S = synth.make_surface(20_000, 6)
    rng = np.random.default_rng(7)
    iso = rng.uniform(3.0, 4.0, (3, 200))
    src, tgt, R, t, R0, t0, _ = scene(S, 61)
    tgt = np.concatenate([tgt, R @ iso + t[:, None]], axis=1)
    src = np.concatenate([src, iso + rng.normal(0, 1e-3, iso.shape)], axis=1)
    N = radius_normals(tgt, 4 * spacing(S))
    assert not np.isfinite(N[:, -200:]).all(axis=0).any()
    add("nan_normals", src, tgt, R0, t0, N)
    ns = [p[0].shape[1] for p in out]
    assert any(n % 128 == 0 for n in ns if n) and any(n % 128 for n in ns)
    return out, names, d


@pytest.mark.parametrize("point_to_plane", [False, True])
def test_batch_is_bit_identical_to_single_calls(mixed, point_to_plane):
    pairs, names, d = mixed
    got = batch(pairs, d, point_to_plane, trace=True)
    assert len(got) == len(pairs)
    for name, pair, g in zip(names, pairs, got):
        want = single(pair, d, point_to_plane, trace=True)
        assert same(g, want), name
    # far from the origin, point-to-plane's J = [p' x n, n] puts |p'|^2 ~ 1e10 into the condition of J^T J, so its
    # update is step-locked in point-to-point only (as in test_gpu_icp.py); bit identity above holds for every pair
    for name in ("bunny21", "bunny22") if point_to_plane else ("bunny21", "far_from_origin"):
        k = names.index(name)
        src, tgt, _, _, N = pairs[k]
        check_step_locked(src, tgt, d, got[k], normals=N, point_to_plane=point_to_plane)
    by = dict(zip(names, got))
    for name in ("empty_source", "empty_target"):
        assert by[name].status == OI.NO_UPDATE and by[name].iterations == 0 and len(by[name].trace["fitness"]) == 1
    assert (by["empty_target"].correspondences == -1).all() and by["empty_target"].correspondences.size == 50
    assert by["bunny21"].iterations >= 2
    if point_to_plane:
        c = by["nan_normals"].correspondences
        assert (c[-200:] == -1).all()


def test_pairs_stop_at_different_rounds(bunny):
    d = 3.0 * spacing(bunny)
    R, _ = synth.random_rigid(np.random.default_rng(70))
    t = np.array([0.3, -0.1, 0.2])
    pairs = [(bunny, R @ bunny + t[:, None], R, t, None)]          # starts at the truth: converges at k = 1
    for seed, angle in ((71, 0.2), (72, 2.0), (73, 6.0), (74, 0.5), (75, 10.0)):
        src, tgt, R, t, _, _, _ = scene(bunny, seed)
        R0, t0 = perturbed(R, t, np.random.default_rng(seed), angle, 0.002 * angle * extent(bunny))
        pairs.append((src, tgt, R0, t0, None))
    for cap in (30, 6):
        got = batch(pairs, d, False, max_iterations=cap, trace=True)
        for pair, g in zip(pairs, got):
            assert same(g, single(pair, d, False, max_iterations=cap, trace=True))
        its = {g.iterations for g in got}
        assert len(its) >= 2, its
        if cap == 6:
            st = {g.status for g in got}
            assert OI.CONVERGED in st and OI.MAX_ITERATIONS in st, [(g.status, g.iterations) for g in got]


def test_order_host_device_stream_and_dirty_workspace(mixed):
    import torch

    pairs, names, d = mixed
    for p2l in (False, True):
        kw = dict(point_to_plane=p2l, trace=True, max_iterations=12, relative_fitness=0, relative_rmse=0)
        ref = batch(pairs, d, p2l, **{k: v for k, v in kw.items() if k != "point_to_plane"})
        perm = np.random.default_rng(5).permutation(len(pairs))
        shuffled = batch([pairs[i] for i in perm], d, p2l, **{k: v for k, v in kw.items() if k != "point_to_plane"})
        for j, i in enumerate(perm):
            assert same(shuffled[j], ref[i]), names[i]
        ds = [stages.to_device_points(p[0]) for p in pairs]
        dt = [stages.to_device_points(p[1]) for p in pairs]
        dn = [None if p[4] is None else stages.to_device_points(p[4]) for p in pairs]
        if p2l:
            dn = [n if n is not None else torch.empty((0, 3), dtype=torch.float64, device="cuda") for n in dn]
        R0s, t0s = np.array([p[2] for p in pairs]), np.array([p[3] for p in pairs])
        cpairs = (capi.IcpPair * len(pairs))()
        for b, (s, t) in enumerate(zip(ds, dt)):
            cpairs[b].n_s, cpairs[b].n_t = s.shape[0], t.shape[0]
        nbytes = capi.lib().psulvsb_icp_batch_workspace_bytes(cpairs, len(pairs))
        work = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, device="cuda")
        side = torch.cuda.Stream()
        for _ in range(2):                          # the second call finds the first one's leftovers
            with torch.cuda.stream(side):
                got = icp.icp_batch_device(ds, dt, R0s, t0s, d, d_target_normals=dn if p2l else None, work=work, **kw)
            side.synchronize()
            for name, g, r in zip(names, got, ref):
                assert same(g, r), name


def test_592_pairs_of_5000_points(bunny):
    B, n = 592, 5000
    rng = np.random.default_rng(592)
    bases = [synth.make_surface(n, s) for s in range(8)]
    sp = spacing(bases[0])
    d = 3.0 * sp
    pairs, truth = [], []
    for b in range(B):
        P = bases[b % 8]
        R, _ = synth.random_rigid(rng)
        t = rng.normal(size=3)
        src = P + rng.normal(0, 0.1 * sp, P.shape)
        # T0: the truth moved by 0.5 degrees and 0.2 % of the extent, so that every point starts within d of its
        # counterpart (a rotation about the origin moves these clouds by up to 0.5 degrees x 2.9)
        R0, t0 = perturbed(R, t, rng, 0.5, 0.002 * extent(P))
        pairs.append((src, R @ P + t[:, None], R0, t0, None))
        truth.append((R, t, R0, t0))
    kw = dict(relative_fitness=0, relative_rmse=0)                # every pair runs 30 iterations
    got = batch(pairs, d, False, **kw)
    assert len(got) == B
    sample = [0, B - 1] + sorted(np.random.default_rng(1).choice(np.arange(1, B - 1), 14, replace=False).tolist())
    for b in sample:
        assert same(got[b], single(pairs[b], d, False, **kw)), b
    for b, (g, (R, t, R0, t0)) in enumerate(zip(got, truth)):
        assert g.fitness > 0.95, (b, g.fitness)
        assert synth.rotation_error(g.R, R) < 0.5 * synth.rotation_error(R0, R), b
        assert np.linalg.norm(g.t - t) < 0.5 * np.linalg.norm(t0 - t), b


def test_solve_batch_then_icp_batch_end_to_end(bunny):
    """bunny pairs -> FPFH -> correspondences -> one solve_batch -> icp_batch: every refined transform is closer to the
    truth than the solve's.  Point-to-plane refines the noise-free pairs (the truth is a fixed point there); the pairs
    with noise (sigma = 0.002 extent, as in test_end_to_end_bunny_with_noise) are refined point-to-point, whose
    correspondence sums average the noise out, while radius normals of the noisy target carry it into every row."""
    ext = extent(bunny)
    fs, _ = features.fpfh(bunny, 0.08, 0.15)
    problems, truth, tgts, normals = [], [], [], []
    seeds = {12: 0.0, 13: 0.0, 14: 0.002, 15: 0.002}
    for seed, noise in seeds.items():
        R, _ = synth.random_rigid(np.random.default_rng(seed))
        t = np.array([0.4, -0.3, 0.2])
        perm = np.random.default_rng(seed + 1).permutation(bunny.shape[1])
        tgt = (R @ bunny + t[:, None])[:, perm]
        if noise:
            tgt = tgt + np.random.default_rng(seed + 2).normal(0, noise * ext, tgt.shape)
        ft, nt = features.fpfh(tgt, 0.08, 0.15, viewpoint=t)
        m = features.match(bunny, tgt, fs, ft, crosscheck=True)
        problems.append(capi.HostProblem(bunny[:, m[:, 0]], tgt[:, m[:, 1]]))
        truth.append((R, t))
        tgts.append(tgt)
        normals.append(nt)
    kw = dict(noise_bound=0.01 * ext, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005,
              wallclock_cap_s=0.0, seed=1)
    sols = capi.Handle(0).solve_batch(capi.default_params(**kw), problems)
    assert all(s.valid for s in sols)
    d = 3.0 * spacing(bunny)
    for p2l in (True, False):
        idx = [k for k, noise in enumerate(seeds.values()) if (noise == 0.0) == p2l]
        out = icp.icp_batch([bunny] * len(idx), [tgts[k] for k in idx], np.array([sols[k].R for k in idx]),
                            np.array([sols[k].t for k in idx]), d,
                            target_normals=[normals[k] for k in idx] if p2l else None, point_to_plane=p2l)
        for k, o in zip(idx, out):
            s, (R, t) = sols[k], truth[k]
            print("p2l" if p2l else "p2p", "solve", synth.rotation_error(s.R, R), np.linalg.norm(s.t - t), "icp",
                  synth.rotation_error(o.R, R), np.linalg.norm(o.t - t), o.fitness, o.iterations, o.status)
            assert synth.rotation_error(o.R, R) <= synth.rotation_error(s.R, R)
            assert np.linalg.norm(o.t - t) <= np.linalg.norm(s.t - t)
            if p2l:
                assert o.fitness == 1.0
