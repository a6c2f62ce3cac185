"""Batched FPFH and matcher on the GPU: every item of a mixed batch is bit-identical to the single call on it alone
(edge clouds, NN boundary shapes, empty sides, short lists, tuple tests over several rounds), whatever the order, host
against device, on a side stream with a dirty workspace; 592 pairs of 5 000 points; and the raw-cloud chain
fpfh_batch -> match_batch -> solve_batch -> icp_batch against the loop of single calls."""
import os

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from psulvsb_b200 import capi, features, icp, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bunny():
    return np.load(os.path.join(ROOT, "tests", "golden", "bunny_res3.npz"))["vertices"].astype(np.float64) * 10


def cap(n, seed, radius=0.1):
    rng = np.random.default_rng(seed)
    th = np.arccos(rng.uniform(np.cos(1.0), 1.0, n))
    ph = rng.uniform(0, 2 * np.pi, n)
    P = radius * np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)])
    return P - P.mean(axis=1, keepdims=True)


def same_f(a, b):
    return np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


def same_n(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


def edge_clouds(bunny):
    """(cloud, viewpoint): tiny clouds with colliding cells, one bucket holding the cloud, far and negative cells,
    duplicates, an empty cloud, multiples of 128 and not, a 50 000-point surface."""
    rng = np.random.default_rng(5)
    S = synth.make_surface(4000, 21)
    dup = np.concatenate([S, S[:, rng.choice(4000, 200, replace=False)]], axis=1)[:, rng.permutation(4200)]
    one = bunny - bunny.min(axis=1, keepdims=True) + 0.01
    out = [(cap(n, 100 + n, 0.05), (0.0, 0.0, 10.0 + n)) for n in (1, 2, 3, 7, 33, 127, 128, 129)]
    out += [(one * 0.05, (1.0, 2.0, 3.0)), (bunny - bunny.mean(axis=1, keepdims=True) + np.array([[1e3], [-1e3], [5e2]]),
                                            (1e3, -1e3, 6e2)),
            (dup, (0.0, 0.0, 0.0)), (np.zeros((3, 0)), (0.0, 0.0, 0.0)), (bunny, (0.4, -0.3, 0.2)),
            (synth.make_surface(256, 3), (0.0, -5.0, 0.0)), (synth.make_surface(50000, 4), (0.0, 0.0, 5.0))]
    return out


def test_fpfh_batch_bit_identical_to_single_calls(bunny):
    items = edge_clouds(bunny)
    P = [p for p, _ in items]
    vps = [v for _, v in items]
    got = features.fpfh_batch(P, 0.06, 0.12, viewpoints=vps)
    for (p, v), (f, n) in zip(items, got):
        wf, wn = features.fpfh(p, 0.06, 0.12, viewpoint=v)
        assert f.shape == wf.shape and same_f(f, wf) and same_n(n, wn), p.shape
    # a permuted batch gives the same per-cloud results
    perm = np.random.default_rng(1).permutation(len(items))
    again = features.fpfh_batch([P[k] for k in perm], 0.06, 0.12, viewpoints=[vps[k] for k in perm])
    for k, (f, n) in zip(perm, again):
        assert same_f(f, got[k][0]) and same_n(n, got[k][1])


def test_fpfh_batch_device_dirty_workspace_side_stream(bunny):
    import torch

    from psulvsb_b200 import stages

    items = edge_clouds(bunny)[:10]
    want = features.fpfh_batch([p for p, _ in items], 0.06, 0.12, viewpoints=[v for _, v in items])
    d = [stages.to_device_points(p) if p.shape[1] else torch.empty((0, 3), dtype=torch.float64, device="cuda")
         for p, _ in items]
    work = torch.full((64 << 20,), 0xFF, dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        feats, normals, views = features.fpfh_batch_device(d, 0.06, 0.12, viewpoints=[v for _, v in items], work=work)
    side.synchronize()
    for (f, n), (wf, wn) in zip(views, want):
        assert same_f(f.cpu().numpy(), wf) and same_n(n.cpu().numpy().T, wn)


def nn_pair(base, ns, nt, seed):
    rng = np.random.default_rng(seed)
    fs = base[rng.integers(0, base.shape[0], ns)] + rng.normal(0, 0.3, (ns, 33)).astype(np.float32)
    ft = base[rng.integers(0, base.shape[0], nt)] + rng.normal(0, 0.3, (nt, 33)).astype(np.float32)
    if ns and nt:
        ft[1::5] = fs[rng.integers(0, ns, ft[1::5].shape[0])]
    return rng.uniform(-1, 1, (3, ns)), rng.uniform(-1, 1, (3, nt)), fs.astype(np.float32), ft.astype(np.float32)


def mixed_pairs(bunny):
    base = features.fpfh(bunny, 0.08, 0.15)[0]
    shapes = [(255, 63), (256, 64), (257, 65), (513, 2047), (300, 2048), (300, 2049), (1, 4097), (4097, 1),
              (2500, 1700), (1700, 2500), (0, 5), (5, 0), (1, 1), (2, 2), (700, 700)]
    return [nn_pair(base, ns, nt, 10 + k) for k, (ns, nt) in enumerate(shapes)]


@pytest.mark.parametrize("cross", [True, False])
@pytest.mark.parametrize("tuple_test", [False, True])
def test_match_batch_bit_identical_to_single_calls(bunny, cross, tuple_test):
    pairs = mixed_pairs(bunny)
    seeds = [1000 + 7 * b for b in range(len(pairs))]
    got = features.match_batch(*zip(*pairs), crosscheck=cross, tuple_test=tuple_test, tuple_scale=0.5, seeds=seeds)
    for (s, t, fs, ft), seed, g in zip(pairs, seeds, got):
        want = features.match(s, t, fs, ft, crosscheck=cross, tuple_test=tuple_test, tuple_scale=0.5, seed=seed)
        assert np.array_equal(g, want), (s.shape, t.shape)
    # the default seeds are seed + b
    dflt = features.match_batch(*zip(*pairs), crosscheck=cross, tuple_test=tuple_test, tuple_scale=0.5, seed=1000)
    for b, (s, t, fs, ft) in enumerate(pairs[:4]):
        want = features.match(s, t, fs, ft, crosscheck=cross, tuple_test=tuple_test, tuple_scale=0.5, seed=1000 + b)
        assert np.array_equal(dflt[b], want)


def test_tuple_test_over_several_rounds():
    """11 000 identity correspondences between independent random clouds: few trials pass, so every pair runs many
    rounds; pairs of different list lengths and seeds finish at different rounds."""
    items = []
    for k, (n, scale) in enumerate(((11000, 0.95), (11000, 0.935), (3000, 0.9), (20, 0.5))):
        rng = np.random.default_rng(k + 1)
        f = rng.uniform(0, 100, (n, 33)).astype(np.float32)
        items.append((rng.uniform(-1, 1, (3, n)), rng.uniform(-1, 1, (3, n)), f, f))
    for scale in (0.95, 0.935):
        got = features.match_batch(*zip(*items), crosscheck=True, tuple_test=True, tuple_scale=scale, seed=1)
        for b, (s, t, fs, ft) in enumerate(items):
            want = features.match(s, t, fs, ft, crosscheck=True, tuple_test=True, tuple_scale=scale, seed=1 + b)
            assert np.array_equal(got[b], want)


def test_match_batch_independence(bunny):
    """Permutation, host against device, a side stream and a dirty workspace: the same per-pair results."""
    import torch

    pairs = mixed_pairs(bunny)
    seeds = [5 * b + 3 for b in range(len(pairs))]
    for tuple_test in (False, True):
        want = features.match_batch(*zip(*pairs), crosscheck=True, tuple_test=tuple_test, tuple_scale=0.5, seeds=seeds)
        perm = np.random.default_rng(2).permutation(len(pairs))
        got = features.match_batch(*zip(*[pairs[k] for k in perm]), crosscheck=True, tuple_test=tuple_test,
                                   tuple_scale=0.5, seeds=[seeds[k] for k in perm])
        for k, g in zip(perm, got):
            assert np.array_equal(g, want[k])
        dev = [tuple(torch.from_numpy(np.ascontiguousarray(a.T if a.dtype == np.float64 else a)).cuda() for a in p)
               for p in pairs]
        work = torch.full((256 << 20,), 0xFF, dtype=torch.uint8, device="cuda")
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            out, counts, offs = features.match_batch_device(*zip(*dev), crosscheck=True, tuple_test=tuple_test,
                                                            tuple_scale=0.5, seeds=seeds, work=work)
        side.synchronize()
        out, counts = out.cpu().numpy(), counts.cpu().numpy()
        for b in range(len(pairs)):
            assert np.array_equal(out[offs[b]:offs[b] + counts[b]], want[b])


def test_592_pairs_of_5000_points():
    rng = np.random.default_rng(0)
    clouds, vps = [], []
    for b in range(592):
        R, _ = synth.random_rigid(rng)
        S = synth.make_surface(5000, b % 37)
        clouds += [S, R @ S + rng.normal(0, 0.002, S.shape)]
        vps += [(0.0, 0.0, 0.0), tuple(rng.uniform(-1, 1, 3))]
    feats = features.fpfh_batch(clouds, 0.06, 0.12, viewpoints=vps)
    for k in (0, 1, 591, 1183):
        f, n = features.fpfh(clouds[k], 0.06, 0.12, viewpoint=vps[k])
        assert same_f(feats[k][0], f) and same_n(feats[k][1], n)
    srcs, tgts = clouds[0::2], clouds[1::2]
    fss, fts = [f for f, _ in feats[0::2]], [f for f, _ in feats[1::2]]
    for tuple_test in (False, True):
        got = features.match_batch(srcs, tgts, fss, fts, crosscheck=True, tuple_test=tuple_test, seed=11)
        for b in (0, 295, 591):
            want = features.match(srcs[b], tgts[b], fss[b], fts[b], crosscheck=True, tuple_test=tuple_test,
                                  seed=11 + b)
            assert np.array_equal(got[b], want)


def test_fpfh_batch_match_batch_solve_batch_icp_batch_end_to_end(bunny):
    """The raw-cloud chain in four calls gives the same correspondences, solutions and refinements as the loop of
    single FPFH and match calls, and meets the accuracy bars of the loop's end-to-end test."""
    ext = float(np.linalg.norm(np.ptp(bunny, axis=1)))
    seeds = {12: 0.0, 13: 0.0, 14: 0.002, 15: 0.002}
    tgts, vps, truth = [], [], []
    for seed, noise in seeds.items():
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
    fs = out[0][0]
    matches = features.match_batch([bunny] * 4, tgts, [fs] * 4, [f for f, _ in out[1:]], crosscheck=True)
    fs1, _ = features.fpfh(bunny, 0.08, 0.15)
    assert same_f(fs, fs1)
    for k, tgt in enumerate(tgts):
        ft, nt = features.fpfh(tgt, 0.08, 0.15, viewpoint=vps[k])
        assert same_f(out[k + 1][0], ft) and same_n(out[k + 1][1], nt)
        assert np.array_equal(matches[k], features.match(bunny, tgt, fs1, ft, crosscheck=True))
    problems = [capi.HostProblem(bunny[:, m[:, 0]], tgt[:, m[:, 1]]) for m, tgt in zip(matches, tgts)]
    kw = dict(noise_bound=0.01 * ext, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005,
              wallclock_cap_s=0.0, seed=1)
    sols = capi.Handle(0).solve_batch(capi.default_params(**kw), problems)
    assert all(s.valid for s in sols)
    from scipy.spatial import cKDTree

    d = 3.0 * float(cKDTree(bunny.T).query(bunny.T, k=2)[0][:, 1].mean())
    for p2l in (True, False):
        idx = [k for k, noise in enumerate(seeds.values()) if (noise == 0.0) == p2l]
        res = icp.icp_batch([bunny] * len(idx), [tgts[k] for k in idx], np.array([sols[k].R for k in idx]),
                            np.array([sols[k].t for k in idx]), d,
                            target_normals=[out[k + 1][1] for k in idx] if p2l else None, point_to_plane=p2l)
        for k, o in zip(idx, res):
            s, (R, t) = sols[k], truth[k]
            assert synth.rotation_error(o.R, R) <= synth.rotation_error(s.R, R)
            assert np.linalg.norm(o.t - t) <= np.linalg.norm(s.t - t)
            if p2l:
                assert o.fitness == 1.0
