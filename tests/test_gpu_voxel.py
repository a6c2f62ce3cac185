"""The voxel filter on the GPU (psulvsb_voxel_down_sample*, csrc/k8_voxel.cu; DESIGN.md section 10, "Voxel
downsampling") against the numpy restatement (tests/voxel_restatement.py), bit for bit with the same order and count:
the bunny and a 50 000-point surface from below the spacing (identity) to a handful of voxels, a far-shifted cloud,
boundary lattices, duplicates, NaN / Inf points, tiny and empty clouds, buckets holding several voxels; determinism on a
side stream with a dirty workspace, host against device, batches against single calls; and the raw-scan chain
voxel_down_sample_batch -> fpfh_batch -> match_batch -> solve_batch -> icp_batch on the dense clouds."""
import os

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from psulvsb_b200 import capi, features, icp, stages, synth
from tests import voxel_restatement as VR

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bunny():
    return np.load(os.path.join(ROOT, "tests", "golden", "bunny_res3.npz"))["vertices"].astype(np.float64) * 10


@pytest.fixture(scope="module")
def surface():
    return synth.make_surface(50000, 9)


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a, b)


def check(P, v):
    got = features.voxel_down_sample(P, v)
    want = VR.voxel_down_sample(P, v)
    assert same(got, want), (P.shape, v, got.shape, want.shape)
    return got


def lattice(seed=0):
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(np.arange(6), np.arange(5), np.arange(4)), 0).reshape(3, -1).astype(np.float64)
    return g[:, rng.permutation(g.shape[1])] - 3.0


def dirty(seed=1):
    """A surface with duplicated points and NaN / Inf coordinates sprinkled in."""
    rng = np.random.default_rng(seed)
    S = synth.make_surface(3000, 5)
    P = np.concatenate([S, S[:, rng.choice(3000, 400)]], axis=1)[:, rng.permutation(3400)]
    for k, bad in zip(rng.choice(3400, 60, replace=False), [np.nan, np.inf, -np.inf] * 20):
        P[rng.integers(3), k] = bad
    return P


# ---- against the restatement ----------------------------------------------------------------------------------------

def test_bunny_and_surface_across_voxel_sizes(bunny, surface):
    for P, sizes in ((bunny, (1e-4, 0.01, 0.03, 0.1, 0.3, 1.0, 5.0)), (surface, (1e-4, 0.005, 0.02, 0.05, 0.2, 0.7, 3.0))):
        counts = [check(P, v).shape[1] for v in sizes]
        assert counts[0] > 0.99 * P.shape[1] and counts[-1] <= 8 and counts == sorted(counts, reverse=True), counts
    assert same(features.voxel_down_sample(bunny, 1e-4), bunny)          # one point per voxel: the input, in order


def test_far_shifted_cloud(bunny):
    ext = float(np.linalg.norm(np.ptp(bunny, axis=1)))
    P = bunny - bunny.mean(axis=1, keepdims=True) + 1e4 * ext * np.array([[1.0], [-0.5], [0.25]])
    for v in (0.01, 0.05, 0.3):
        check(P, v)


def test_boundaries_duplicates_and_non_finite_points():
    L = lattice()
    assert same(check(L, 1.0), L)                                        # exact k + 0.5: one point per cell
    for v in (2.0, 3.0, 0.5):
        check(L, v)
    check(np.concatenate([L, L, L[:, ::-1]], axis=1), 1.0)              # every cell three times
    P = dirty()
    for v in (0.01, 0.05, 0.4):
        check(P, v)
    nan = np.full((3, 300), np.nan)
    assert features.voxel_down_sample(nan, 0.1).shape == (3, 0)
    mixed = np.concatenate([nan[:, :5], L, np.full((3, 2), np.inf)], axis=1)
    assert same(check(mixed, 1.0), L)


def test_tiny_and_empty_clouds():
    assert features.voxel_down_sample(np.zeros((3, 0)), 0.1).shape == (3, 0)
    P = np.array([[1.5], [-2.0], [3.25]])
    assert same(check(P, 0.1), P)
    for n in (2, 127, 128, 129, 257):
        check(synth.make_surface(n, n), 0.3)


def test_buckets_holding_several_voxels():
    """About 4 points per voxel: n / 4 voxels over bucket_count(n) buckets, several voxels share a bucket (shown by
    the restatement's hash), and the exact cell test keeps them apart."""
    P = np.random.default_rng(4).uniform(0.0, 1.0, (3, 8192))
    v = 1.0 / 12.0
    assert VR.voxels_per_bucket(P, v) >= 3
    check(P, v)
    Q = np.random.default_rng(5).uniform(0.0, 1.0, (3, 300))           # 300 voxels, 512 buckets, cells far apart
    Q = np.floor(Q * 1e3) * 7.0
    assert VR.voxels_per_bucket(Q, 1.0) >= 2
    assert same(check(Q, 1.0), Q)


# ---- determinism, host and device -----------------------------------------------------------------------------------

def test_device_entry_dirty_workspace_side_stream(bunny, surface):
    import torch

    L = capi.lib()
    big = surface[:, :20000]
    work = torch.full((int(L.psulvsb_voxel_down_sample_workspace_bytes(big.shape[1])),), 0xFF, dtype=torch.uint8,
                      device="cuda")
    side = torch.cuda.Stream()
    for P, v in ((big, 0.02), (bunny, 0.05), (dirty(), 0.05), (lattice(), 1.0)):
        n = P.shape[1]
        d_pts = stages.to_device_points(P)
        want = VR.voxel_down_sample(P, v)
        outs = []
        for _ in range(2):
            out = torch.full((n, 3), 7.0, dtype=torch.float64, device="cuda")
            cnt = torch.full((1,), -5, dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()
            capi.check(L.psulvsb_voxel_down_sample(side.cuda_stream, d_pts.data_ptr(), n, v, work.data_ptr(),
                                                   out.data_ptr(), cnt.data_ptr()))
            side.synchronize()
            outs.append(out[:int(cnt.item())].cpu().numpy().T)
            work.fill_(0xFF)
        assert same(outs[0], outs[1]) and same(outs[0], want)
        assert same(features.voxel_down_sample(P, v), want)
        with torch.cuda.stream(side):
            dv, dc = features.voxel_down_sample_device(d_pts, v, work=work)
        side.synchronize()
        assert same(dv[:int(dc.item())].cpu().numpy().T, want)


# ---- batches --------------------------------------------------------------------------------------------------------

def mixed(bunny):
    return [bunny, lattice(2), np.zeros((3, 0)), np.full((3, 200), np.nan), synth.make_surface(5000, 3), dirty(6),
            np.array([[0.5], [0.5], [0.5]]), np.zeros((3, 0)), synth.make_surface(129, 4)]


def test_batch_items_equal_single_calls(bunny):
    clouds = mixed(bunny)
    for v in (0.05, 1.0):
        want = [features.voxel_down_sample(P, v) for P in clouds]
        for P, w in zip(clouds, want):
            assert same(w, VR.voxel_down_sample(P, v))
        for order in (list(range(len(clouds))), list(reversed(range(len(clouds))))):
            got = features.voxel_down_sample_batch([clouds[c] for c in order], v)
            for k, c in enumerate(order):
                assert same(got[k], want[c]), (v, order, c)
        for P, w in zip(clouds, want):                                   # B = 1
            assert same(features.voxel_down_sample_batch([P], v)[0], w)


def test_batch_592_clouds_of_5000_on_the_device():
    import torch

    clouds = [synth.make_surface(5000, b) for b in range(592)]
    d = [stages.to_device_points(P) for P in clouds]
    v = 0.04
    allv, counts, offsets = features.voxel_down_sample_batch_device(d, v)
    torch.cuda.synchronize()
    counts = counts.cpu().numpy()
    assert allv.shape == (592 * 5000, 3) and list(offsets) == [5000 * b for b in range(592)]
    allv = allv.cpu().numpy()
    for b in range(592):
        single, c = features.voxel_down_sample_device(d[b], v)
        assert int(c.item()) == counts[b]
        got = allv[offsets[b]:offsets[b] + counts[b]]
        assert same(got, single[:counts[b]].cpu().numpy()), b
        if b % 74 == 0:
            assert same(got.T, VR.voxel_down_sample(clouds[b], v)), b
    assert same(features.voxel_down_sample_batch(clouds[:3], v)[2], allv[10000:10000 + counts[2]].T)


# ---- the raw-scan chain ---------------------------------------------------------------------------------------------

def test_voxel_fpfh_match_solve_then_icp_on_the_dense_clouds():
    """Two 200 000-point surfaces related by a known rigid transform (the target is the moved, shuffled source):
    downsampled to a few thousand voxels each, the correspondence chain and the solver find the transform, and ICP on
    the dense clouds refines it."""
    src = synth.make_surface(200000, 31)
    truth = []
    tgts = []
    for seed in (41, 42):
        R, _ = synth.random_rigid(np.random.default_rng(seed))
        t = np.array([0.4, -0.3, 0.2])
        tgts.append((R @ src + t[:, None])[:, np.random.default_rng(seed + 1).permutation(src.shape[1])])
        truth.append((R, t))
    v = 0.04
    down = features.voxel_down_sample_batch([src] + tgts, v)
    for P, dn in zip([src] + tgts, down):
        assert 2000 <= dn.shape[1] <= 5000, dn.shape
        assert same(dn, features.voxel_down_sample(P, v))
    out = features.fpfh_batch(down, 2.0 * v, 5.0 * v)
    fs = out[0][0]
    matches = features.match_batch([down[0]] * 2, down[1:], [fs] * 2, [f for f, _ in out[1:]], crosscheck=True)
    problems = [capi.HostProblem(down[0][:, m[:, 0]], dn[:, m[:, 1]]) for m, dn in zip(matches, down[1:])]
    kw = dict(noise_bound=1.5 * v, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005, wallclock_cap_s=0.0,
              seed=1)
    sols = capi.Handle(0).solve_batch(capi.default_params(**kw), problems)
    assert all(s.valid for s in sols)
    res = icp.icp_batch([src] * 2, tgts, np.array([s.R for s in sols]), np.array([s.t for s in sols]), v,
                        max_iterations=60)
    for s, o, (R, t) in zip(sols, res, truth):
        print(f"solve: {synth.rotation_error(s.R, R):.2e} rad {np.linalg.norm(s.t - t):.2e}; "
              f"icp: {synth.rotation_error(o.R, R):.2e} rad {np.linalg.norm(o.t - t):.2e} fitness {o.fitness:.4f}")
        assert synth.rotation_error(s.R, R) < 0.05 and np.linalg.norm(s.t - t) < 0.1
        assert synth.rotation_error(o.R, R) <= synth.rotation_error(s.R, R)
        assert np.linalg.norm(o.t - t) <= np.linalg.norm(s.t - t)
        assert synth.rotation_error(o.R, R) < 2e-3 and np.linalg.norm(o.t - t) < 5e-3
        assert o.fitness > 0.99
