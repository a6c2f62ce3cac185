"""Normals alone on the GPU (psulvsb_normals*, csrc/k8_features.cu; DESIGN.md section 10, "Normals alone").

Radius mode: bit-identical to the normals of psulvsb_fpfh with the same normal radius and a feature radius r or r / 2
(the same grid, so the same walk), on the bunny, a 50 000-point surface, a far-shifted cloud and the edge shapes of
test_gpu_feature_edges.py.  Hybrid mode: against the restatement (tests/normals_restatement.py) with the bars of
check_normals -- the same NaN pattern, |cos| > 1 - 1e-6 with the same sign on every point that is not fragile, at
most 5 % fragile -- at radii where at least half of the points are capped; exact ties at the cap and more than max_nn
duplicates of one point; bit-identical to the radius mode when the cap does not bind.  Then determinism on a side
stream with a dirty workspace, host against device, and batches against single calls."""
import ctypes as C
import os

import numpy as np
import pytest
from scipy.spatial import cKDTree

import psulvsb_b200  # noqa: F401
from oracle import features as OF
from psulvsb_b200 import capi, features, stages, synth
from tests import normals_restatement as NR
from tests.test_gpu_feature_edges import cap, check_normals, tied_cloud

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bunny():
    return np.load(os.path.join(ROOT, "tests", "golden", "bunny_res3.npz"))["vertices"].astype(np.float64) * 10


@pytest.fixture(scope="module")
def surface():
    return synth.make_surface(50000, 9)


def same(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


def one_bucket(P):
    return P - P.min(axis=1, keepdims=True) + 0.01, 1.2 * float(np.linalg.norm(np.ptp(P, axis=1)))


def duplicated(seed=5):
    S = synth.make_surface(4000, 21)
    rng = np.random.default_rng(seed)
    P = np.concatenate([S, S[:, rng.choice(4000, 200, replace=False)]], axis=1)
    return P[:, rng.permutation(4200)]


# ---- radius mode == FPFH's normals ----------------------------------------------------------------------------------

def radius_cases(bunny, surface):
    out = [("bunny", bunny, 0.08, (0.0, 0.0, 0.0)), ("surface", surface, 0.03, (0.0, 0.0, 10.0)),
           ("far", bunny - bunny.mean(axis=1, keepdims=True) + np.array([[1e3], [-1e3], [5e2]]), 0.08, (0.0,) * 3),
           ("duplicates", duplicated(), 0.06, (0.0, 0.0, 0.0))]
    P, r = one_bucket(bunny)
    out.append(("one bucket", P, r, (0.0, 0.0, 0.0)))
    for n in (1, 2, 3, 4, 5, 7, 33, 127, 128, 129):          # tiny clouds, colliding cells
        out.append((f"cap {n}", cap(n, 100 + n), 1.0 if n < 33 else 0.06, (0.0, 0.0, 10.0)))
    return out


def test_radius_mode_is_fpfh_normals_bit_for_bit(bunny, surface):
    for name, P, r, vp in radius_cases(bunny, surface):
        got = features.normals(P, r, viewpoint=vp)
        for rf in (r, r / 2):
            assert same(got, features.fpfh(P, r, rf, viewpoint=vp)[1]), (name, rf)
        if P.shape[1] <= 2:
            assert np.isnan(got).all()


# ---- hybrid mode against the restatement ----------------------------------------------------------------------------

def capping_radius(P, max_nn, r0):
    """The smallest radius r0 * 1.25^k at which at least 60 % of the radius neighbourhoods exceed max_nn."""
    tree = cKDTree(P.T)
    r = r0
    while np.mean(tree.query_ball_point(P.T, r, return_length=True) > max_nn) < 0.6:
        r *= 1.25
    return r


@pytest.mark.parametrize("max_nn", [3, 16, 30, 32])
@pytest.mark.parametrize("cloud", ["bunny", "surface"])
def test_hybrid_vs_restatement(bunny, surface, cloud, max_nn):
    P, r0, vp = (bunny, 0.05, (0.0, 0.0, 0.0)) if cloud == "bunny" else (surface, 0.01, (0.0, 0.0, 10.0))
    r = capping_radius(P, max_nn, r0)
    want, frag, sizes = NR.hybrid_normals(P, r, max_nn, vp, return_sizes=True)
    capped = float(np.mean(sizes > max_nn))
    assert capped >= 0.5, capped
    got = features.normals(P, r, max_nn, viewpoint=vp)
    share = check_normals(got, want, frag, 0.05)
    assert not same(got, features.normals(P, r, viewpoint=vp))
    print(f"r={r:.4f} capped={capped:.3f} fragile={share:.4f}")


def test_hybrid_exact_ties_at_the_cap():
    """Integer coordinates: FP32 distances are exact integers, so the max_nn-th and (max_nn + 1)-th candidates often
    tie exactly; the lower index wins on both sides."""
    P = tied_cloud()
    shares = []
    for max_nn in (8, 20, 32):
        r = capping_radius(P, max_nn, 2.3)                           # r^2 stays clear of the integers
        ii, jj, d2, _, _ = OF.neighbours(P, r)
        sizes = np.bincount(ii, minlength=P.shape[1])
        start = np.concatenate([[0], np.cumsum(sizes)])
        k = np.flatnonzero(sizes > max_nn)
        tie = [np.sort(d2[start[i]:start[i + 1]])[max_nn - 1] == np.sort(d2[start[i]:start[i + 1]])[max_nn] for i in k]
        assert np.mean(tie) > 0.2 and k.size > 0.5 * P.shape[1]   # the premise
        want, frag = NR.hybrid_normals(P, r, max_nn)
        got = features.normals(P, r, max_nn)
        shares.append(check_normals(got, want, frag, 0.05))
    print("fragile share per max_nn:", shares)


def test_hybrid_more_duplicates_than_max_nn():
    """40 copies of one point among 2000: with max_nn = 16 each copy keeps the 16 lowest-index copies (d^2 = 0), so
    copies of higher index leave themselves out; their covariance is zero (fragile).  Everything else must match."""
    S = synth.make_surface(2000, 4)
    rng = np.random.default_rng(8)
    P = np.concatenate([S, np.repeat(S[:, :1], 39, axis=1)], axis=1)[:, rng.permutation(2039)]
    ii, jj, _, _ = NR.hybrid_neighbours(P, 0.12, 16)
    copies = np.flatnonzero((P == S[:, :1]).all(axis=0))
    assert copies.size == 40 and np.isin(jj[ii == copies[-1]], copies[:16]).all()
    want, frag = NR.hybrid_normals(P, 0.12, 16)
    got = features.normals(P, 0.12, 16)
    check_normals(got, want, frag, 0.05)


def test_hybrid_without_a_binding_cap_is_the_radius_mode(bunny):
    r = 0.08
    _, _, sizes = NR.hybrid_normals(bunny, r, 32, return_sizes=True)
    assert 3 < sizes.max() <= 32 and (sizes >= 3).mean() > 0.9
    want = features.normals(bunny, r)
    for max_nn in (max(3, int(sizes.max())), 16, 32):
        assert same(features.normals(bunny, r, int(max_nn)), want)
    for n in (1, 2, 3, 5, 32):                                    # the whole cloud is the neighbourhood
        P = cap(n, 200 + n)
        assert same(features.normals(P, 1.0, 32), features.normals(P, 1.0))
        assert same(features.normals(P, 1.0, max(3, n)), features.normals(P, 1.0))


# ---- determinism, host and device -----------------------------------------------------------------------------------

def test_device_entry_dirty_workspace_side_stream(bunny, surface):
    """psulvsb_normals with the caller's workspace pre-filled with 0xFF, reused for smaller clouds, on a non-default
    stream, twice: bit-identical every time and to psulvsb_normals_host."""
    import torch

    L = capi.lib()
    big = surface[:, :20000]
    work = torch.full((int(L.psulvsb_normals_workspace_bytes(big.shape[1])),), 0xFF, dtype=torch.uint8,
                      device="cuda")
    side = torch.cuda.Stream()
    vp = (C.c_double * 3)(0.0, 0.0, 10.0)
    for P, r in ((big, 0.05), (bunny, 0.08), (cap(129, 7), 0.06), (cap(33, 8), 1.0)):
        n = P.shape[1]
        d_pts = stages.to_device_points(P)
        for max_nn in (0, 3, 30):
            outs = []
            for _ in range(2):
                out = torch.full((n, 3), 7.0, dtype=torch.float64, device="cuda")
                torch.cuda.synchronize()
                capi.check(L.psulvsb_normals(side.cuda_stream, d_pts.data_ptr(), n, r, max_nn, vp, work.data_ptr(),
                                             out.data_ptr()))
                side.synchronize()
                outs.append(out.cpu().numpy().T)
                work.fill_(0xFF)
            assert same(outs[0], outs[1])
            assert same(outs[0], features.normals(P, r, max_nn, viewpoint=(0.0, 0.0, 10.0))), (n, max_nn)
            with torch.cuda.stream(side):
                dn = features.normals_device(d_pts, r, max_nn, viewpoint=(0.0, 0.0, 10.0), work=work)
            side.synchronize()
            assert same(dn.cpu().numpy().T, outs[0])


# ---- batches --------------------------------------------------------------------------------------------------------

def mixed(bunny):
    return [bunny, cap(129, 1), np.zeros((3, 0)), cap(1, 2), synth.make_surface(5000, 3), np.zeros((3, 0)),
            cap(33, 4), cap(2, 5)]


@pytest.mark.parametrize("max_nn", [0, 16])
def test_batch_items_equal_single_calls(bunny, max_nn):
    clouds = mixed(bunny)
    vps = [(0.0, 0.0, 10.0 * (c % 3 - 1)) for c in range(len(clouds))]
    r = 0.08
    want = [features.normals(P, r, max_nn, viewpoint=v) for P, v in zip(clouds, vps)]
    for order in (list(range(len(clouds))), list(reversed(range(len(clouds))))):
        got = features.normals_batch([clouds[c] for c in order], r, max_nn, [vps[c] for c in order])
        for k, c in enumerate(order):
            assert got[k].shape == want[c].shape and same(got[k], want[c]), (order, c)
    for P, v, w in zip(clouds, vps, want):                        # B = 1
        assert same(features.normals_batch([P], r, max_nn, [v])[0], w)


def test_batch_viewpoints_belong_to_each_cloud(bunny):
    """The same cloud twice with opposite viewpoints: the same normals up to sign, each flipped towards its own."""
    vps = [(0.0, 0.0, 100.0), (0.0, 0.0, -100.0)]
    got = features.normals_batch([bunny, bunny], 0.08, 16, vps)
    ok = ~np.isnan(got[0][0])
    assert ok.mean() > 0.9 and same(np.abs(got[0]), np.abs(got[1]))
    for g, v in zip(got, vps):
        assert (((np.array(v)[:, None] - bunny) * g).sum(axis=0)[ok] >= 0).all()
    assert np.mean(got[0][2, ok] != got[1][2, ok]) > 0.5


@pytest.mark.parametrize("max_nn", [0, 30])
def test_batch_592_clouds_of_5000_on_the_device(max_nn):
    import torch

    clouds = [synth.make_surface(5000, b) for b in range(592)]
    d = [stages.to_device_points(P) for P in clouds]
    vps = [(0.0, 0.0, 5.0 + b) for b in range(592)]
    r = 0.08 if max_nn == 0 else 0.1
    allp, views = features.normals_batch_device(d, r, max_nn, vps)
    torch.cuda.synchronize()
    assert allp.shape == (592 * 5000, 3)
    for b in range(592):
        single = features.normals_device(d[b], r, max_nn, vps[b])
        assert torch.equal(views[b].isnan(), single.isnan())
        assert same(views[b].cpu().numpy(), single.cpu().numpy()), b
    for b in (0, 591):                                            # the host variants agree
        assert same(features.normals_batch([clouds[b]], r, max_nn, [vps[b]])[0], views[b].cpu().numpy().T)
