"""The correspondence kernels (csrc/k8_features.cu) and the k-NN normals (csrc/k6_normals.cu) at the shapes where
kernels go wrong, against the numpy restatements (oracle/features.py, oracle/prefilter.py) and, for the descriptor
nearest neighbour, against a float64 brute force.

FPFH and radius normals: clouds of 1 ... 129 points whose 27 neighbour cells collide in 1 ... 256 buckets, a cloud
inside one grid cell, cell sizes set by r_n, negative and far-from-origin cells, duplicated points and a reused,
dirty workspace on a side stream.  Nearest neighbour: the 64-column tile, the 2048-column range and the 256-row CTA
boundaries, empty sides, all-tied and overflowing distances.  Matcher: tuple tests over two 2^20-trial chunks, one-way
lists with n_s != n_t, degenerate lists and the capacity error.  k-NN normals: several shared-memory tiles,
k in {3, 20, 32}, n < k, n < 3, exact ties at the k-th neighbour and refused k.

The bars: a descriptor within L1 1e-3 of the restatement unless fragile (and within 1e-3 plus the restatement's
bound on what its fragile pairs can move, unless a hard flag reaches it); a normal with the same NaN pattern and
|cos| > 1 - 1e-6 with the same sign at every point that is not fragile."""
import ctypes as C
import os

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from oracle import features as OF
from oracle import prefilter as OP
from psulvsb_b200 import capi, features, io, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bunny():
    return np.load(os.path.join(ROOT, "tests", "golden", "bunny_res3.npz"))["vertices"].astype(np.float64) * 10


@pytest.fixture(scope="module")
def bunny_desc(bunny):
    return features.fpfh(bunny, 0.08, 0.15)[0]


def cap(n, seed, radius=0.1):
    """n jittered points on a spherical cap (curved everywhere), centred on the origin: the cloud straddles the
    grid's cells -1 and 0 on every axis."""
    rng = np.random.default_rng(seed)
    th = np.arccos(rng.uniform(np.cos(1.0), 1.0, n))
    ph = rng.uniform(0, 2 * np.pi, n)
    P = radius * np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)])
    return P - P.mean(axis=1, keepdims=True)


def check_normals(got, want, fragile, max_fragile):
    assert np.array_equal(np.isnan(got[0]), np.isnan(want[0]))
    ok = ~np.isnan(want[0]) & ~fragile
    assert np.allclose(np.linalg.norm(got[:, ok], axis=0), 1.0, atol=1e-9)
    dot = (got[:, ok] * want[:, ok]).sum(axis=0)
    assert (dot > 1 - 1e-6).all(), (np.flatnonzero(ok)[np.argmin(dot)], dot.min())
    share = fragile.mean() if fragile.size else 0.0
    assert share <= max_fragile, share
    return share


def check_fpfh(got_f, got_n, P, rn, rf, viewpoint=(0.0, 0.0, 0.0), max_fragile=0.05):
    """Descriptors and radius normals against the restatement; returns the fragile shares (normals, descriptors)."""
    want_n, nfrag = OF.radius_normals(P, rn, viewpoint)
    want, _, frag, hard, soft = OF.fpfh(P, rn, rf, viewpoint, bounds=True)
    shares = (check_normals(got_n, want_n, nfrag, max_fragile),)
    l1 = np.abs(got_f.astype(np.float64) - want).sum(axis=1)
    assert not np.isnan(l1).any()
    assert l1[~frag].max(initial=0) <= 1e-3, (np.argmax(np.where(frag, 0, l1)), l1[~frag].max())
    assert (l1 <= 1e-3 + soft)[~hard].all(), np.argmax(np.where(hard, 0, l1 - soft))
    share = float(frag.mean()) if frag.size else 0.0
    assert share <= max_fragile and (hard.mean() if hard.size else 0.0) <= 0.05, (share, hard.mean())
    return shares + (share,)


# ---- FPFH and radius normals ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 7, 33, 127, 128, 129])
def test_fpfh_tiny_clouds_with_colliding_cells(n):
    """r_f covers the whole cloud (cell size 1, up to 8 occupied cells) and n sets nb = 2^ceil(log2 n) buckets, so
    the 27 cells of a walk share buckets: the walk's de-duplication decides K and the neighbourhoods."""
    P = cap(n, 100 + n)
    rn = 1.0 if n < 33 else 0.06                  # below 33 points every normal uses the whole cloud
    vp = (0.0, 0.0, 10.0)
    got, gn = features.fpfh(P, rn, 1.0, viewpoint=vp)
    shares = check_fpfh(got, gn, P, rn, 1.0, vp)
    if n <= 2:
        assert np.isnan(gn).all() and (got == 0).all()
    else:
        assert not np.isnan(gn).any() and (got.sum(axis=1) > 0).all()
    print("fragile share (normals, descriptors):", shares)


def test_fpfh_one_bucket_holds_the_cloud(bunny):
    """The bunny inside one grid cell (r_f larger than its extent): every point lands in one bucket, which
    k8_grid_order ranks by index, and every neighbourhood is the whole cloud."""
    P = bunny - bunny.min(axis=1, keepdims=True) + 0.01
    rf = 1.2 * float(np.linalg.norm(np.ptp(P, axis=1)))
    got, gn = features.fpfh(P, 0.08, rf)
    # with 1889 neighbours per point every descriptor has some fragile pair: the hard flags and the soft bound decide
    shares = check_fpfh(got, gn, P, 0.08, rf, max_fragile=1.0)
    print("fragile share (normals, descriptors):", shares)


@pytest.mark.parametrize("rn,rf", [(0.15, 0.08), (0.1, 0.1)])
def test_fpfh_cell_size_set_by_normal_radius(bunny, rn, rf):
    got, gn = features.fpfh(bunny, rn, rf)
    print("fragile share (normals, descriptors):", check_fpfh(got, gn, bunny, rn, rf))


@pytest.mark.parametrize("shift", [(0.0, 0.0, 0.0), (1e3, -1e3, 5e2)])
def test_fpfh_negative_and_far_cells(bunny, shift):
    P = bunny - bunny.mean(axis=1, keepdims=True) + np.array(shift)[:, None]
    got, gn = features.fpfh(P, 0.08, 0.15)
    print("fragile share (normals, descriptors):", check_fpfh(got, gn, P, 0.08, 0.15))


def test_fpfh_duplicate_points():
    """About 5 % of a surface duplicated: copies count in K and in the normals' neighbourhoods, and are skipped as
    pairs (zero length) and in the FPFH sum (d^2 == 0)."""
    S = synth.make_surface(4000, 21)
    rng = np.random.default_rng(5)
    P = np.concatenate([S, S[:, rng.choice(4000, 200, replace=False)]], axis=1)[:, rng.permutation(4200)]
    got, gn = features.fpfh(P, 0.06, 0.1)
    # a copy at distance 0 has its own weight-1/d^2 neighbours: 5.8 % of the descriptors carry a soft bound > 5e-4
    print("fragile share (normals, descriptors):", check_fpfh(got, gn, P, 0.06, 0.1, max_fragile=0.08))


def test_fpfh_device_entry_dirty_workspace_side_stream(bunny):
    """psulvsb_fpfh with the caller's workspace, pre-filled with 0xFF and reused for a smaller cloud after a larger
    one, on a non-default stream: bit-identical to psulvsb_fpfh_host."""
    import torch

    from psulvsb_b200 import stages

    L = capi.lib()
    clouds = [bunny, cap(129, 7), cap(33, 8)]
    work = torch.full((int(L.psulvsb_fpfh_workspace_bytes(bunny.shape[1])),), 0xFF, dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    vp = (C.c_double * 3)(0.0, 0.0, 10.0)
    for P in clouds:
        n = P.shape[1]
        d_pts = stages.to_device_points(P)
        feats = torch.full((n, 33), float("nan"), dtype=torch.float32, device="cuda")
        normals = torch.full((n, 3), 7.0, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        assert L.psulvsb_fpfh_workspace_bytes(n) <= work.numel()
        capi.check(L.psulvsb_fpfh(side.cuda_stream, d_pts.data_ptr(), n, 0.06, 0.12, vp, work.data_ptr(),
                                  normals.data_ptr(), feats.data_ptr()))
        side.synchronize()
        want, wn = features.fpfh(P, 0.06, 0.12, viewpoint=(0.0, 0.0, 10.0))
        assert np.array_equal(feats.cpu().numpy().view(np.uint32), want.view(np.uint32))
        assert np.array_equal(normals.cpu().numpy().T, wn, equal_nan=True)


# ---- two-way descriptor nearest neighbour ---------------------------------------------------------------------------

def brute64(fs, ft):
    """Exact float64 squared distances of float32 descriptors (differences and squares are exact in float64)."""
    a, b = fs.astype(np.float64), ft.astype(np.float64)
    return ((a[:, None, :] - b[None, :, :]) ** 2).sum(axis=2)


def check_picks_f64(fs, ft, a, b):
    """Every pick is a minimum of the exact float64 distances, up to FP32 accumulation (1e-5 relative)."""
    for r0 in range(0, fs.shape[0], 512):
        D = brute64(fs[r0:r0 + 512], ft)
        rows = np.arange(D.shape[0])
        assert (D[rows, a[r0:r0 + 512]] <= D.min(axis=1) * (1 + 1e-5)).all()
    for c0 in range(0, ft.shape[0], 512):
        D = brute64(fs, ft[c0:c0 + 512])
        cols = np.arange(D.shape[1])
        assert (D[b[c0:c0 + 512], cols] <= D.min(axis=0) * (1 + 1e-5)).all()


@pytest.mark.parametrize("ns,nt", [(255, 63), (256, 64), (257, 65), (513, 2047), (300, 2048), (300, 2049),
                                   (1, 4097), (4097, 1)])
def test_feature_nn_tile_and_range_boundaries(bunny_desc, ns, nt):
    rng = np.random.default_rng(ns * 31 + nt)
    f = bunny_desc
    fs = f[rng.integers(0, f.shape[0], ns)] + rng.normal(0, 0.2, (ns, 33)).astype(np.float32)
    ft = f[rng.integers(0, f.shape[0], nt)] + rng.normal(0, 0.2, (nt, 33)).astype(np.float32)
    ft[1::5] = fs[rng.integers(0, ns, ft[1::5].shape[0])]      # exact matches for some columns
    a, b = features.nearest_neighbours(fs, ft)
    wa, wb, fa, fb = OF.nearest_neighbours(fs, ft)
    assert np.array_equal(a[~fa], wa[~fa]) and np.array_equal(b[~fb], wb[~fb])
    assert fa.mean() <= 0.05 and fb.mean() <= 0.05, (fa.mean(), fb.mean())
    check_picks_f64(fs, ft, a, b)
    print("fragile share (rows, columns):", fa.mean(), fb.mean())


@pytest.mark.parametrize("ns,nt", [(0, 5), (5, 0)])
def test_feature_nn_device_entry_empty_side(ns, nt):
    import torch

    d_fs = torch.rand((ns, 33), dtype=torch.float32, device="cuda")
    d_ft = torch.rand((nt, 33), dtype=torch.float32, device="cuda")
    a, b = features.nearest_neighbours_device(d_fs, d_ft)
    torch.cuda.synchronize()
    assert a.shape == (ns,) and b.shape == (nt,)
    assert (a.cpu() == -1).all() and (b.cpu() == -1).all()


@pytest.mark.parametrize("scale", [None, 1e19])
def test_feature_nn_all_tied(scale):
    """Every distance ties -- at 0 (identical descriptors) or at inf (descriptors scaled by 1e19 overflow FP32):
    both directions answer index 0, across tiles, column ranges and row CTAs."""
    ns, nt = 600, 2100
    if scale is None:
        fs = np.full((ns, 33), 3.25, np.float32)
        ft = fs[:1].repeat(nt, axis=0)
    else:
        rng = np.random.default_rng(3)
        fs = (rng.uniform(0, 100, (ns, 33)) * scale).astype(np.float32)
        ft = (rng.uniform(0, 100, (nt, 33)) * scale).astype(np.float32)
        assert np.isinf(OF.descriptor_distances(fs, ft)).all()
    a, b = features.nearest_neighbours(fs, ft)
    assert (a == 0).all() and (b == 0).all()
    wa, wb, _, _ = OF.nearest_neighbours(fs, ft)
    assert (wa == 0).all() and (wb == 0).all()
    if scale is None:
        check_picks_f64(fs, ft, a, b)


# ---- matcher --------------------------------------------------------------------------------------------------------

def pass_trials(src, tgt, corr, scale, seed):
    """Indices of the passing tuple trials among all 100 * ncorr (the restatement's rule, every trial)."""
    n = corr.shape[0]
    r = OF.tuple_draws(seed, 0, 100 * n, n)
    s32, t32 = OF._f32(src), OF._f32(tgt)
    s = np.float32(scale)
    ok = np.ones(100 * n, dtype=bool)
    for e in range(3):
        a, b = r[:, e], r[:, (e + 1) % 3]
        li = np.sqrt(OF.sqdist32(s32[corr[a, 0]], s32[corr[b, 0]]))
        lj = np.sqrt(OF.sqdist32(t32[corr[a, 1]], t32[corr[b, 1]]))
        ok &= ((li * s).astype(np.float32) < lj) & (lj < (li / s).astype(np.float32))
    return np.flatnonzero(ok)


@pytest.mark.parametrize("scale,seed,where", [(0.95, 0, "under 1000 in all"), (0.935, 1, "1000th in chunk 2")])
def test_tuple_test_over_two_chunks(scale, seed, where):
    """11 000 identity correspondences (fs == ft, distinct descriptors) between two independent random clouds:
    1.1 M trials, two 2^20-trial chunks, few passes.  The kept count carries from the first chunk into the second."""
    n, chunk = 11000, 1 << 20
    rng = np.random.default_rng(1)
    src, tgt = rng.uniform(-1, 1, (3, n)), rng.uniform(-1, 1, (3, n))
    f = rng.uniform(0, 100, (n, 33)).astype(np.float32)
    corr = np.stack([np.arange(n), np.arange(n)], axis=1)
    passes = pass_trials(src, tgt, corr, scale, seed)
    assert (passes < chunk).sum() < 1000 and (passes >= chunk).any()
    if where == "under 1000 in all":
        assert passes.size < 1000
    else:
        assert passes.size >= 1000 and passes[999] >= chunk
    assert np.array_equal(features.match(src, tgt, f, f, crosscheck=True), corr)
    got = features.match(src, tgt, f, f, crosscheck=True, tuple_test=True, tuple_scale=scale, seed=seed)
    want, fragile = OF.tuple_test(src, tgt, corr, scale, seed)
    assert got.shape[0] == 3 * min(1000, passes.size)
    if fragile:
        pytest.skip("a trial near a ratio bound decides the kept set")
    assert np.array_equal(got, want)


@pytest.mark.parametrize("ns,nt", [(2500, 1700), (1700, 2500)])
def test_one_way_and_mutual_lists_unequal_sides(bunny_desc, ns, nt):
    rng = np.random.default_rng(ns)
    f = bunny_desc
    fs = f[rng.integers(0, f.shape[0], ns)] + rng.normal(0, 0.5, (ns, 33)).astype(np.float32)
    ft = f[rng.integers(0, f.shape[0], nt)] + rng.normal(0, 0.5, (nt, 33)).astype(np.float32)
    src, tgt = rng.uniform(-1, 1, (3, ns)), rng.uniform(-1, 1, (3, nt))
    nn_t, nn_s = features.nearest_neighbours(fs, ft)
    wa, wb, fa, fb = OF.nearest_neighbours(fs, ft)
    assert not fa.any() and not fb.any()
    assert np.array_equal(nn_t, wa) and np.array_equal(nn_s, wb)
    assert np.setdiff1d(np.arange(ns), nn_s).size > 0          # some sources are nobody's nearest neighbour
    for cross in (True, False):
        got = features.match(src, tgt, fs, ft, crosscheck=cross)
        assert np.array_equal(got, OF.match_list(wa, wb, cross))


@pytest.mark.parametrize("n", [1, 2])
def test_tuple_test_degenerate_lists(n):
    """ncorr 1 or 2: every triangle repeats a vertex, so no trial passes."""
    rng = np.random.default_rng(n)
    P = rng.uniform(-1, 1, (3, n))
    f = rng.uniform(0, 100, (n, 33)).astype(np.float32)
    assert features.match(P, P, f, f, crosscheck=True).shape == (n, 2)
    got = features.match(P, P, f, f, crosscheck=True, tuple_test=True)
    want, _ = OF.tuple_test(P, P, np.stack([np.arange(n)] * 2, axis=1), 0.95, 0)
    assert got.shape == (0, 2) and want.shape == (0, 2)


@pytest.mark.parametrize("ns,nt", [(0, 5), (5, 0)])
def test_match_empty_side(ns, nt):
    rng = np.random.default_rng(0)
    for tuple_test in (False, True):
        got = features.match(rng.uniform(size=(3, ns)), rng.uniform(size=(3, nt)),
                             rng.uniform(size=(ns, 33)), rng.uniform(size=(nt, 33)), crosscheck=False,
                             tuple_test=tuple_test)
        assert got.shape == (0, 2)


def test_match_capacity_one_short():
    rng = np.random.default_rng(4)
    ns, nt = 300, 200
    src, tgt = np.asfortranarray(rng.uniform(-1, 1, (3, ns))), np.asfortranarray(rng.uniform(-1, 1, (3, nt)))
    fs = rng.uniform(0, 100, (ns, 33)).astype(np.float32)
    ft = rng.uniform(0, 100, (nt, 33)).astype(np.float32)
    L = capi.lib()
    for cross, tuple_test in ((1, 0), (0, 0), (1, 1)):
        full = features.match(src, tgt, fs, ft, crosscheck=bool(cross), tuple_test=bool(tuple_test), tuple_scale=0.5)
        need = full.shape[0]
        assert need > 0
        out = np.full((need, 2), -7, dtype=np.int32)
        n = C.c_longlong(-1)
        rc = L.psulvsb_match_host(src.ctypes.data, ns, tgt.ctypes.data, nt, fs.ctypes.data, ft.ctypes.data, cross,
                                  tuple_test, 0.5, 0, out.ctypes.data, need - 1, C.byref(n))
        assert rc == capi.ERR_CAPACITY and n.value == need
        assert (out[need - 1] == -7).all()                    # nothing written past the capacity
        rc = L.psulvsb_match_host(src.ctypes.data, ns, tgt.ctypes.data, nt, fs.ctypes.data, ft.ctypes.data, cross,
                                  tuple_test, 0.5, 0, out.ctypes.data, need, C.byref(n))
        assert rc == capi.OK and n.value == need and np.array_equal(out, full)


# ---- k-NN normals ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [1, 2, 3, 10, 1025, 1889, 5000])
def test_knn_normals_vs_restatement(n):
    if n == 1889:
        P = np.load(os.path.join(ROOT, "tests", "golden", "bunny_res3.npz"))["vertices"].astype(np.float64)
    else:
        P = synth.make_surface(n, 60 + n)
    shares = []
    for k in (3, 20, 32):
        got = io.estimate_normals(P, k=k)
        want, fragile = OP.knn_pca_normals(P, k=k, return_fragile=True)
        if n < 3:
            assert np.isnan(got).all() and np.isnan(want).all()
        shares.append(check_normals(got, want, fragile, 0.05))
    print("fragile share per k:", shares)


def tied_cloud():
    """1500 points with integer coordinates on a curved sheet, 5 % of them duplicated: FP32 distances are exact
    integers, so the k-th and (k+1)-th neighbours often tie exactly, between different points."""
    rng = np.random.default_rng(12)
    xy = rng.choice(60 * 60, 1425, replace=False)
    x, y = (xy // 60 - 30).astype(np.float64), (xy % 60 - 30).astype(np.float64)
    P = np.stack([x, y, np.floor((x * x - 0.5 * y * y) / 20.0 + x * y / 30.0)])
    P = np.concatenate([P, P[:, rng.choice(1425, 75, replace=False)]], axis=1)
    return P[:, rng.permutation(P.shape[1])]


def test_knn_normals_exact_ties_go_to_the_lower_index():
    P = tied_cloud()
    Pf = P.astype(np.float32)
    shares = []
    for k in (8, 20, 32):                                        # (k = 3 picks collinear triples on this grid)
        d = np.sort(OP.knn_sqdist32(Pf, np.arange(P.shape[1])), axis=1)
        assert (d[:, k - 1] == d[:, k]).mean() > 0.2            # the premise: ties at the k-th neighbour are common
        got = io.estimate_normals(P, k=k)
        want, fragile = OP.knn_pca_normals(P, k=k, return_fragile=True)
        shares.append(check_normals(got, want, fragile, 0.05))
    print("fragile share per k:", shares)


@pytest.mark.parametrize("k", [2, 33])
def test_knn_normals_refuse_k(k):
    with pytest.raises(capi.PsulvsbError) as e:
        io.estimate_normals(synth.make_surface(10, 0), k=k)
    assert e.value.code == capi.ERR_INVALID
