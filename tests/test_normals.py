"""CPU-side checks of the normals-alone entry points (psulvsb_normals*, csrc/k8_features.cu): the hybrid restatement
(tests/normals_restatement.py) pinned on hand-built clouds, the workspace sizes against FPFH's, and every argument
refusal before any device work."""
import ctypes as C

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from oracle import features as OF
from psulvsb_b200 import capi, features, synth
from tests import normals_restatement as NR

BUF = np.zeros(4 * 33)


def clouds(specs):
    arr = (capi.FpfhCloud * max(len(specs), 1))()
    for c, spec in enumerate(specs):
        arr[c].pts, arr[c].n = BUF.ctypes.data, 4
        for k, v in spec.items():
            setattr(arr[c], k, v)
    return arr


# ---- the restatement ------------------------------------------------------------------------------------------------

def test_hybrid_restatement_without_a_binding_cap_is_the_radius_restatement():
    P = synth.make_surface(1500, 3)
    r = 0.2
    _, _, sizes = NR.hybrid_normals(P, r, 32, return_sizes=True)
    cap = int(sizes.max())
    assert cap > 32                                            # the premise: radius 0.2 holds about 47 points
    want, wfrag = OF.radius_normals(P, r, (0.0, 0.0, 5.0))
    got, gfrag = NR.hybrid_normals(P, r, cap, (0.0, 0.0, 5.0))
    assert np.array_equal(got, want, equal_nan=True) and np.array_equal(gfrag, wfrag)
    capped, _ = NR.hybrid_normals(P, r, 16, (0.0, 0.0, 5.0))
    assert not np.array_equal(capped, want, equal_nan=True)


def test_hybrid_restatement_exact_ties_keep_the_lower_indices():
    """Point 4 sits at the origin; six points at FP32 distance exactly 1 (the unit axes), one at 0.5 and one far; radius
    1.5.  With max_nn = 5, point 4 keeps itself (d^2 = 0), the 0.5 point and the three lowest indices of the six tied points."""
    P = np.zeros((3, 9))
    axes = {0: (1, 0, 0), 7: (-1, 0, 0), 2: (0, 1, 0), 8: (0, -1, 0), 5: (0, 0, 1), 1: (0, 0, -1)}
    for j, v in axes.items():
        P[:, j] = v
    P[:, 3] = (0.5, 0.0, 0.0)
    P[:, 6] = (50.0, 50.0, 50.0)
    ii, jj, sizes, frag = NR.hybrid_neighbours(P, 1.5, 5)
    assert sizes[4] == 8
    assert sorted(jj[ii == 4]) == [0, 1, 2, 3, 4]            # 4 itself, 3 at 0.5, then ties 0 < 1 < 2 of {0,1,2,5,7,8}
    assert not frag[4]                                         # an exact tie is no near-tie
    assert sizes[6] == 1 and list(jj[ii == 6]) == [6]


def test_hybrid_restatement_duplicates_can_push_the_point_out():
    """Five copies of one point: with max_nn = 3 the copy with the highest index keeps the three lowest copies (all at
    d^2 = 0), not itself -- the k-NN estimator's rule."""
    P = np.concatenate([np.zeros((3, 5)), np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0]]).T], axis=1)
    ii, jj, _, _ = NR.hybrid_neighbours(P, 2.0, 3)
    assert list(jj[ii == 4]) == [0, 1, 2]


def test_hybrid_restatement_small_clouds():
    """max_nn = 3 on 4 points of a tetrahedron: every point keeps itself and its two nearest, so its normal is the
    normal of that triangle.  Isolated points and clouds under 3 points give NaN."""
    P = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 2.0, 0.0], [0.0, 0.0, 3.0]]).T
    got, _ = NR.hybrid_normals(P, 10.0, 3, viewpoint=(-5.0, -5.0, -5.0))
    for i in range(4):
        d = ((P - P[:, [i]]) ** 2).sum(axis=0)
        tri = np.argsort(d, kind="stable")[:3]
        nrm = np.cross(P[:, tri[1]] - P[:, tri[0]], P[:, tri[2]] - P[:, tri[0]])
        nrm /= np.linalg.norm(nrm)
        assert abs(abs(float(nrm @ got[:, i])) - 1.0) < 1e-12, i
        assert float((np.array([-5.0, -5.0, -5.0]) - P[:, i]) @ got[:, i]) >= 0.0
    far = np.concatenate([P, [[100.0], [0.0], [0.0]]], axis=1)
    got, _ = NR.hybrid_normals(far, 10.0, 3)
    assert np.isnan(got[:, 4]).all() and not np.isnan(got[:, :4]).any()
    for n in (0, 1, 2):
        got, _ = NR.hybrid_normals(P[:, :n], 10.0, 3)
        assert got.shape == (3, n) and np.isnan(got).all()


# ---- workspace sizes ------------------------------------------------------------------------------------------------

def test_workspace_answers_from_sizes_and_stays_within_fpfh():
    L = capi.lib()
    for n in (0, 1, 127, 128, 129, 5000, 50000, 500000):
        w = L.psulvsb_normals_workspace_bytes(n)
        assert w == L.psulvsb_normals_workspace_bytes(n)
        assert w <= L.psulvsb_fpfh_workspace_bytes(n)
        if n:
            assert w < L.psulvsb_fpfh_workspace_bytes(n)      # no descriptor counts
    assert L.psulvsb_normals_workspace_bytes(-1) == 0

    def nw(sizes, **kw):
        return L.psulvsb_normals_batch_workspace_bytes(clouds([dict(n=n, **kw) for n in sizes]), len(sizes))

    def fw(sizes):
        return L.psulvsb_fpfh_batch_workspace_bytes(clouds([{"n": n} for n in sizes]), len(sizes))

    base = [5000, 129, 0, 1]
    assert nw(base) == nw(base, pts=None) == nw(base) > 0     # the pointers do not matter
    assert nw(base) <= fw(base) and nw([50000] + base[1:]) > nw(base)
    assert nw([5000]) == L.psulvsb_normals_workspace_bytes(5000)
    assert nw([5000] * 592) <= fw([5000] * 592)
    assert nw([]) == 0 and nw([-1, 5]) == 0 and L.psulvsb_normals_batch_workspace_bytes(None, 3) == 0


# ---- refusals -------------------------------------------------------------------------------------------------------

def four(sel=(0, 1, 2, 3), r=0.1, max_nn=0, n=4, arr=None, B=1, pts=True, work=True, out=True, vp=True):
    """Return codes of psulvsb_normals, _host, _batch and _batch_host (the indices in `sel` only: a call that is not
    refused would run on host pointers)."""
    L = capi.lib()
    p = BUF.ctypes.data if pts else None
    w = BUF.ctypes.data if work else None
    o = BUF.ctypes.data if out else None
    v = (C.c_double * 3)(0.0, 0.0, 0.0) if vp else None
    arr = clouds([{}]) if arr is None else arr
    calls = (lambda: L.psulvsb_normals(None, p, n, r, max_nn, v, w, o),
             lambda: L.psulvsb_normals_host(p, n, r, max_nn, v, o),
             lambda: L.psulvsb_normals_batch(None, arr, B, r, max_nn, w, o),
             lambda: L.psulvsb_normals_batch_host(arr, B, r, max_nn, o))
    return tuple(calls[k]() for k in sel)


def test_refusals_come_before_any_device_work():
    L = capi.lib()
    inv = (capi.ERR_INVALID,) * 4
    for r in (0.0, -1.0, float("nan"), float("inf"), -float("inf")):
        assert four(r=r) == inv, r
    for k in (-1, 1, 2, 33, 64, 1 << 30):
        assert four(max_nn=k) == inv, k
    assert four(out=False) == inv
    assert four((0, 1), pts=False) == inv[:2]
    assert four((0, 2), work=False) == inv[:2]
    assert four((0, 1), n=-1) == inv[:2]
    assert four((2, 3), B=-1) == inv[:2]
    for spec in ({"n": -1}, {"pts": None}):                   # the bad cloud is the last of three
        assert four((2, 3), arr=clouds([{}, {}, spec]), B=3) == inv[:2], spec
    assert L.psulvsb_normals_batch(None, None, 1, 0.1, 0, BUF.ctypes.data, BUF.ctypes.data) == capi.ERR_INVALID
    assert L.psulvsb_normals_batch_host(None, 1, 0.1, 0, BUF.ctypes.data) == capi.ERR_INVALID
    big = 2 ** 30
    assert four((2, 3), arr=clouds([{"n": big}, {"n": big}]), B=2) == (capi.ERR_UNSUPPORTED,) * 2
    # B = 0 does nothing (and needs no pointer); the radius and max_nn are still checked
    assert four((2, 3), B=0) == (capi.OK, capi.OK)
    assert (L.psulvsb_normals_batch(None, None, 0, 0.1, 0, None, None),
            L.psulvsb_normals_batch_host(None, 0, 0.1, 32, None)) == (capi.OK, capi.OK)
    assert L.psulvsb_normals_batch(None, None, 0, 0.1, 2, None, None) == capi.ERR_INVALID
    if L.psulvsb_device_count() == 0:
        ok = (capi.ERR_NO_DEVICE,) * 4
        for k in (0, 3, 32):
            assert four(max_nn=k) == ok
        assert four(vp=False) == ok                        # the viewpoint may be NULL
        with pytest.raises(capi.PsulvsbError):
            features.normals(np.zeros((3, 4)), 0.1)
        with pytest.raises(capi.PsulvsbError):
            features.normals_batch([np.zeros((3, 4))], 0.1, 16)
    assert features.normals_batch([], 0.1) == []
    with pytest.raises(capi.PsulvsbError) as e:
        features.normals(np.zeros((3, 4)), 0.1, max_nn=2)
    assert e.value.code == capi.ERR_INVALID
