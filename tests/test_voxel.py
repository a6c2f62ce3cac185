"""CPU-side checks of the voxel filter (psulvsb_voxel_down_sample*, csrc/k8_voxel.cu): the restatement
(tests/voxel_restatement.py) pinned on hand-built clouds, the workspace sizes, every argument refusal before any device
work, and the kernels' registers, stack frames and spills from an sm_100a compile."""
import os
import re
import subprocess

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from psulvsb_b200 import capi, features
from tests import voxel_restatement as VR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "probabilistic-self-update-line-vector-set-based-point-cloud-registration_b200", "csrc")
BUF = np.zeros(4 * 33)


def clouds(specs):
    arr = (capi.FpfhCloud * max(len(specs), 1))()
    for c, spec in enumerate(specs):
        arr[c].pts, arr[c].n = BUF.ctypes.data, 4
        for k, v in spec.items():
            setattr(arr[c], k, v)
    return arr


def same(a, b):
    return a.shape == b.shape and np.array_equal(a, b)


# ---- the restatement ------------------------------------------------------------------------------------------------

def test_restatement_cells_on_an_integer_lattice():
    """v = 1 on integer points: origin = lo - 0.5, so (p - origin) / v = k + 0.5 exactly and every point is the only one
    of its cell; the output is the input, in input order."""
    rng = np.random.default_rng(1)
    P = rng.permutation(np.stack(np.meshgrid(np.arange(4), np.arange(3), np.arange(5)), 0).reshape(3, -1).T).T
    P = P.astype(np.float64) - 7.0
    fin, c = VR.cells(P, 1.0)
    assert fin.all() and np.array_equal(c, (P - P.min(axis=1, keepdims=True)).astype(np.int64))
    assert same(VR.voxel_down_sample(P, 1.0), np.asfortranarray(P))


def test_restatement_points_exactly_on_cell_boundaries():
    """lo = 0, v = 1: origin = -0.5, so x = k + 0.5 lies exactly on the boundary and goes to cell k + 1 (floor)."""
    P = np.array([[0.0, 0.5, 0.25, 1.5, 1.0], [0.0] * 5, [0.0] * 5])
    _, c = VR.cells(P, 1.0)
    assert list(c[0]) == [0, 1, 0, 2, 1]
    got = VR.voxel_down_sample(P, 1.0)
    want = np.array([[(0.0 + 0.25) / 2, (0.5 + 1.0) / 2, 1.5], [0.0] * 3, [0.0] * 3])
    assert same(got, np.asfortranarray(want))


def test_restatement_duplicates_and_non_finite_points():
    nan, inf = float("nan"), float("inf")
    P = np.array([[5.0, nan, 1.0, 5.0, 1.0, 2.0, -inf],
                  [5.0, 0.0, 1.0, 5.0, 1.0, 2.0, 0.0],
                  [5.0, 0.0, 1.0, 5.0, 1.0, 2.0, 0.0]])
    fin, _ = VR.cells(P, 0.5)
    assert list(fin) == [True, False, True, True, True, True, False]
    assert np.array_equal(VR.origin(P, 0.5), [0.75, 0.75, 0.75])      # NaN and -inf take no part in the bound
    got = VR.voxel_down_sample(P, 0.5)
    assert same(got, np.asfortranarray(np.array([[5.0, 1.0, 2.0]] * 3)))  # first occurrences 0, 2, 5
    assert VR.voxel_down_sample(np.full((3, 4), nan), 1.0).shape == (3, 0)
    assert VR.voxel_down_sample(np.zeros((3, 0)), 1.0).shape == (3, 0)


def test_restatement_all_points_in_one_voxel_sum_in_input_order():
    rng = np.random.default_rng(2)
    P = rng.uniform(0.0, 1.0, (3, 1000)) * np.array([[1e-3], [1.0], [1e3]])
    got = VR.voxel_down_sample(P, 1e4)
    acc = np.zeros(3)
    for k in range(P.shape[1]):
        acc = acc + P[:, k]
    assert same(got, np.asfortranarray((acc / 1000.0)[:, None]))


def test_restatement_saturates_far_cells():
    P = np.array([[0.0, 1e300, 3.0], [0.0, 0.0, 0.0], [0.0, 0.0, 0.0]])
    _, c = VR.cells(P, 1e-10)
    assert c[0, 1] == VR.I64_MAX and c[0, 0] == 0 and c[0, 2] == 30000000000
    assert VR.voxel_down_sample(P, 1e-10).shape == (3, 3)


def test_restatement_bucket_hash_groups_several_voxels():
    """bucket_count(n) buckets for n points: with about 4 points per voxel there are n / 4 voxels in n buckets, and
    some buckets still hold several voxels, which the exact-cell test must keep apart."""
    rng = np.random.default_rng(3)
    P = rng.uniform(0.0, 1.0, (3, 4096))
    assert VR.bucket_count(4096) == 4096 and VR.bucket_count(4097) == 8192 and VR.bucket_count(0) == 1
    assert VR.voxels_per_bucket(P, 1.0 / 10.0) >= 2


# ---- workspace sizes ------------------------------------------------------------------------------------------------

def test_workspace_answers_from_sizes():
    L = capi.lib()
    prev = 0
    for n in (0, 1, 127, 128, 129, 5000, 50000, 500000):
        w = L.psulvsb_voxel_down_sample_workspace_bytes(n)
        assert w == L.psulvsb_voxel_down_sample_workspace_bytes(n) and w >= prev
        prev = w
    assert L.psulvsb_voxel_down_sample_workspace_bytes(-1) == 0

    def vw(sizes, **kw):
        return L.psulvsb_voxel_down_sample_batch_workspace_bytes(clouds([dict(n=n, **kw) for n in sizes]), len(sizes))

    base = [5000, 129, 0, 1]
    assert vw(base) == vw(base, pts=None) > 0                       # the pointers do not matter
    assert vw([50000] + base[1:]) > vw(base)
    assert vw([5000]) == L.psulvsb_voxel_down_sample_workspace_bytes(5000)
    assert vw([5000] * 592) > vw([5000] * 16)
    assert vw([]) == 0 and vw([-1, 5]) == 0 and L.psulvsb_voxel_down_sample_batch_workspace_bytes(None, 3) == 0


# ---- refusals -------------------------------------------------------------------------------------------------------

def four(sel=(0, 1, 2, 3), v=0.1, n=4, arr=None, B=1, pts=True, work=True, out=True, count=True):
    """Return codes of psulvsb_voxel_down_sample, _host, _batch and _batch_host (the indices in `sel` only: a call that
    is not refused would run on host pointers)."""
    L = capi.lib()
    p = BUF.ctypes.data if pts else None
    w = BUF.ctypes.data if work else None
    o = BUF.ctypes.data if out else None
    k = BUF.ctypes.data if count else None
    arr = clouds([{}]) if arr is None else arr
    calls = (lambda: L.psulvsb_voxel_down_sample(None, p, n, v, w, o, k),
             lambda: L.psulvsb_voxel_down_sample_host(p, n, v, o, k),
             lambda: L.psulvsb_voxel_down_sample_batch(None, arr, B, v, w, o, k),
             lambda: L.psulvsb_voxel_down_sample_batch_host(arr, B, v, o, k))
    return tuple(calls[j]() for j in sel)


def test_refusals_come_before_any_device_work():
    L = capi.lib()
    inv = (capi.ERR_INVALID,) * 4
    for v in (0.0, -0.0, -1.0, float("nan"), float("inf"), -float("inf")):
        assert four(v=v) == inv, v
        assert four((2, 3), B=0, v=v) == inv[:2], v
    assert four(out=False) == inv
    assert four(count=False) == inv
    assert four((0, 1), pts=False) == inv[:2]
    assert four((0, 2), work=False) == inv[:2]
    assert four((0, 1), n=-1) == inv[:2]
    assert four((2, 3), B=-1) == inv[:2]
    for spec in ({"n": -1}, {"pts": None}):                     # the bad cloud is the last of three
        assert four((2, 3), arr=clouds([{}, {}, spec]), B=3) == inv[:2], spec
    assert L.psulvsb_voxel_down_sample_batch(None, None, 1, 0.1, BUF.ctypes.data, BUF.ctypes.data,
                                             BUF.ctypes.data) == capi.ERR_INVALID
    assert L.psulvsb_voxel_down_sample_batch_host(None, 1, 0.1, BUF.ctypes.data, BUF.ctypes.data) == capi.ERR_INVALID
    big = 2 ** 30
    assert four((2, 3), arr=clouds([{"n": big}, {"n": big}]), B=2) == (capi.ERR_UNSUPPORTED,) * 2
    # B = 0 does nothing and needs no pointer; the voxel size is still checked
    assert four((2, 3), B=0) == (capi.OK, capi.OK)
    assert (L.psulvsb_voxel_down_sample_batch(None, None, 0, 0.1, None, None, None),
            L.psulvsb_voxel_down_sample_batch_host(None, 0, 0.1, None, None)) == (capi.OK, capi.OK)
    # an empty device call needs no points, workspace or output, only the count (written on the device)
    if L.psulvsb_device_count() == 0:
        ok = (capi.ERR_NO_DEVICE,) * 4
        assert four() == ok
        assert four((0,), n=0, pts=False, work=False, out=False) == ok[:1]
        assert four((2,), arr=clouds([{"n": 0, "pts": None}])) == ok[:1]
        with pytest.raises(capi.PsulvsbError):
            features.voxel_down_sample(np.zeros((3, 4)), 0.1)
        with pytest.raises(capi.PsulvsbError):
            features.voxel_down_sample_batch([np.zeros((3, 4))], 0.1)
    # an empty host call writes its zero count on the host and needs no device
    m = np.full(2, 7, dtype=np.int32)
    assert L.psulvsb_voxel_down_sample_host(None, 0, 0.1, None, m.ctypes.data) == capi.OK and m[0] == 0
    m[:] = 7
    assert L.psulvsb_voxel_down_sample_batch_host(clouds([{"n": 0, "pts": None}] * 2), 2, 0.1, BUF.ctypes.data,
                                                  m.ctypes.data) == capi.OK and list(m) == [0, 0]
    assert features.voxel_down_sample(np.zeros((3, 0)), 0.1).shape == (3, 0)
    assert [a.shape for a in features.voxel_down_sample_batch([np.zeros((3, 0))] * 2, 0.1)] == [(3, 0)] * 2
    assert features.voxel_down_sample_batch([], 0.1) == []
    with pytest.raises(capi.PsulvsbError) as e:
        features.voxel_down_sample(np.zeros((3, 4)), 0.0)
    assert e.value.code == capi.ERR_INVALID


# ---- registers ------------------------------------------------------------------------------------------------------

def test_voxel_kernels_registers(tmp_path):
    """sm_100a, -Xptxas -v: every kernel of k8_voxel.cu (batch and batch-of-one instantiations) has no stack frame and
    no spills; the file holds the six voxel kernels and the grid's scan and scatter, nothing else."""
    nvcc = "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    r = subprocess.run([nvcc, "-O3", "-std=c++17", "-fmad=false", "-gencode", "arch=compute_100a,code=sm_100a",
                        "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", os.path.join(CSRC, "k8_voxel.cu"), "-o",
                        str(tmp_path / "k8v.o")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = r.stderr.splitlines()
    seen = {}
    for i, line in enumerate(lines):
        m = re.search(r"Function properties for \S*?\d(k8_[a-z0-9_]+?)(?:ILb[01]E|E)", line)
        if not m:
            continue
        f = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", lines[i + 1])
        assert f and f.groups() == ("0", "0", "0"), lines[i:i + 3]
        seen[m.group(1)] = seen.get(m.group(1), 0) + 1
    assert seen == {"k8_voxel_bounds": 2, "k8_voxel_count": 2, "k8_cloud_scan": 2, "k8_grid_scatter": 1,
                    "k8_voxel_order": 2, "k8_voxel_first": 2, "k8_voxel_scan": 2, "k8_voxel_mean": 2}, seen
