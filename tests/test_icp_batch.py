"""CPU-side checks of the batched ICP entry points: argument refusals before any device work, B = 0, the error without
a device, psulvsb_icp_pair_t against its ctypes mirror, the workspace size, and the batched kernels' registers."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from psulvsb_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "probabilistic-self-update-line-vector-set-based-point-cloud-registration_b200", "csrc")
PTS = np.zeros((3, 4))


def params(**kw):
    p = capi.IcpParams()
    capi.lib().psulvsb_icp_default_params(C.byref(p))
    p.max_correspondence_distance = 0.1
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def pairs(specs):
    """psulvsb_icp_pair_t[len(specs)] from dicts overriding a valid 4-point pair (pointers are never dereferenced by a
    refused call)."""
    arr = (capi.IcpPair * max(len(specs), 1))()
    for b, spec in enumerate(specs):
        q = arr[b]
        q.src = q.tgt = q.tgt_normals = PTS.ctypes.data
        q.n_s = q.n_t = 4
        q.R0[:] = [1, 0, 0, 0, 1, 0, 0, 0, 1]
        q.t0[:] = [0, 0, 0]
        for k, v in spec.items():
            if k in ("R0", "t0"):
                getattr(q, k)[:] = v
            else:
                setattr(q, k, v)
    return arr


def both(arr, B, p):
    """Return codes of the device and the host entry (non-NULL outputs and workspace)."""
    L = capi.lib()
    res = (capi.IcpResult * max(B, 1))()
    dev = L.psulvsb_icp_batch(None, arr, B, C.byref(p) if p is not None else None, PTS.ctypes.data, PTS.ctypes.data,
                              None, None)
    host = L.psulvsb_icp_batch_host(arr, B, C.byref(p) if p is not None else None, res, None, None)
    return dev, host


def test_batch_refuses_bad_arguments_before_any_device_work():
    good = params()
    bad_params = [params(max_correspondence_distance=v) for v in (0.0, -1.0, float("nan"), float("inf"))]
    bad_params += [params(max_iterations=-1), params(relative_fitness=-1e-6), params(relative_rmse=float("nan")),
                   params(point_to_plane=2), None]
    for b in bad_params:
        assert both(pairs([{}, {}]), 2, b) == (capi.ERR_INVALID, capi.ERR_INVALID)
    assert both(pairs([{}]), -1, good) == (capi.ERR_INVALID, capi.ERR_INVALID)
    nan, inf = float("nan"), float("inf")
    bad_pairs = [{"n_s": -1}, {"n_t": -1}, {"src": None}, {"tgt": None},
                 {"R0": [1, 0, 0, 0, nan, 0, 0, 0, 1]}, {"t0": [0, inf, 0]}]
    for spec in bad_pairs:                                    # the bad pair is the last of three
        assert both(pairs([{}, {}, spec]), 3, good) == (capi.ERR_INVALID, capi.ERR_INVALID), spec
    p2l = params(point_to_plane=1)
    assert both(pairs([{}, {"tgt_normals": None}]), 2, p2l) == (capi.ERR_INVALID, capi.ERR_INVALID)
    # an empty cloud needs no pointer; point-to-plane needs no normals where n_t = 0
    L = capi.lib()
    ok = pairs([{"n_s": 0, "src": None}, {"n_t": 0, "tgt": None, "tgt_normals": None}])
    # required outputs: pairs, workspace, results
    assert L.psulvsb_icp_batch(None, None, 1, C.byref(good), PTS.ctypes.data, PTS.ctypes.data, None, None) == \
        capi.ERR_INVALID
    assert L.psulvsb_icp_batch(None, ok, 2, C.byref(good), None, PTS.ctypes.data, None, None) == capi.ERR_INVALID
    assert L.psulvsb_icp_batch(None, ok, 2, C.byref(good), PTS.ctypes.data, None, None, None) == capi.ERR_INVALID
    assert L.psulvsb_icp_batch_host(ok, 2, C.byref(good), None, None, None) == capi.ERR_INVALID
    assert L.psulvsb_icp_batch_host(None, 1, C.byref(good), (capi.IcpResult * 1)(), None, None) == capi.ERR_INVALID
    # the pairs' clouds must add up to fewer than 2^31 points (refused before anything is read)
    big = 2 ** 30
    for spec in ({"n_s": big}, {"n_t": big}):
        assert both(pairs([spec, spec]), 2, good) == (capi.ERR_UNSUPPORTED, capi.ERR_UNSUPPORTED)
    # B = 0 does nothing and needs no device
    assert both(None, 0, good) == (capi.OK, capi.OK)
    if L.psulvsb_device_count() == 0:
        assert both(ok, 2, good) == (capi.ERR_NO_DEVICE, capi.ERR_NO_DEVICE)
        assert both(pairs([{}, {}]), 2, p2l) == (capi.ERR_NO_DEVICE, capi.ERR_NO_DEVICE)
        assert b"no CUDA device" in L.psulvsb_last_error()
        from psulvsb_b200 import icp

        with pytest.raises(capi.PsulvsbError):
            icp.icp_batch([PTS, PTS], [PTS, PTS], np.tile(np.eye(3), (2, 1, 1)), np.zeros((2, 3)), 0.1)
    assert icp_batch_empty() == []


def icp_batch_empty():
    from psulvsb_b200 import icp

    return icp.icp_batch([], [], np.zeros((0, 3, 3)), np.zeros((0, 3)), 0.1)


def test_pair_struct_matches_the_header(tmp_path):
    src = tmp_path / "pair.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "psulvsb.h"\n'
                   "int main(void) {\n"
                   '  printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(psulvsb_icp_pair_t), '
                   "offsetof(psulvsb_icp_pair_t, src), offsetof(psulvsb_icp_pair_t, n_s), "
                   "offsetof(psulvsb_icp_pair_t, tgt), offsetof(psulvsb_icp_pair_t, n_t), "
                   "offsetof(psulvsb_icp_pair_t, tgt_normals), offsetof(psulvsb_icp_pair_t, R0), "
                   "offsetof(psulvsb_icp_pair_t, t0));\n"
                   "  return 0;\n}\n")
    exe = str(tmp_path / "pair")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe])
    got = list(map(int, subprocess.check_output([exe], text=True).split()))
    P = capi.IcpPair
    assert got == [C.sizeof(P), P.src.offset, P.n_s.offset, P.tgt.offset, P.n_t.offset, P.tgt_normals.offset,
                   P.R0.offset, P.t0.offset]


def test_batch_workspace_depends_on_sizes_and_grows():
    L = capi.lib()

    def ws(sizes):
        arr = pairs([{"n_s": ns, "n_t": nt} for ns, nt in sizes])
        return L.psulvsb_icp_batch_workspace_bytes(arr, len(sizes))

    base = [(5000, 5000), (300, 7), (1, 1)]
    assert ws(base) == ws(base) > 0
    # pointers and transforms do not matter, sizes do
    a = pairs([{"n_s": ns, "n_t": nt} for ns, nt in base])
    b = pairs([{"n_s": ns, "n_t": nt, "src": None, "tgt": None, "t0": [5, 6, 7]} for ns, nt in base])
    assert L.psulvsb_icp_batch_workspace_bytes(a, 3) == L.psulvsb_icp_batch_workspace_bytes(b, 3)
    assert ws([(5000, 50000)] + base[1:]) > ws(base)          # grows with the targets
    assert ws([(50000, 5000)] + base[1:]) > ws(base)          # ... and with the sources
    assert ws(base + [(5000, 5000)]) > ws(base)
    # a batch of one is psulvsb_icp's workspace
    assert ws([(5000, 5000)]) == L.psulvsb_icp_workspace_bytes(5000, 5000)
    assert ws([]) == 0 and ws([(-1, 5)]) == 0 and L.psulvsb_icp_batch_workspace_bytes(None, 3) == 0


def test_batched_kernels_do_not_spill(tmp_path):
    """Every per-point kernel of the batch (both correspondence instantiations, cross, the grid) keeps its state in
    registers (sm_100a, -Xptxas -v).  The step kernels are left out: their one-thread update (6x6 Cholesky, 3x3 SVD in
    svd3.cuh, which the solver shares) indexes small arrays at run time and keeps them in a stack frame."""
    nvcc = "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    r = subprocess.run([nvcc, "-O3", "-std=c++17", "-fmad=false", "-gencode", "arch=compute_100a,code=sm_100a",
                        "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", os.path.join(CSRC, "k9_icp.cu"), "-o",
                        str(tmp_path / "k9_icp.o")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = r.stderr.splitlines()
    seen = {}
    for i, line in enumerate(lines):
        m = re.search(r"Function properties for (\S+)", line)
        if not m:
            continue
        for k in ("k9_icp_correspond", "k9_icp_cross", "k9_icp_bounds", "k9_icp_grid_count", "k9_icp_grid_scan",
                  "k9_icp_grid_order", "k8_grid_scatter"):
            if k in m.group(1):
                f = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", lines[i + 1])
                assert f and f.groups() == ("0", "0", "0"), lines[i:i + 3]
                seen[k] = seen.get(k, 0) + 1
    assert seen == {"k9_icp_correspond": 2, "k9_icp_cross": 1, "k9_icp_bounds": 1, "k9_icp_grid_count": 1,
                    "k9_icp_grid_scan": 1, "k9_icp_grid_order": 1, "k8_grid_scatter": 1}, seen
