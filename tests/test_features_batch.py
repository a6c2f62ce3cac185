"""CPU-side checks of the batched correspondence entry points: argument refusals before any device work, B = 0, the
error without a device, both structs against the header, the workspace sizes, the output-offset formula and the
batched kernels' registers."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from psulvsb_b200 import capi, features

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


def mpairs(specs):
    arr = (capi.MatchPair * max(len(specs), 1))()
    for b, spec in enumerate(specs):
        q = arr[b]
        q.src = q.tgt = q.fs = q.ft = BUF.ctypes.data
        q.n_src = q.n_tgt = 4
        for k, v in spec.items():
            setattr(q, k, v)
    return arr


def fpfh_both(arr, B, rn=0.1, rf=0.2):
    L = capi.lib()
    return (L.psulvsb_fpfh_batch(None, arr, B, rn, rf, BUF.ctypes.data, None, BUF.ctypes.data),
            L.psulvsb_fpfh_batch_host(arr, B, rn, rf, None, BUF.ctypes.data))


def match_both(arr, B, cross=1, tup=0, scale=0.95):
    L = capi.lib()
    counts = np.zeros(max(B, 1), dtype=np.int64)
    return (L.psulvsb_match_batch(None, arr, B, cross, tup, scale, BUF.ctypes.data, BUF.ctypes.data,
                                  counts.ctypes.data),
            L.psulvsb_match_batch_host(arr, B, cross, tup, scale, BUF.ctypes.data, counts.ctypes.data))


def test_fpfh_batch_refuses_bad_arguments_before_any_device_work():
    L = capi.lib()
    inv = (capi.ERR_INVALID, capi.ERR_INVALID)
    for rn, rf in ((0.0, 0.2), (0.1, -1.0), (float("nan"), 0.2), (0.1, float("inf"))):
        assert fpfh_both(clouds([{}, {}]), 2, rn, rf) == inv
    assert fpfh_both(clouds([{}]), -1) == inv
    for spec in ({"n": -1}, {"pts": None}):                   # the bad cloud is the last of three
        assert fpfh_both(clouds([{}, {}, spec]), 3) == inv, spec
    ok = clouds([{"n": 0, "pts": None}, {}])                  # an empty cloud needs no pointer
    assert L.psulvsb_fpfh_batch(None, None, 1, 0.1, 0.2, BUF.ctypes.data, None, BUF.ctypes.data) == capi.ERR_INVALID
    assert L.psulvsb_fpfh_batch(None, ok, 2, 0.1, 0.2, None, None, BUF.ctypes.data) == capi.ERR_INVALID
    assert L.psulvsb_fpfh_batch(None, ok, 2, 0.1, 0.2, BUF.ctypes.data, None, None) == capi.ERR_INVALID
    assert L.psulvsb_fpfh_batch_host(ok, 2, 0.1, 0.2, None, None) == capi.ERR_INVALID
    big = 2 ** 30
    assert fpfh_both(clouds([{"n": big}, {"n": big}]), 2) == (capi.ERR_UNSUPPORTED, capi.ERR_UNSUPPORTED)
    assert fpfh_both(None, 0) == (capi.OK, capi.OK)
    if L.psulvsb_device_count() == 0:
        assert fpfh_both(ok, 2) == (capi.ERR_NO_DEVICE, capi.ERR_NO_DEVICE)
        with pytest.raises(capi.PsulvsbError):
            features.fpfh_batch([np.zeros((3, 4))], 0.1, 0.2)
    assert features.fpfh_batch([], 0.1, 0.2) == []


def test_match_batch_refuses_bad_arguments_before_any_device_work():
    L = capi.lib()
    inv = (capi.ERR_INVALID, capi.ERR_INVALID)
    assert match_both(mpairs([{}]), -1) == inv
    for spec in ({"n_src": -1}, {"n_tgt": -1}, {"src": None}, {"tgt": None}, {"fs": None}, {"ft": None}):
        assert match_both(mpairs([{}, {}, spec]), 3) == inv, spec
    for scale in (float("nan"), float("inf")):
        assert match_both(mpairs([{}]), 1, tup=1, scale=scale) == inv
    ok = mpairs([{"n_src": 0, "src": None, "fs": None}, {"n_tgt": 0, "tgt": None, "ft": None}])
    d, c = BUF.ctypes.data, np.zeros(2, dtype=np.int64).ctypes.data
    for args in ((None, 1, d, d, c), (ok, 2, None, d, c), (ok, 2, d, None, c), (ok, 2, d, d, None)):
        arr, B, work, out, cnt = args
        assert L.psulvsb_match_batch(None, arr, B, 1, 0, 0.95, work, out, cnt) == capi.ERR_INVALID, args
    assert L.psulvsb_match_batch_host(ok, 2, 1, 0, 0.95, None, c) == capi.ERR_INVALID
    assert L.psulvsb_match_batch_host(ok, 2, 1, 0, 0.95, d, None) == capi.ERR_INVALID
    big = 2 ** 30
    for spec in ({"n_src": big}, {"n_tgt": big}):
        assert match_both(mpairs([spec, spec]), 2) == (capi.ERR_UNSUPPORTED, capi.ERR_UNSUPPORTED)
    assert match_both(None, 0) == (capi.OK, capi.OK)
    if L.psulvsb_device_count() == 0:
        assert match_both(ok, 2) == (capi.ERR_NO_DEVICE, capi.ERR_NO_DEVICE)
        assert b"no CUDA device" in L.psulvsb_last_error()
    assert features.match_batch([], [], [], []) == []


def test_structs_match_the_header(tmp_path):
    src = tmp_path / "structs.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "psulvsb.h"\n'
                   "int main(void) {\n"
                   '  printf("%zu %zu %zu %zu\\n", sizeof(psulvsb_fpfh_cloud_t), offsetof(psulvsb_fpfh_cloud_t, pts), '
                   "offsetof(psulvsb_fpfh_cloud_t, n), offsetof(psulvsb_fpfh_cloud_t, viewpoint));\n"
                   '  printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(psulvsb_match_pair_t), '
                   "offsetof(psulvsb_match_pair_t, src), offsetof(psulvsb_match_pair_t, n_src), "
                   "offsetof(psulvsb_match_pair_t, tgt), offsetof(psulvsb_match_pair_t, n_tgt), "
                   "offsetof(psulvsb_match_pair_t, fs), offsetof(psulvsb_match_pair_t, ft), "
                   "offsetof(psulvsb_match_pair_t, seed));\n"
                   "  return 0;\n}\n")
    exe = str(tmp_path / "structs")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe])
    got = [list(map(int, line.split())) for line in subprocess.check_output([exe], text=True).splitlines()]
    F, M = capi.FpfhCloud, capi.MatchPair
    assert got[0] == [C.sizeof(F), F.pts.offset, F.n.offset, F.viewpoint.offset]
    assert got[1] == [C.sizeof(M), M.src.offset, M.n_src.offset, M.tgt.offset, M.n_tgt.offset, M.fs.offset,
                      M.ft.offset, M.seed.offset]


def test_workspace_depends_on_sizes_and_grows():
    L = capi.lib()

    def fw(sizes):
        return L.psulvsb_fpfh_batch_workspace_bytes(clouds([{"n": n} for n in sizes]), len(sizes))

    base = [5000, 129, 1]
    assert fw(base) == fw(base) > 0
    assert fw([50000] + base[1:]) > fw(base) and fw(base + [7]) > fw(base)
    assert fw([5000]) == L.psulvsb_fpfh_workspace_bytes(5000)
    assert fw([]) == 0 and fw([-1, 5]) == 0 and L.psulvsb_fpfh_batch_workspace_bytes(None, 3) == 0

    def mw(sizes, cross=1, tup=0):
        arr = mpairs([{"n_src": a, "n_tgt": b} for a, b in sizes])
        return L.psulvsb_match_batch_workspace_bytes(arr, len(sizes), cross, tup)

    mb = [(5000, 5000), (300, 7), (0, 9)]
    assert mw(mb) == mw(mb) > 0
    a = mpairs([{"n_src": x, "n_tgt": y} for x, y in mb])
    b = mpairs([{"n_src": x, "n_tgt": y, "src": None, "seed": 9} for x, y in mb])
    assert L.psulvsb_match_batch_workspace_bytes(a, 3, 1, 0) == L.psulvsb_match_batch_workspace_bytes(b, 3, 1, 0)
    assert mw([(50000, 5000)] + mb[1:]) > mw(mb) and mw([(5000, 50000)] + mb[1:]) > mw(mb)
    assert mw(mb, tup=1) > mw(mb)                                  # the tuple test's list and pass flags
    assert mw([]) == 0 and mw([(-1, 5)]) == 0 and L.psulvsb_match_batch_workspace_bytes(None, 3, 1, 0) == 0


def test_output_offset_formula_matches_the_header():
    """The header states cap = 0 with an empty side, 3000 with the tuple test, n_src with crosscheck, n_src + n_tgt
    without; the Python helper sizes the outputs with it."""
    text = open(os.path.join(ROOT, "include", "psulvsb.h")).read()
    assert "cap = 0 when a side is empty, else 3000 with the tuple test, else n_src with crosscheck and n_src + n_tgt" \
        in re.sub(r"\s*\n\s*\*\s*", " ", text)
    ns, nt = [5, 0, 7, 3000], [9, 4, 0, 1]
    assert features.match_caps(ns, nt, True, False) == [5, 0, 0, 3000]
    assert features.match_caps(ns, nt, False, False) == [14, 0, 0, 3001]
    assert features.match_caps(ns, nt, True, True) == [3000, 0, 0, 3000]
    assert features.match_caps(ns, nt, False, True) == [3000, 0, 0, 3000]


def test_batched_kernels_registers(tmp_path):
    """sm_100a, -Xptxas -v: no spills in any kernel of k8_features.cu (batch and batch-of-one instantiations); no stack
    frame in the NN, grid, list and tuple kernels; the neighbour walks keep the stack frames of their 27-bucket de-duplication (normals 184 bytes, SPFH and
    FPFH 112)."""
    nvcc = "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    r = subprocess.run([nvcc, "-O3", "-std=c++17", "-fmad=false", "-gencode", "arch=compute_100a,code=sm_100a",
                        "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", os.path.join(CSRC, "k8_features.cu"), "-o",
                        str(tmp_path / "k8.o")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = r.stderr.splitlines()
    frames = {}
    for i, line in enumerate(lines):
        m = re.search(r"Function properties for \S*?\d(k8_[a-z0-9_]+?)(?:ILb[01]E|E)", line)
        if not m:
            continue
        f = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", lines[i + 1])
        assert f and f.group(2) == "0" and f.group(3) == "0", lines[i:i + 3]
        frames[m.group(1)] = max(frames.get(m.group(1), 0), int(f.group(1)))   # both instantiations (batch, one)
    limits = {"k8_radius_normals": 184, "k8_spfh": 112, "k8_fpfh": 112}
    for k in ("k8_feature_nn", "k8_nn_finish", "k8_grid_count", "k8_cloud_scan", "k8_grid_scatter", "k8_grid_order",
              "k8_match_mark", "k8_match_flags", "k8_match_scan", "k8_match_place", "k8_tuple_trials", "k8_tuple_keep"):
        limits[k] = 0
    assert set(frames) == set(limits), frames
    for k, v in limits.items():
        assert frames[k] <= v, (k, frames[k])
