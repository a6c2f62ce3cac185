"""CPU-side checks of generalized ICP: argument refusals before any device work, psulvsb_gicp_pair_t against its ctypes
mirror, the batch workspace, the correspondence kernels' registers, and self-checks of the numpy restatement
(tests/gicp_restatement.py)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from oracle import icp as OI
from psulvsb_b200 import capi
from tests import gicp_restatement as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "probabilistic-self-update-line-vector-set-based-point-cloud-registration_b200", "csrc")
PTS = np.zeros((3, 4))
BAD_EPS = (0.0, -1.0, 1.5, float("nan"), float("inf"))


def params(**kw):
    p = capi.IcpParams()
    capi.lib().psulvsb_icp_default_params(C.byref(p))
    p.max_correspondence_distance = 0.1
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def gpairs(specs):
    """psulvsb_gicp_pair_t[len(specs)] from dicts overriding a valid 4-point pair (never dereferenced by a refused
    call)."""
    arr = (capi.GicpPair * max(len(specs), 1))()
    for b, spec in enumerate(specs):
        q = arr[b]
        q.src = q.tgt = q.src_normals = q.tgt_normals = PTS.ctypes.data
        q.n_s = q.n_t = 4
        q.R0[:] = [1, 0, 0, 0, 1, 0, 0, 0, 1]
        q.t0[:] = [0, 0, 0]
        for k, v in spec.items():
            if k in ("R0", "t0"):
                getattr(q, k)[:] = v
            else:
                setattr(q, k, v)
    return arr


def batch_codes(arr, B, p, eps=1e-3):
    L = capi.lib()
    res = (capi.IcpResult * max(B, 1))()
    pp = C.byref(p) if p is not None else None
    return (L.psulvsb_gicp_batch(None, arr, B, pp, eps, PTS.ctypes.data, PTS.ctypes.data, None, None),
            L.psulvsb_gicp_batch_host(arr, B, pp, eps, res, None, None))


def single_codes(p, eps=1e-3, n_s=4, n_t=4, src=True, tgt=True, sn=True, tn=True, R0=None, t0=None):
    L = capi.lib()
    R = (C.c_double * 9)(*(R0 if R0 is not None else [1, 0, 0, 0, 1, 0, 0, 0, 1]))
    t = (C.c_double * 3)(*(t0 if t0 is not None else [0, 0, 0]))
    ptr = PTS.ctypes.data
    a = [ptr if src else None, n_s, ptr if sn else None, ptr if tgt else None, n_t, ptr if tn else None,
         C.byref(p) if p is not None else None, eps, R, t]
    dev = L.psulvsb_gicp(None, *a, ptr, ptr, None, None)
    host = L.psulvsb_gicp_host(*a, (capi.IcpResult * 1)(), None, None)
    return dev, host


INV = (capi.ERR_INVALID, capi.ERR_INVALID)


def test_single_calls_refuse_bad_arguments_before_any_device_work():
    good = params()
    for e in BAD_EPS:
        assert single_codes(good, eps=e) == INV, e
    assert single_codes(params(point_to_plane=1)) == INV          # the entry point is the mode
    for b in (params(max_correspondence_distance=0.0), params(max_iterations=-1), params(relative_rmse=float("nan")),
              None):
        assert single_codes(b) == INV
    nan = float("nan")
    for kw in ({"n_s": -1}, {"n_t": -1}, {"src": False}, {"tgt": False}, {"sn": False}, {"tn": False},
               {"R0": [1, 0, 0, 0, nan, 0, 0, 0, 1]}, {"t0": [0, float("inf"), 0]}):
        assert single_codes(good, **kw) == INV, kw
    L = capi.lib()
    if L.psulvsb_device_count() == 0:
        # an empty cloud needs no normals; the call then only lacks a device
        assert single_codes(good, n_s=0, src=False, sn=False, tn=False) == (capi.ERR_NO_DEVICE,) * 2
        assert single_codes(good) == (capi.ERR_NO_DEVICE,) * 2
        from psulvsb_b200 import icp

        with pytest.raises(capi.PsulvsbError):
            icp.gicp(PTS, PTS, PTS, PTS, np.eye(3), np.zeros(3), 0.1)


def test_batch_refuses_bad_arguments_before_any_device_work():
    good = params()
    for e in BAD_EPS:
        assert batch_codes(gpairs([{}, {}]), 2, good, e) == INV, e
    assert batch_codes(gpairs([{}]), 1, params(point_to_plane=1)) == INV
    assert batch_codes(gpairs([{}]), 1, None) == INV
    assert batch_codes(gpairs([{}]), -1, good) == INV
    nan = float("nan")
    for spec in ({"n_s": -1}, {"n_t": -1}, {"src": None}, {"tgt": None}, {"src_normals": None}, {"tgt_normals": None},
                 {"R0": [1, 0, 0, 0, nan, 0, 0, 0, 1]}, {"t0": [0, float("inf"), 0]}):
        assert batch_codes(gpairs([{}, {}, spec]), 3, good) == INV, spec
    L = capi.lib()
    # required outputs: pairs, workspace, results
    ok = gpairs([{}])
    assert L.psulvsb_gicp_batch(None, None, 1, C.byref(good), 1e-3, PTS.ctypes.data, PTS.ctypes.data, None, None) == \
        capi.ERR_INVALID
    assert L.psulvsb_gicp_batch(None, ok, 1, C.byref(good), 1e-3, None, PTS.ctypes.data, None, None) == capi.ERR_INVALID
    assert L.psulvsb_gicp_batch(None, ok, 1, C.byref(good), 1e-3, PTS.ctypes.data, None, None, None) == capi.ERR_INVALID
    assert L.psulvsb_gicp_batch_host(ok, 1, C.byref(good), 1e-3, None, None, None) == capi.ERR_INVALID
    big = 2 ** 30
    for spec in ({"n_s": big}, {"n_t": big}):
        assert batch_codes(gpairs([spec, spec]), 2, good) == (capi.ERR_UNSUPPORTED,) * 2
    assert batch_codes(None, 0, good) == (capi.OK, capi.OK)
    # a pair with an empty side needs no normals
    empty = gpairs([{"n_s": 0, "src": None, "src_normals": None, "tgt_normals": None},
                    {"n_t": 0, "tgt": None, "src_normals": None, "tgt_normals": None}])
    if L.psulvsb_device_count() == 0:
        assert batch_codes(empty, 2, good) == (capi.ERR_NO_DEVICE,) * 2
        assert batch_codes(gpairs([{}, {}]), 2, good, 1.0) == (capi.ERR_NO_DEVICE,) * 2
    from psulvsb_b200 import icp

    assert icp.gicp_batch([], [], [], [], np.zeros((0, 3, 3)), np.zeros((0, 3)), 0.1) == []
    with pytest.raises(ValueError):
        icp.gicp(PTS, PTS, PTS[:, :3], PTS, np.eye(3), np.zeros(3), 0.1)


def test_pair_struct_matches_the_header(tmp_path):
    src = tmp_path / "pair.c"
    fields = ("src", "n_s", "tgt", "n_t", "src_normals", "tgt_normals", "R0", "t0")
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "psulvsb.h"\n'
                   "int main(void) {\n"
                   '  printf("%zu' + " %zu" * len(fields) + '\\n", sizeof(psulvsb_gicp_pair_t)' +
                   "".join(f", offsetof(psulvsb_gicp_pair_t, {f})" for f in fields) + ");\n"
                   "  return 0;\n}\n")
    exe = str(tmp_path / "pair")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe])
    got = list(map(int, subprocess.check_output([exe], text=True).split()))
    P = capi.GicpPair
    assert got == [C.sizeof(P)] + [getattr(P, f).offset for f in fields]


def test_batch_workspace_is_the_icp_batch_workspace():
    L = capi.lib()
    for sizes in ([(5000, 5000)], [(5000, 5000), (300, 7), (1, 1), (0, 9), (9, 0)], [(50000, 17)] * 7):
        g = gpairs([{"n_s": ns, "n_t": nt} for ns, nt in sizes])
        i = (capi.IcpPair * len(sizes))()
        for b, (ns, nt) in enumerate(sizes):
            i[b].n_s, i[b].n_t = ns, nt
        assert L.psulvsb_gicp_batch_workspace_bytes(g, len(sizes)) == \
            L.psulvsb_icp_batch_workspace_bytes(i, len(sizes)) > 0
    assert L.psulvsb_gicp_batch_workspace_bytes(gpairs([{"n_s": 5000, "n_t": 3000}]), 1) == \
        L.psulvsb_icp_workspace_bytes(5000, 3000)
    assert L.psulvsb_gicp_batch_workspace_bytes(None, 2) == 0
    assert L.psulvsb_gicp_batch_workspace_bytes(gpairs([{}]), 0) == 0
    assert L.psulvsb_gicp_batch_workspace_bytes(gpairs([{"n_t": -1}]), 1) == 0


def test_correspondence_kernels_do_not_spill_and_keep_their_registers(tmp_path):
    """The three correspondence passes (k9_icp_correspond for point-to-point and point-to-plane, k9_gicp_correspond)
    run without local memory (sm_100a, -Xptxas -v); the first two at the 58 / 79 registers they had before GICP shared
    their body."""
    nvcc = "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    r = subprocess.run([nvcc, "-O3", "-std=c++17", "-fmad=false", "-gencode", "arch=compute_100a,code=sm_100a",
                        "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", os.path.join(CSRC, "k9_icp.cu"), "-o",
                        str(tmp_path / "k9_icp.o")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    lines = r.stderr.splitlines()
    regs = {}
    for i, line in enumerate(lines):
        m = re.search(r"Function properties for \S*(k9_icp_correspondILi(\d)E|k9_gicp_correspond)", line)
        if not m:
            continue
        key = 2 if m.group(2) is None else int(m.group(2))
        f = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", lines[i + 1])
        assert f and f.groups() == ("0", "0", "0"), lines[i:i + 3]
        regs[key] = int(re.search(r"Used (\d+) registers", lines[i + 2]).group(1))
    assert sorted(regs) == [0, 1, 2], regs
    assert regs[0] == 58 and regs[1] == 79, regs


def random_problem(K, seed):
    rng = np.random.default_rng(seed)
    Pp = rng.normal(size=(3, K))
    Q = Pp + 0.05 * rng.normal(size=(3, K))
    Ns, Nt = rng.normal(size=(3, K)), rng.normal(size=(3, K))
    R, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    return Pp, Q, Ns, Nt, R * np.sign(np.linalg.det(R)), np.arange(K)


def full(h):
    H = np.zeros((6, 6))
    v = 0
    for a in range(6):
        for e in range(a, 6):
            H[a, e] = H[e, a] = h[v]
            v += 1
    return H


def test_restatement_at_epsilon_one_is_linearised_point_to_point():
    Pp, Q, Ns, Nt, R, corr = random_problem(200, 1)
    H, g = G.system(Pp, Q, Ns, Nt, R, corr, 1.0)
    x = G.solve6(H, g)
    # min sum |A_i x + d_i|^2, A_i = [-[p_i]x, I]
    A = np.zeros((3 * Pp.shape[1], 6))
    for i in range(Pp.shape[1]):
        px, py, pz = Pp[:, i]
        A[3 * i:3 * i + 3, :3] = -np.array([[0, -pz, py], [pz, 0, -px], [-py, px, 0]])
        A[3 * i:3 * i + 3, 3:] = np.eye(3)
    want = np.linalg.lstsq(A, -(Pp - Q).T.reshape(-1), rcond=None)[0]
    assert np.abs(x - want).max() <= 1e-12 * max(1.0, np.abs(want).max())
    # C = 2 I exactly, M = I / 2
    h, _ = G.terms(Pp, Q, G.rotate(R, G.unit_normals(Ns)), G.unit_normals(Nt), 0.0)
    assert np.array_equal(h[15:], np.tile(np.array([[0.5], [0], [0], [0.5], [0], [0.5]]), (1, Pp.shape[1])))


def test_restatement_ignores_the_signs_of_the_normals():
    Pp, Q, Ns, Nt, R, corr = random_problem(300, 2)
    rng = np.random.default_rng(3)
    fs, ft = np.where(rng.random(300) < 0.5, -1.0, 1.0), np.where(rng.random(300) < 0.5, -1.0, 1.0)
    for eps in (1e-3, 0.25, 1e-6):
        a = G.system(Pp, Q, Ns, Nt, R, corr, eps)
        b = G.system(Pp, Q, Ns * fs, Nt * ft, R, corr, eps)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
        # and with one transform per call, the update too
        assert np.array_equal(G.update(Pp, Q, Ns, Nt, R, corr, eps)[0], G.update(Pp, Q, Ns * fs, Nt * ft, R, corr,
                                                                                 eps)[0])


def test_restatement_gives_identity_covariance_to_non_finite_and_zero_normals():
    Pp, Q, Ns, Nt, R, corr = random_problem(6, 4)
    Ns[:, 0] = np.nan
    Nt[:, 1] = [np.inf, 0, 0]
    Ns[:, 2] = 0.0
    Nt[:, 3] = 0.0
    Ns[:, 3] = np.nan
    w = 1.0 - 1e-3
    m = G.rotate(R, G.unit_normals(Ns))
    n = G.unit_normals(Nt)
    C = G.covariance(m, n, w)
    for i, (keep_m, keep_n) in enumerate(((False, True), (True, False), (False, True), (False, False))):
        # the sides left: I + (I - w u u^T) summed, I for a side without a usable normal
        want = 2.0 * np.eye(3)
        for keep, u in ((keep_m, m[:, i]), (keep_n, n[:, i])):
            if keep:
                want = want - w * np.outer(u, u)
        got = np.array([[C[0][i], C[1][i], C[2][i]], [C[1][i], C[3][i], C[4][i]], [C[2][i], C[4][i], C[5][i]]])
        assert np.abs(got - want).max() <= 1e-15, i
        if not keep_m and not keep_n:
            assert np.array_equal(got, 2.0 * np.eye(3))
    h, g = G.terms(Pp, Q, m, n, w)
    assert np.isfinite(h).all() and np.isfinite(g).all()
    # the unit normals that are kept are unit to the last bits
    ok = np.isfinite(Ns).all(axis=0) & (np.abs(Ns).sum(axis=0) > 0)
    assert np.abs(np.linalg.norm(G.unit_normals(Ns)[:, ok], axis=0) - 1).max() <= 4e-16


def test_restatement_needs_three_correspondences():
    Pp, Q, Ns, Nt, R, corr = random_problem(8, 5)
    c = np.full(8, -1)
    c[:2] = [0, 1]
    assert G.update(Pp, Q, Ns, Nt, R, c, 1e-3) is None
    c[2] = 2
    assert G.update(Pp, Q, Ns, Nt, R, c, 1e-3) is not None
    # the system matches A^T M A and A^T M d built with dense matrices
    H, g = G.system(Pp, Q, Ns, Nt, R, corr, 1e-3)
    Hw, gw = np.zeros((6, 6)), np.zeros(6)
    for i in range(8):
        p = Pp[:, i]
        A = np.hstack([-np.array([[0, -p[2], p[1]], [p[2], 0, -p[0]], [-p[1], p[0], 0]]), np.eye(3)])
        ns, nt = R @ (Ns[:, i] / np.linalg.norm(Ns[:, i])), Nt[:, i] / np.linalg.norm(Nt[:, i])
        Cm = (np.eye(3) - 0.999 * np.outer(ns, ns)) + (np.eye(3) - 0.999 * np.outer(nt, nt))
        M = np.linalg.inv(Cm)
        Hw += A.T @ M @ A
        gw += A.T @ M @ (p - Q[:, i])
    assert np.abs(full(H) - Hw).max() <= 1e-9 * np.abs(Hw).max()
    assert np.abs(g - gw).max() <= 1e-9 * np.abs(Hw).max()
    assert OI.NO_UPDATE == 2
