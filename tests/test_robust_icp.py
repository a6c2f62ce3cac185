"""CPU-side checks of the robust kernels of point-to-plane ICP and generalized ICP: argument refusals of the eight
entry points before any device work, psulvsb_robust_kernel_t against its ctypes mirror, the new correspondence passes'
registers, and self-checks of the numpy restatement (tests/robust_icp_restatement.py): the weights at their edges, the
closed-form W = C^-1/2, the L2 update against generalized ICP's and a scene where the robust kernels matter."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest
from scipy.linalg import sqrtm

import psulvsb_b200  # noqa: F401
from oracle import icp as OI
from psulvsb_b200 import capi
from psulvsb_b200 import icp as I
from tests import gicp_restatement as G
from tests import robust_icp_restatement as RR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "probabilistic-self-update-line-vector-set-based-point-cloud-registration_b200", "csrc")
PTS = np.zeros((3, 4))
INV = (capi.ERR_INVALID,) * 4
NOD = (capi.ERR_NO_DEVICE,) * 4
nan, inf = float("nan"), float("inf")
BAD_LOSSES = [None, (-1, 1.0), (5, 1.0)] + [(t, k) for t in (1, 2, 3, 4) for k in (0.0, -1.0, nan, inf, -inf)]


def params(**kw):
    p = capi.IcpParams()
    capi.lib().psulvsb_icp_default_params(C.byref(p))
    p.max_correspondence_distance = 0.1
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def kernel(loss):
    return None if loss is None else C.byref(capi.RobustKernel(*loss))


def ipairs(specs):
    arr = (capi.IcpPair * max(len(specs), 1))()
    for b, spec in enumerate(specs):
        q = arr[b]
        q.src = q.tgt = q.tgt_normals = PTS.ctypes.data
        q.n_s = q.n_t = 4
        q.R0[:] = [1, 0, 0, 0, 1, 0, 0, 0, 1]
        for k, v in spec.items():
            setattr(q, k, v)
    return arr


def gpairs(specs):
    arr = (capi.GicpPair * max(len(specs), 1))()
    for b, spec in enumerate(specs):
        q = arr[b]
        q.src = q.tgt = q.src_normals = q.tgt_normals = PTS.ctypes.data
        q.n_s = q.n_t = 4
        q.R0[:] = [1, 0, 0, 0, 1, 0, 0, 0, 1]
        for k, v in spec.items():
            setattr(q, k, v)
    return arr


def icp_codes(p, loss, n_s=4, tn=True, R0=None, pair=None):
    """psulvsb_icp_robust, _host, _batch and _batch_host on the same arguments."""
    L = capi.lib()
    ptr = PTS.ctypes.data
    R = (C.c_double * 9)(*(R0 or [1, 0, 0, 0, 1, 0, 0, 0, 1]))
    t = (C.c_double * 3)(0, 0, 0)
    pp = C.byref(p) if p is not None else None
    a = [ptr, n_s, ptr, 4, ptr if tn else None, pp, kernel(loss), R, t]
    res = (capi.IcpResult * 2)()
    arr = ipairs([pair or {}, {}])
    return (L.psulvsb_icp_robust(None, *a, ptr, ptr, None, None), L.psulvsb_icp_robust_host(*a, res, None, None),
            L.psulvsb_icp_robust_batch(None, arr, 2, pp, kernel(loss), ptr, ptr, None, None),
            L.psulvsb_icp_robust_batch_host(arr, 2, pp, kernel(loss), res, None, None))


def gicp_codes(p, loss, eps=1e-3, n_s=4, sn=True, pair=None):
    """psulvsb_gicp_robust, _host, _batch and _batch_host on the same arguments."""
    L = capi.lib()
    ptr = PTS.ctypes.data
    R = (C.c_double * 9)(1, 0, 0, 0, 1, 0, 0, 0, 1)
    t = (C.c_double * 3)(0, 0, 0)
    pp = C.byref(p) if p is not None else None
    a = [ptr, n_s, ptr if sn else None, ptr, 4, ptr, pp, eps, kernel(loss), R, t]
    res = (capi.IcpResult * 2)()
    arr = gpairs([pair or {}, {}])
    return (L.psulvsb_gicp_robust(None, *a, ptr, ptr, None, None), L.psulvsb_gicp_robust_host(*a, res, None, None),
            L.psulvsb_gicp_robust_batch(None, arr, 2, pp, eps, kernel(loss), ptr, ptr, None, None),
            L.psulvsb_gicp_robust_batch_host(arr, 2, pp, eps, kernel(loss), res, None, None))


def test_robust_icp_refuses_bad_arguments_before_any_device_work():
    p2l = params(point_to_plane=1)
    for loss in BAD_LOSSES:
        assert icp_codes(p2l, loss) == INV, loss
    # the entry points are point-to-plane
    assert icp_codes(params(point_to_plane=0), (4, 0.1)) == INV
    assert icp_codes(params(point_to_plane=2), (4, 0.1)) == INV
    # and refuse what psulvsb_icp[_batch] refuses
    for p in (None, params(point_to_plane=1, max_correspondence_distance=0.0),
              params(point_to_plane=1, max_iterations=-1), params(point_to_plane=1, relative_rmse=nan)):
        assert icp_codes(p, (1, 0.1)) == INV
    assert icp_codes(p2l, (1, 0.1), n_s=-1, pair={"n_s": -1}) == INV
    assert icp_codes(p2l, (1, 0.1), tn=False, pair={"tgt_normals": None}) == INV
    assert icp_codes(p2l, (1, 0.1), R0=[1, 0, 0, 0, nan, 0, 0, 0, 1], pair={"src": None}) == INV
    L = capi.lib()
    assert L.psulvsb_icp_robust_batch(None, ipairs([{}]), 0, C.byref(p2l), kernel((4, 0.1)), None, None, None,
                                      None) == capi.OK
    if L.psulvsb_device_count() == 0:
        for loss in ((0, nan), (0, -1.0), (1, 1e-300), (2, 5.0), (3, 1e300), (4, 0.1)):
            assert icp_codes(p2l, loss) == NOD, loss
        with pytest.raises(capi.PsulvsbError):
            I.icp(PTS, PTS, np.eye(3), np.zeros(3), 0.1, target_normals=PTS, point_to_plane=True,
                  loss=I.TukeyLoss(0.1))
    with pytest.raises(ValueError):
        I.icp(PTS, PTS, np.eye(3), np.zeros(3), 0.1, loss=I.HuberLoss(0.1))
    with pytest.raises(ValueError):
        I.icp_batch([PTS], [PTS], np.eye(3)[None], np.zeros((1, 3)), 0.1, loss=I.L2Loss())


def test_robust_gicp_refuses_bad_arguments_before_any_device_work():
    good = params()
    for loss in BAD_LOSSES:
        assert gicp_codes(good, loss) == INV, loss
    for eps in (0.0, 1.5, nan):
        assert gicp_codes(good, (1, 0.1), eps=eps) == INV
    assert gicp_codes(params(point_to_plane=1), (1, 0.1)) == INV
    assert gicp_codes(None, (1, 0.1)) == INV
    assert gicp_codes(good, (1, 0.1), sn=False, pair={"src_normals": None}) == INV
    assert gicp_codes(good, (1, 0.1), n_s=-1, pair={"n_s": -1}) == INV
    L = capi.lib()
    if L.psulvsb_device_count() == 0:
        for loss in ((0, nan), (1, 0.5), (2, 5.0), (3, 1e-4), (4, 0.1)):
            assert gicp_codes(good, loss) == NOD, loss
        assert gicp_codes(good, (4, 0.1), eps=1.0) == NOD
        with pytest.raises(capi.PsulvsbError):
            I.gicp(PTS, PTS, PTS, PTS, np.eye(3), np.zeros(3), 0.1, loss=I.CauchyLoss(0.1))


def test_robust_kernel_struct_matches_the_header(tmp_path):
    src = tmp_path / "rk.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "psulvsb.h"\n'
                   "int main(void) {\n"
                   '  printf("%zu %zu %zu %d %d %d %d %d\\n", sizeof(psulvsb_robust_kernel_t), '
                   "offsetof(psulvsb_robust_kernel_t, type), offsetof(psulvsb_robust_kernel_t, k), PSULVSB_LOSS_L2, "
                   "PSULVSB_LOSS_HUBER, PSULVSB_LOSS_CAUCHY, PSULVSB_LOSS_GM, PSULVSB_LOSS_TUKEY);\n"
                   "  return 0;\n}\n")
    exe = str(tmp_path / "rk")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe])
    got = list(map(int, subprocess.check_output([exe], text=True).split()))
    K = capi.RobustKernel
    assert got == [C.sizeof(K), K.type.offset, K.k.offset, capi.LOSS_L2, capi.LOSS_HUBER, capi.LOSS_CAUCHY,
                   capi.LOSS_GM, capi.LOSS_TUKEY]
    assert [c.type for c in (I.L2Loss(), I.HuberLoss(1), I.CauchyLoss(1), I.GMLoss(1), I.TukeyLoss(1))] == \
        [RR.L2, RR.HUBER, RR.CAUCHY, RR.GM, RR.TUKEY]


def test_robust_correspondence_kernels_do_not_spill(tmp_path):
    """k9_robust_p2l_correspond and k9_robust_gicp_correspond run without local memory (sm_100a, -Xptxas -v)."""
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
        m = re.search(r"Function properties for \S*(k9_robust_(?:p2l|gicp)_correspond)", line)
        if not m:
            continue
        f = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", lines[i + 1])
        assert f and f.groups() == ("0", "0", "0"), lines[i:i + 3]
        regs[m.group(1)] = int(re.search(r"Used (\d+) registers", lines[i + 2]).group(1))
    assert sorted(regs) == ["k9_robust_gicp_correspond", "k9_robust_p2l_correspond"], regs


def test_weights_at_their_edges():
    k = 0.25
    r = np.array([0.0, -0.0, k, -k, np.nextafter(k, 1), 2 * k, 1e300, -1e-300])
    assert np.array_equal(RR.weight((RR.L2, nan), r), np.ones(r.size))
    for kind in (RR.HUBER, RR.CAUCHY, RR.GM, RR.TUKEY):
        w = RR.weight((kind, k), r)
        assert (w >= 0).all() and np.isfinite(w).all(), kind
        assert w[0] == w[1] == RR.weight((kind, k), np.array([1e-300]))[0], kind          # r = 0: the top weight
        assert w[2] == w[3], kind                                                         # even in r
    h = RR.weight((RR.HUBER, k), r)
    assert h[0] == 1.0 and h[2] == 1.0 and h[5] == 0.5
    assert abs(h[4] - 1.0) <= np.finfo(float).eps                                         # continuous at k
    assert RR.weight((RR.CAUCHY, k), np.array([k]))[0] == 0.5
    assert RR.weight((RR.GM, k), np.array([0.0]))[0] == 1.0 / k                           # k / k^2
    t = RR.weight((RR.TUKEY, k), r)
    assert t[0] == 1.0 and t[2] == 0.0 and t[4] == 0.0 and t[5] == 0.0 and t[6] == 0.0    # 0 from |r| = k on
    assert RR.weight((RR.TUKEY, k), np.array([k / 2]))[0] == 0.5625                       # (1 - 1/4)^2


def _unit(rng, K):
    x = rng.normal(size=(3, K))
    return x / np.linalg.norm(x, axis=0)


def _full(W, i):
    W00, W01, W02, W11, W12, W22 = (w[i] for w in W)
    return np.array([[W00, W01, W02], [W01, W11, W12], [W02, W12, W22]])


@pytest.mark.parametrize("eps", [1.0, 0.5, 1e-3, 1e-6])
def test_whitening_is_the_inverse_square_root_of_the_covariance(eps):
    rng = np.random.default_rng(11)
    K = 60
    m, n = _unit(rng, K), _unit(rng, K)
    n[:, 0], n[:, 1] = m[:, 0], -m[:, 1]                           # m = +-n: v2 = 0
    n[:, 2] = -m[:, 2] + 1e-9 * rng.normal(size=3)                 # nearly antiparallel
    n[:, 2] /= np.linalg.norm(n[:, 2])
    n[:, 3] = m[:, 3] + 1e-12
    n[:, 3] /= np.linalg.norm(n[:, 3])
    m[:, 4] = 0.0                                                  # one normal
    n[:, 5] = 0.0
    m[:, 6] = n[:, 6] = 0.0                                        # neither: I / sqrt2
    n[:, 7] = [-m[1, 7], m[0, 7], 0.0] / np.linalg.norm(m[:2, 7])  # m . n = 0: s = +1
    w = 1.0 - eps
    W = RR.whitening(m, n, w)
    Cm = G.covariance(m, n, w)
    M = G.inverse(Cm)
    for i in range(K):
        Wi = _full(W, i)
        Ci = _full(Cm, i)
        Mi = np.array([[M[r][c][i] for c in range(3)] for r in range(3)])
        ref = np.real(sqrtm(np.linalg.inv(Ci)))
        scale = np.abs(ref).max()
        # sqrtm loses digits as C's condition grows (2 / (2 eps)); the closed form does not
        assert np.abs(Wi - ref).max() <= max(1e-13, 1e-9 * eps ** -0.5 * 1e-3) * scale, (i, eps)
        # M = adj(C) / det(C) carries C's condition (1 / eps) in its rounding too
        assert np.abs(Wi.T @ Wi - Mi).max() <= (1e-13 + 4e-16 / eps) * np.abs(Mi).max(), (i, eps)
    assert np.array_equal(_full(W, 6), np.eye(3) * RR.INV_SQRT2)
    # signs of the normals do not change W
    assert all(np.array_equal(a, b) for a, b in zip(W, RR.whitening(-m, n, w)))


def _problem(K, seed):
    rng = np.random.default_rng(seed)
    Pp = rng.normal(size=(3, K))
    Q = Pp + 0.05 * rng.normal(size=(3, K))
    Ns, Nt = rng.normal(size=(3, K)), rng.normal(size=(3, K))
    R, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    return Pp, Q, Ns, Nt, R * np.sign(np.linalg.det(R)), np.arange(K)


def test_l2_point_to_plane_terms_are_the_plain_terms_bit_for_bit():
    Pp, Q, _, Nt, _, _ = _problem(300, 7)
    Nt = Nt / np.linalg.norm(Nt, axis=0)
    h, g = RR.p2l_terms(Pp, Q, Nt, (RR.L2, 1.0))
    r = ((Pp[0] - Q[0]) * Nt[0] + (Pp[1] - Q[1]) * Nt[1]) + (Pp[2] - Q[2]) * Nt[2]
    J = np.concatenate([G.cross(Pp, Nt), Nt])
    assert np.array_equal(h, np.stack([J[a] * J[e] for a in range(6) for e in range(a, 6)]))
    assert np.array_equal(g, J * r)


@pytest.mark.parametrize("eps", [1e-3, 0.25, 1.0, 1e-6])
def test_l2_robust_gicp_update_is_gicps(eps):
    """W^T W = M: the L2 system is generalized ICP's, summed in another order."""
    Pp, Q, Ns, Nt, R, corr = _problem(400, 3)
    Ns[:, 0] = np.nan
    Nt[:, 1] = 0.0
    Nt[:, 2] = Ns[:, 2] = np.nan
    H0, g0 = G.system(Pp, Q, Ns, Nt, R, corr, eps)
    H1, g1 = RR.system(Pp, Q, corr, (RR.L2, 1.0), src_normals=Ns, tgt_normals=Nt, R_k=R, epsilon=eps)
    scale = np.abs(H0).max()
    assert np.abs(H1 - H0).max() <= 1e-11 * scale and np.abs(g1 - g0).max() <= 1e-11 * scale
    x0, x1 = G.solve6(H0, g0), G.solve6(H1, g1)
    assert np.abs(x1 - x0).max() <= 1e-9 * max(1.0, np.abs(x0).max())


def rot(axis, deg):
    ax = np.asarray(axis, dtype=np.float64)
    ax = ax / np.linalg.norm(ax)
    a = np.deg2rad(deg)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    return np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K


def outlier_scene(seed, n=20, clutter=0.25, offset=0.04, sigma=0.002):
    """Three orthogonal n x n planes (a room corner) seen twice with noise sigma, and in the source a clutter sheet of
    clutter * 3 n^2 points `offset` above the floor: each finds a floor point within d and pulls the floor's pose by
    offset.  Returns src, src normals, tgt, tgt normals (3 x N each), R_true, t_true."""
    rng = np.random.default_rng(seed)
    g = (np.arange(n) + 0.5) / n
    u, v = [a.ravel() for a in np.meshgrid(g, g)]
    z = np.zeros_like(u)
    P = np.concatenate([np.stack([u, v, z]), np.stack([u, z, v]), np.stack([z, u, v])], axis=1)
    N = np.concatenate([np.tile([[0], [0], [1.0]], n * n), np.tile([[0], [1.0], [0]], n * n),
                        np.tile([[1.0], [0], [0]], n * n)], axis=1)
    m = int(clutter * P.shape[1])
    sheet = np.stack([rng.random(m), rng.random(m), np.full(m, offset)])
    R_true, t_true = rot(rng.normal(size=3), 3.0), np.array([0.02, -0.01, 0.015])
    Q = R_true @ P + t_true[:, None] + sigma * rng.normal(size=P.shape)
    return (np.concatenate([P, sheet], axis=1), np.concatenate([N, np.tile([[0], [0], [1.0]], m)], axis=1), Q,
            R_true @ N, R_true, t_true)


def pose_errors(R, t, R_true, t_true):
    """(rotation error in degrees, translation error)."""
    c = np.clip((np.trace(R.T @ R_true) - 1) / 2, -1, 1)
    return float(np.rad2deg(np.arccos(c))), float(np.linalg.norm(t - t_true))


OUTLIER_D, OUTLIER_START = 0.08, (rot([1, 2, 3], 2.0), 0.01)


@pytest.mark.parametrize("objective", ["p2l", "gicp"])
def test_robust_kernels_reject_structured_outliers_in_the_restatement(objective):
    """With the clutter sheet inside d, L2's translation is pulled about 0.015 off; Tukey and Cauchy with k = 5 sigma
    (the sheet's residuals are 20 sigma) land at least 5 times closer."""
    for seed in (0, 1):
        S, Sn, Q, Nt, R_true, t_true = outlier_scene(seed)
        R0, t0 = OUTLIER_START[0] @ R_true, t_true + OUTLIER_START[1]
        kw = dict(normals=Nt) if objective == "p2l" else dict(src_normals=Sn, tgt_normals=Nt, epsilon=1e-3)
        err = {name: pose_errors(*(lambda r: (r["R"], r["t"]))(RR.icp(S, Q, R0, t0, OUTLIER_D, loss, **kw)), R_true,
                                 t_true)
               for name, loss in (("l2", (RR.L2, 1.0)), ("tukey", (RR.TUKEY, 0.01)), ("cauchy", (RR.CAUCHY, 0.01)))}
        assert err["l2"][1] > 0.01, err
        for name in ("tukey", "cauchy"):
            assert err[name][1] < err["l2"][1] / 5, (seed, name, err)
    assert OI.NO_UPDATE == 2
