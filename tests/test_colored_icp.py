"""CPU-side checks of colored ICP and its colour-gradient stage: argument refusals of the six entry points before any
device work, psulvsb_colored_icp_pair_t and psulvsb_color_cloud_t against their ctypes mirrors, the workspace sizes,
the new kernels' registers, and self-checks of the numpy restatement (tests/colored_icp_restatement.py): gradients of
linear fields, degenerate neighbourhoods, lambda = 1 against point-to-plane's terms bit for bit, and a textured plane
on which point-to-plane has no update and colored ICP recovers the in-plane motion."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from oracle import icp as OI
from psulvsb_b200 import capi, features
from psulvsb_b200 import icp as I
from tests import colored_icp_restatement as CR
from tests import robust_icp_restatement as RR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "probabilistic-self-update-line-vector-set-based-point-cloud-registration_b200", "csrc")
PTS = np.zeros((3, 4))
INV = (capi.ERR_INVALID,) * 4
NOD = (capi.ERR_NO_DEVICE,) * 4
nan, inf = float("nan"), float("inf")

# the textured plane (textured_plane): n points on z = 0 at unit mean spacing, intensity 0.5 + 0.25 sin(2 pi x / L)
# sin(2 pi y / L), the source an independent resampling moved by 1 degree about z and (0.8, 0.6, 0)
PLANE_L, PLANE_D = 20.0, 3.0
# bounds on the recovered motion, from the numpy loop (about 6e-4 degrees and 6e-4 spacings on seeds 0-2) with margin
PLANE_MAX_DEG, PLANE_MAX_T = 0.01, 0.01


def plane_field(x, y):
    return 0.5 + 0.25 * np.sin(2 * np.pi * x / PLANE_L) * np.sin(2 * np.pi * y / PLANE_L)


def textured_plane(seed=0, n=20_000):
    """(P, Q, Cs, Ct, Nt, R_true, t_true): Q ~ R_true P + t_true on z = 0, Nt exactly (0, 0, 1)."""
    rng = np.random.default_rng(seed)
    W = np.sqrt(n)

    def sample():
        xy = rng.uniform(0.0, W, (2, n))
        I = plane_field(xy[0], xy[1])
        return np.vstack([xy, np.zeros(n)]), np.vstack([I, I, I])

    Q, Ct = sample()
    Sw, Cs = sample()
    a = np.deg2rad(1.0)
    R = np.array([[np.cos(a), -np.sin(a), 0.0], [np.sin(a), np.cos(a), 0.0], [0.0, 0.0, 1.0]])
    t = np.array([0.8, 0.6, 0.0])
    P = R.T @ (Sw - t[:, None])
    P[2] = 0.0
    Nt = np.zeros((3, n))
    Nt[2] = 1.0
    return P, Q, Cs, Ct, Nt, R, t


def pose_errors(R, t, R_true, t_true):
    """(rotation error in degrees, translation error)."""
    c = np.clip((np.trace(R @ R_true.T) - 1.0) / 2.0, -1.0, 1.0)
    return float(np.degrees(np.arccos(c))), float(np.linalg.norm(t - t_true))


def params(**kw):
    p = capi.IcpParams()
    capi.lib().psulvsb_icp_default_params(C.byref(p))
    p.max_correspondence_distance = 0.1
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def kernel(loss):
    return None if loss is None else C.byref(capi.RobustKernel(*loss))


def cpairs(specs):
    arr = (capi.ColoredIcpPair * max(len(specs), 1))()
    for b, spec in enumerate(specs):
        q = arr[b]
        q.src = q.tgt = q.src_colors = q.tgt_colors = q.tgt_normals = PTS.ctypes.data
        q.n_s = q.n_t = 4
        q.R0[:] = [1, 0, 0, 0, 1, 0, 0, 0, 1]
        for k, v in spec.items():
            setattr(q, k, v)
    return arr


def colored_codes(p, lam=0.968, loss=None, pair=None, R0=None):
    """psulvsb_colored_icp, _host, _batch and _batch_host on the same arguments (pair: fields of the pair)."""
    L = capi.lib()
    q = cpairs([pair or {}])[0]
    R = (C.c_double * 9)(*(R0 or [1, 0, 0, 0, 1, 0, 0, 0, 1]))
    t = (C.c_double * 3)(0, 0, 0)
    pp = C.byref(p) if p is not None else None
    a = [q.src, q.n_s, q.src_colors, q.tgt, q.n_t, q.tgt_colors, q.tgt_normals, pp, lam, kernel(loss), R, t]
    res = (capi.IcpResult * 2)()
    ptr = PTS.ctypes.data
    arr = cpairs([pair or {}, {}])
    arr[0].R0[:] = list(R)
    return (L.psulvsb_colored_icp(None, *a, ptr, ptr, None, None), L.psulvsb_colored_icp_host(*a, res, None, None),
            L.psulvsb_colored_icp_batch(None, arr, 2, pp, lam, kernel(loss), ptr, ptr, None, None),
            L.psulvsb_colored_icp_batch_host(arr, 2, pp, lam, kernel(loss), res, None, None))


def test_colored_icp_refuses_bad_arguments_before_any_device_work():
    good = params()
    for loss in [(-1, 1.0), (5, 1.0)] + [(t, k) for t in (1, 2, 3, 4) for k in (0.0, -1.0, nan, inf, -inf)]:
        assert colored_codes(good, loss=loss) == INV, loss
    for lam in (-0.1, 1.0 + 1e-12, nan, inf, -inf):
        assert colored_codes(good, lam=lam) == INV, lam
    # the entry points are the mode, and refuse what psulvsb_icp[_batch] refuses
    for p in (None, params(point_to_plane=1), params(point_to_plane=2), params(max_correspondence_distance=0.0),
              params(max_correspondence_distance=nan), params(max_iterations=-1), params(relative_rmse=nan),
              params(relative_fitness=-1.0)):
        assert colored_codes(p) == INV
    for pair in ({"n_s": -1}, {"n_t": -1}, {"src": None}, {"tgt": None}, {"src_colors": None}, {"tgt_colors": None},
                 {"tgt_normals": None}, {"src_colors": None, "n_t": 0}, {"tgt_normals": None, "n_s": 0}):
        assert colored_codes(good, pair=pair) == INV, pair
    assert colored_codes(good, R0=[1, 0, 0, 0, nan, 0, 0, 0, 1]) == INV
    L = capi.lib()
    p = C.byref(good)
    assert L.psulvsb_colored_icp_batch(None, cpairs([{}]), -1, p, 0.5, None, PTS.ctypes.data, PTS.ctypes.data, None,
                                       None) == capi.ERR_INVALID
    assert L.psulvsb_colored_icp_batch(None, cpairs([{}]), 1, p, 0.5, None, None, PTS.ctypes.data, None,
                                       None) == capi.ERR_INVALID
    assert L.psulvsb_colored_icp_batch_host(None, 1, p, 0.5, None, None, None, None) == capi.ERR_INVALID
    assert L.psulvsb_colored_icp_batch(None, cpairs([{}]), 0, p, 0.5, None, None, None, None, None) == capi.OK
    # the sizes past 2^31 - 1 in all, before any device work
    big = cpairs([{"n_s": 2 ** 30, "n_t": 4}, {"n_s": 2 ** 30, "n_t": 4}])
    assert L.psulvsb_colored_icp_batch_host(big, 2, p, 0.5, None, (capi.IcpResult * 2)(), None,
                                            None) == capi.ERR_UNSUPPORTED
    if L.psulvsb_device_count() == 0:
        for lam, loss in ((0.0, None), (1.0, None), (0.968, (0, nan)), (0.5, (4, 0.1)), (0.3, (3, 1e-4))):
            assert colored_codes(good, lam=lam, loss=loss) == NOD, (lam, loss)
        assert colored_codes(good, pair={"src_colors": None, "n_s": 0}) == NOD      # an empty cloud needs no colours
        with pytest.raises(capi.PsulvsbError):
            I.colored_icp(PTS, PTS, PTS, PTS, PTS, np.eye(3), np.zeros(3), 0.1)
    with pytest.raises(ValueError):
        I.colored_icp(PTS, PTS, PTS[:, :3], PTS, PTS, np.eye(3), np.zeros(3), 0.1)
    with pytest.raises(ValueError):
        I.colored_icp_batch([PTS], [PTS], [PTS], [PTS], [], np.eye(3)[None], np.zeros((1, 3)), 0.1)


def gradient_codes(clouds, B, radius=0.5, max_nn=30, out=True):
    L = capi.lib()
    ptr = PTS.ctypes.data
    return (L.psulvsb_color_gradients_batch(None, clouds, B, radius, max_nn, ptr, ptr if out else None),
            L.psulvsb_color_gradients_batch_host(clouds, B, radius, max_nn, ptr if out else None))


def ccloud(**kw):
    arr = (capi.ColorCloud * 2)()
    for q in arr:
        q.points = q.colors = q.normals = PTS.ctypes.data
        q.n = 4
    for k, v in kw.items():
        setattr(arr[0], k, v)
    return arr


def test_color_gradients_refuse_bad_arguments_before_any_device_work():
    inv2 = (capi.ERR_INVALID,) * 2
    for radius in (0.0, -1.0, nan, inf):
        assert gradient_codes(ccloud(), 2, radius=radius) == inv2, radius
    for max_nn in (0, 3, 33, -1):
        assert gradient_codes(ccloud(), 2, max_nn=max_nn) == inv2, max_nn
    for kw in ({"n": -1}, {"points": None}, {"colors": None}, {"normals": None}):
        assert gradient_codes(ccloud(**kw), 2) == inv2, kw
    assert gradient_codes(ccloud(), -1) == inv2
    assert gradient_codes(ccloud(), 2, out=False) == inv2
    assert gradient_codes(ccloud(), 0) == (capi.OK,) * 2
    big = ccloud(n=2 ** 30)
    big[1].n = 2 ** 30
    assert gradient_codes(big, 2) == (capi.ERR_UNSUPPORTED,) * 2
    if capi.lib().psulvsb_device_count() == 0:
        assert gradient_codes(ccloud(), 2, max_nn=4) == (capi.ERR_NO_DEVICE,) * 2
        assert gradient_codes(ccloud(n=0, colors=None, normals=None, points=None), 2, max_nn=32) == \
            (capi.ERR_NO_DEVICE,) * 2
        with pytest.raises(capi.PsulvsbError):
            features.color_gradients(PTS, PTS, PTS, 0.5)


def test_colored_structs_match_the_header(tmp_path):
    src = tmp_path / "sizes.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "psulvsb.h"\n'
                   "int main(void) {\n"
                   '  printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(psulvsb_colored_icp_pair_t), '
                   "offsetof(psulvsb_colored_icp_pair_t, src_colors), offsetof(psulvsb_colored_icp_pair_t, n_t), "
                   "offsetof(psulvsb_colored_icp_pair_t, tgt_colors), offsetof(psulvsb_colored_icp_pair_t, "
                   "tgt_normals), offsetof(psulvsb_colored_icp_pair_t, R0), offsetof(psulvsb_colored_icp_pair_t, t0),"
                   " sizeof(psulvsb_color_cloud_t));\n"
                   '  printf("%zu %zu %zu\\n", offsetof(psulvsb_color_cloud_t, n), '
                   "offsetof(psulvsb_color_cloud_t, colors), offsetof(psulvsb_color_cloud_t, normals));\n"
                   "  return 0;\n}\n")
    exe = str(tmp_path / "sizes")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe])
    a, b = [list(map(int, line.split())) for line in subprocess.check_output([exe], text=True).splitlines()]
    P, K = capi.ColoredIcpPair, capi.ColorCloud
    assert a == [C.sizeof(P), P.src_colors.offset, P.n_t.offset, P.tgt_colors.offset, P.tgt_normals.offset,
                 P.R0.offset, P.t0.offset, C.sizeof(K)]
    assert b == [K.n.offset, K.colors.offset, K.normals.offset]


def test_workspace_sizes():
    """The sizes only: ICP's workspace (or the gradient stage's scratch, whichever is larger) plus the side table and
    24 bytes per live target point; ICP's own published sizes do not change."""
    L = capi.lib()
    assert L.psulvsb_colored_icp_workspace_bytes(-1, 5) == 0 and L.psulvsb_colored_icp_workspace_bytes(5, -1) == 0
    assert L.psulvsb_colored_icp_batch_workspace_bytes(cpairs([{}]), 0) == 0
    assert L.psulvsb_colored_icp_batch_workspace_bytes(cpairs([{"n_s": -1}]), 1) == 0
    assert L.psulvsb_color_gradients_batch_workspace_bytes(ccloud(n=-1), 2) == 0
    for ns, nt in ((1, 1), (1000, 5000), (5000, 1000), (100_000, 300_000), (0, 1000), (1000, 0)):
        w = L.psulvsb_colored_icp_workspace_bytes(ns, nt)
        live_t = nt if ns and nt else 0
        assert w >= L.psulvsb_icp_workspace_bytes(ns, nt) + 24 * live_t, (ns, nt)
        arr = cpairs([{"n_s": ns, "n_t": nt, "src": None, "tgt": None}])
        assert L.psulvsb_colored_icp_batch_workspace_bytes(arr, 1) == w
        cl = ccloud(n=live_t)
        assert w >= L.psulvsb_color_gradients_batch_workspace_bytes(cl, 1) + 24 * live_t
    assert L.psulvsb_icp_workspace_bytes(1000, 5000) == L.psulvsb_gicp_batch_workspace_bytes(
        (capi.GicpPair * 1)(capi.GicpPair(None, 1000, None, 5000)), 1)
    arr = cpairs([{"n_s": 7000, "n_t": 9000}, {"n_s": 0, "n_t": 50}, {"n_s": 3000, "n_t": 4000}])
    assert L.psulvsb_colored_icp_batch_workspace_bytes(arr, 3) >= \
        L.psulvsb_colored_icp_workspace_bytes(7000, 9000) + 24 * 4000


def test_new_kernels_do_not_spill(tmp_path):
    """k9_colored_correspond and k8_color_gradients run without a stack frame or local memory (sm_100a,
    -Xptxas -v)."""
    nvcc = "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    found = {}
    for src, name in (("k9_icp.cu", "k9_colored_correspond"), ("k8_colors.cu", "k8_color_gradients")):
        r = subprocess.run([nvcc, "-O3", "-std=c++17", "-fmad=false", "-gencode", "arch=compute_100a,code=sm_100a",
                            "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", os.path.join(CSRC, src), "-o",
                            str(tmp_path / (src + ".o"))], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr
        lines = r.stderr.splitlines()
        for i, line in enumerate(lines):
            if "Function properties for" in line and name in line:
                f = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                              lines[i + 1])
                assert f and f.groups() == ("0", "0", "0"), lines[i:i + 3]
                found[name] = int(re.search(r"Used (\d+) registers", lines[i + 2]).group(1))
    assert sorted(found) == ["k8_color_gradients", "k9_colored_correspond"], found


def jittered_plane(n_side, normal, seed, jitter=0.3):
    """(points, e1, e2): a jittered n_side^2 grid of unit spacing on the plane through the origin normal to `normal`."""
    rng = np.random.default_rng(seed)
    n = np.asarray(normal, dtype=np.float64)
    n = n / np.linalg.norm(n)
    e1 = np.cross(n, [1.0, 0.0, 0.0] if abs(n[0]) < 0.9 else [0.0, 1.0, 0.0])
    e1 /= np.linalg.norm(e1)
    e2 = np.cross(n, e1)
    u, v = np.meshgrid(np.arange(n_side, dtype=np.float64), np.arange(n_side, dtype=np.float64))
    u = u.ravel() + rng.uniform(-jitter, jitter, u.size)
    v = v.ravel() + rng.uniform(-jitter, jitter, v.size)
    return np.outer(e1, u) + np.outer(e2, v), e1, e2, n


def test_linear_field_on_a_plane_gives_its_in_plane_gradient():
    for seed, normal in enumerate(([0, 0, 1], [0.3, -0.5, 0.8], [1, 2, -0.5])):
        P, e1, e2, n = jittered_plane(30, normal, seed)
        alpha, beta = 0.013, -0.021
        I = 0.4 + alpha * (e1 @ P) + beta * (e2 @ P)
        N = np.repeat(n[:, None], P.shape[1], axis=1)
        G, frag = CR.gradients(P, np.vstack([I, I, I]), N, 2.5)
        want = alpha * e1 + beta * e2
        ok = ~frag
        assert ok.sum() > 0.9 * P.shape[1]
        err = np.abs(G[:, ok] - want[:, None]).max()
        assert err <= 1e-12 * np.linalg.norm(want), (seed, err)


def test_gradients_are_nearly_perpendicular_to_the_normal():
    """The row (nn - 1) n pins g . n: on a sphere of radius 20 with exact normals and a smooth colour field, |g . n| is
    far below |g|."""
    rng = np.random.default_rng(5)
    X = rng.normal(size=(3, 8000))
    N = X / np.linalg.norm(X, axis=0)
    P = 20.0 * N
    I = 0.5 + 0.3 * np.sin(P[0] / 7.0) * np.cos(P[1] / 5.0)
    G, frag = CR.gradients(P, np.vstack([I, I, I]), N, 2.0)
    gn = np.abs((G * N).sum(axis=0))
    g = np.linalg.norm(G, axis=0)
    sel = (~frag) & (g > 0)
    assert sel.sum() > 7000
    assert (gn[sel] <= 0.05 * g[sel]).all(), (gn[sel] / g[sel]).max()
    # exactly perpendicular where the plane is exact: z = 0 with n = e_z
    P2, _, _, _ = jittered_plane(20, [0, 0, 1], 3)
    P2[2] = 0.0
    N2 = np.zeros_like(P2)
    N2[2] = 1.0
    I2 = 0.5 + 0.2 * np.sin(P2[0] / 3.0) * np.sin(P2[1] / 4.0)
    G2, _ = CR.gradients(P2, np.vstack([I2, I2, I2]), N2, 2.0)
    assert np.array_equal(G2[2], np.zeros(P2.shape[1])) and np.abs(G2[:2]).max() > 0.01


def test_too_few_and_collinear_neighbourhoods_give_zero():
    # nn < 4: three points, or points whose neighbourhoods hold at most three
    P = np.array([[0.0, 1.0, 0.0, 10.0, 11.0, 10.0, 10.5], [0.0, 0.0, 1.0, 0.0, 0.0, 1.0, 0.5],
                  [0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0]])
    Cc = np.vstack([np.linspace(0, 1, 7)] * 3)
    N = np.zeros((3, 7))
    N[2] = 1.0
    G, _ = CR.gradients(P, Cc, N, 1.5)
    assert np.array_equal(G[:, :3], np.zeros((3, 3)))            # nn = 3
    assert np.abs(G[:, 3:]).max() > 0                             # nn = 4
    G, _ = CR.gradients(P, Cc, N, 1.5, max_nn=4)
    assert np.abs(G[:, 3:]).max() > 0
    # collinear: every row along x, the constraint along z: the second pivot is exactly 0
    x = np.arange(12, dtype=np.float64)
    L = np.vstack([x, np.zeros(12), np.zeros(12)])
    G, _ = CR.gradients(L, np.vstack([x / 12] * 3), np.repeat([[0.0], [0.0], [1.0]], 12, axis=1), 3.0)
    assert np.array_equal(G, np.zeros((3, 12)))
    # a non-finite normal: g = 0
    P3, _, _, n3 = jittered_plane(10, [0, 0, 1], 1)
    N3 = np.repeat(n3[:, None], 100, axis=1)
    N3[:, 7] = nan
    I3 = 0.1 * P3[0]
    G3, _ = CR.gradients(P3, np.vstack([I3] * 3), N3, 2.0)
    assert np.array_equal(G3[:, 7], np.zeros(3)) and np.abs(G3[:, 6]).max() > 0


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def test_lambda_one_terms_are_point_to_plane_bit_for_bit():
    """With lambda = 1 the photometric row is sqrt(0) times finite numbers: zeros, which leave the geometric terms as
    they are, signed zeros included (p' on z = 0 with n = e_z makes many of them -0)."""
    rng = np.random.default_rng(11)
    K = 4000
    p = rng.normal(size=(3, K)) * 5
    q = p + rng.normal(size=(3, K)) * 0.1
    n = rng.normal(size=(3, K))
    n /= np.linalg.norm(n, axis=0)
    p[2, :1000] = q[2, :1000] = 0.0
    n[:, :1000] = [[0.0], [0.0], [1.0]]
    g = rng.normal(size=(3, K)) * 0.05
    Is, It = rng.uniform(size=K), rng.uniform(size=K)
    h, gg = CR.terms(p, q, n, g, Is, It, 1.0)
    hr, gr = RR.p2l_terms(p, q, n, (RR.L2, 1.0))
    assert np.array_equal(bits(h), bits(hr)) and np.array_equal(bits(gg), bits(gr))
    assert (np.signbit(h) & (h == 0)).any()                      # the case the zero rule is for
    # an IEEE sum would have lost those signs
    h2, _ = CR.terms(p, q, n, g, Is, It, 0.5)
    assert not np.array_equal(bits(h2), bits(hr))
    # the photometric row alone at lambda = 0
    h0, g0 = CR.terms(p, q, n, g, Is, It, 0.0)
    m = -(g - ((g[0] * n[0] + g[1] * n[1]) + g[2] * n[2]) * n)
    J = np.concatenate([np.cross(p.T, m.T).T, m])
    r = Is - (((g[0] * (p[0] - q[0]) + g[1] * (p[1] - q[1])) + g[2] * (p[2] - q[2])) + It)
    assert np.allclose(h0.sum(axis=1), np.array([(J[a] * J[e]).sum() for a in range(6) for e in range(a, 6)]),
                       rtol=1e-12)
    assert np.allclose(g0.sum(axis=1), (J * r).sum(axis=1), rtol=1e-12)


def test_nonfinite_colours_stop_the_loop_with_no_update():
    P, Q, Cs, Ct, Nt, R, t = textured_plane(4, n=2000)
    Cs[:, 17] = nan
    out = CR.colored_icp(P, Q, Cs, Ct, Nt, np.eye(3), np.zeros(3), PLANE_D, 0.968)
    assert out["status"] == OI.NO_UPDATE and out["iterations"] == 0


def test_textured_plane_point_to_plane_stalls_and_colored_icp_recovers_the_motion():
    for seed in (0, 1):
        P, Q, Cs, Ct, Nt, R_true, t_true = textured_plane(seed)
        p2l = OI.icp(P, Q, np.eye(3), np.zeros(3), PLANE_D, normals=Nt, point_to_plane=True)
        assert p2l["status"] == OI.NO_UPDATE and p2l["iterations"] == 0
        Gt, _ = CR.gradients(Q, Ct, Nt, 2 * PLANE_D)
        for lam in (0.968, 0.5):
            out = CR.colored_icp(P, Q, Cs, Ct, Nt, np.eye(3), np.zeros(3), PLANE_D, lam, Gt=Gt)
            err = pose_errors(out["R"], out["t"], R_true, t_true)
            assert out["status"] == OI.CONVERGED and out["iterations"] >= 2, (seed, lam, out["status"])
            assert err[0] < PLANE_MAX_DEG and err[1] < PLANE_MAX_T, (seed, lam, err)
