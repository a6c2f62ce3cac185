"""CPU-side checks of the ICP refinement: the numpy restatement (oracle/icp.py) on hand-built cases, the C ABI's errors
without a device, the ctypes structs against the header, and the correspondence kernel's registers."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from oracle import icp as OI
from psulvsb_b200 import capi, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "probabilistic-self-update-line-vector-set-based-point-cloud-registration_b200", "csrc")


def small_rotation(rng, angle):
    axis = rng.normal(size=3)
    axis /= np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * K @ K


def surface_normals(P):
    """Unit normals of z = 0.3 sin(2x) cos(3y) + 0.1 x y (synth.make_surface)."""
    x, y = P[0], P[1]
    fx = 0.6 * np.cos(2 * x) * np.cos(3 * y) + 0.1 * y
    fy = -0.9 * np.sin(2 * x) * np.sin(3 * y) + 0.1 * x
    n = np.stack([-fx, -fy, np.ones_like(x)])
    return n / np.linalg.norm(n, axis=0)


def test_point_to_point_recovers_a_rigid_transform_in_one_update():
    rng = np.random.default_rng(0)
    g = np.stack(np.meshgrid(*[np.arange(6) * 0.2] * 3, indexing="ij")).reshape(3, -1)
    P = g + rng.uniform(-0.02, 0.02, g.shape)                    # nearest neighbours >= 0.16 apart
    R, _ = synth.random_rigid(rng)
    t = np.array([0.3, -2.0, 1.5])
    Q = R @ P + t[:, None]
    R0 = small_rotation(rng, 0.01) @ R
    t0 = t + 0.005
    out = OI.icp(P, Q, R0, t0, 0.05, max_iterations=1)
    assert out["trace"][0][4] == P.shape[1]                      # T0 already pairs every point with its counterpart
    assert out["status"] == OI.MAX_ITERATIONS and out["iterations"] == 1
    assert np.abs(out["R"] - R).max() <= 1e-12 and np.abs(out["t"] - t).max() <= 1e-12
    assert np.array_equal(out["corr"], np.arange(P.shape[1])) and out["inlier_rmse"] <= 1e-12


def test_point_to_plane_converges_on_the_surface():
    P = synth.make_surface(3000, 1)
    rng = np.random.default_rng(1)
    R, _ = synth.random_rigid(rng)
    t = np.array([0.5, 0.1, -0.2])
    Q, N = R @ P + t[:, None], R @ surface_normals(P)
    R0, t0 = small_rotation(rng, np.deg2rad(1.0)) @ R, t + np.array([0.01, -0.005, 0.008])
    out = OI.icp(P, Q, R0, t0, 0.1, normals=N, point_to_plane=True, max_iterations=6, relative_fitness=0,
                 relative_rmse=0)
    err = [np.abs(Rk - R).max() + np.abs(tk - t).max() for Rk, tk, *_ in out["trace"]]   # (arccos: no digits < 1e-8)
    assert out["status"] == OI.MAX_ITERATIONS and len(err) == 7
    for a, b in zip(err, err[1:]):
        assert b < a or b <= 1e-12, err                          # shrinks until it reaches the rounding floor
    assert err[-1] <= 1e-9, err


def test_correspondence_ties_boundary_and_nan_normals():
    Q = np.array([[0.0, 1.0, 5.0, 1.0, 0.0], [0.0, 0.0, 5.0, 0.0, 0.0], [0.0, 0.0, 5.0, 0.0, 0.5]])
    # source 0 sits on target 0; source 1 at d = 1 from target 0 and on targets 1 and 3 (a tie: the lower index);
    # source 2 has nothing within d; source 3 is one ulp further than d from target 0
    P = np.array([[0.0, 1.0, 3.0, 0.0], [0.0, 0.0, 3.0, 0.0], [0.0, 0.0, 3.0, np.nextafter(-1.0, -2.0)]])
    corr, d2 = OI.correspond(P, Q, 1.0)
    assert corr.tolist() == [0, 1, -1, -1]
    assert d2[1] == 0.0 and np.isinf(d2[2])
    # the d^2 <= d d boundary: at exactly d the pair counts, one ulp further it does not
    corr, d2 = OI.correspond(np.array([[0.0], [0.0], [-1.0]]), Q[:, :1], 1.0)
    assert corr.tolist() == [0] and d2[0] == 1.0
    assert OI.correspond(P[:, 3:], Q[:, :1], 1.0)[0].tolist() == [-1]
    # point-to-plane: a NaN normal takes its point out; the next nearest answers
    N = np.tile([[0.0], [0.0], [1.0]], (1, 5))
    N[:, 0] = np.nan
    corr, _ = OI.correspond(P, Q, 1.0, normals=N)
    assert corr.tolist() == [4, 1, -1, -1]
    assert OI.candidate_mask(Q, N).tolist() == [False, True, True, True, True]


def test_transform_order_and_squared_distance_order():
    rng = np.random.default_rng(5)
    P = rng.normal(0, 1e3, (3, 50))
    R, _ = synth.random_rigid(rng)
    t = rng.normal(0, 1e3, 3)
    got = OI.transform(P, R, t)
    for r in range(3):
        want = [((R[r, 0] * x + R[r, 1] * y) + R[r, 2] * z) + t[r] for x, y, z in P.T]
        assert got[r].tolist() == want
    Q = rng.normal(0, 1e3, (3, 50))
    i, j = np.arange(50), np.arange(50)[::-1]
    want = []
    for a, b in zip(i.tolist(), j.tolist()):
        dx, dy, dz = (float(Q[r, b]) - float(got[r, a]) for r in range(3))
        want.append((dx * dx + dy * dy) + dz * dz)
    assert OI.sqdist(got, Q, i, j).tolist() == want


def test_status_two_cases():
    rng = np.random.default_rng(2)
    P = rng.uniform(0, 1, (3, 40))
    Q = P.copy()
    eye, zero = np.eye(3), np.zeros(3)
    for n in (1, 2):                                             # fewer than 3 correspondences: no update
        out = OI.icp(P[:, :n], Q, eye, zero, 0.1)
        assert out["status"] == OI.NO_UPDATE and out["iterations"] == 0 and out["n_corr"] == n
        assert len(out["trace"]) == 1
    N = np.tile([[0.0], [0.0], [1.0]], (1, 40))
    out = OI.icp(P[:, :5], Q, eye, zero, 0.1, normals=N, point_to_plane=True)
    assert out["status"] == OI.NO_UPDATE and out["n_corr"] == 5   # fewer than 6
    # all normals parallel: J^T J has zero rows (rotation about z, x and y translation), a zero pivot
    out = OI.icp(P, Q, eye, zero, 0.1, normals=N, point_to_plane=True)
    assert out["status"] == OI.NO_UPDATE and out["n_corr"] == 40 and out["iterations"] == 0
    for a, b in ((P[:, :0], Q), (P, Q[:, :0])):                  # empty clouds
        out = OI.icp(a, b, eye, zero, 0.1)
        assert out["status"] == OI.NO_UPDATE and out["fitness"] == 0.0 and out["iterations"] == 0
    out = OI.icp(P, Q, eye, zero, 0.1, max_iterations=0)
    assert out["status"] == OI.MAX_ITERATIONS and len(out["trace"]) == 1 and out["fitness"] == 1.0


def test_stop_rule():
    assert OI.stop(0, None, (0.5, 0.1), 30, 1e-6, 1e-6) is None
    assert OI.stop(1, (0.5, 0.1), (0.5, 0.1), 30, 1e-6, 1e-6) == OI.CONVERGED
    assert OI.stop(1, (0.5, 0.1), (0.5, 0.1), 30, 0.0, 0.0) is None         # strict: criteria 0 never converge
    assert OI.stop(3, (0.5, 0.1), (0.6, 0.1), 3, 1e-6, 1e-6) == OI.MAX_ITERATIONS
    assert OI.stop(3, (0.5, 0.1), (0.5, 0.1), 3, 1e-6, 1e-6) == OI.CONVERGED


def test_icp_entries_refuse_bad_arguments_and_need_a_device():
    L = capi.lib()
    pts = np.zeros((3, 4))
    P = pts.ctypes.data
    corr = np.zeros(4, np.int32)
    R = (C.c_double * 9)(1, 0, 0, 0, 1, 0, 0, 0, 1)
    t = (C.c_double * 3)(0, 0, 0)
    res = capi.IcpResult()

    def params(**kw):
        p = capi.IcpParams()
        L.psulvsb_icp_default_params(C.byref(p))
        p.max_correspondence_distance = 0.1
        for k, v in kw.items():
            setattr(p, k, v)
        return p

    p = params()
    assert (p.max_iterations, p.relative_fitness, p.relative_rmse, p.point_to_plane) == (30, 1e-6, 1e-6, 0)
    bad = [params(max_correspondence_distance=v) for v in (0.0, -1.0, float("nan"), float("inf"))]
    bad += [params(max_iterations=-1), params(relative_fitness=-1e-6), params(relative_rmse=float("nan")),
            params(point_to_plane=2)]
    for b in bad:
        assert L.psulvsb_icp_host(P, 4, P, 4, P, C.byref(b), R, t, C.byref(res), None, None) == capi.ERR_INVALID
        assert L.psulvsb_icp(None, P, 4, P, 4, P, C.byref(b), R, t, P, P, None, None) == capi.ERR_INVALID
    good = params()
    for badR in ((C.c_double * 9)(1, 0, 0, 0, float("nan"), 0, 0, 0, 1), None):
        assert L.psulvsb_icp_host(P, 4, P, 4, None, C.byref(good), badR, t, C.byref(res), None, None) == capi.ERR_INVALID
    for badt in ((C.c_double * 3)(0, float("inf"), 0), None):
        assert L.psulvsb_icp_host(P, 4, P, 4, None, C.byref(good), R, badt, C.byref(res), None, None) == capi.ERR_INVALID
    p2l = params(point_to_plane=1)
    assert L.psulvsb_icp_host(P, 4, P, 4, None, C.byref(p2l), R, t, C.byref(res), None, None) == capi.ERR_INVALID
    assert L.psulvsb_icp(None, P, 4, P, 4, None, C.byref(p2l), R, t, P, P, None, None) == capi.ERR_INVALID
    assert L.psulvsb_icp_host(P, -1, P, 4, None, C.byref(good), R, t, C.byref(res), None, None) == capi.ERR_INVALID
    assert L.psulvsb_icp_host(P, 4, P, -1, None, C.byref(good), R, t, C.byref(res), None, None) == capi.ERR_INVALID
    assert L.psulvsb_icp_host(None, 4, P, 4, None, C.byref(good), R, t, C.byref(res), None, None) == capi.ERR_INVALID
    assert L.psulvsb_icp_host(P, 4, None, 4, None, C.byref(good), R, t, C.byref(res), None, None) == capi.ERR_INVALID
    assert L.psulvsb_icp_host(P, 4, P, 4, None, None, R, t, C.byref(res), None, None) == capi.ERR_INVALID
    assert L.psulvsb_icp_host(P, 4, P, 4, None, C.byref(good), R, t, None, None, None) == capi.ERR_INVALID
    assert L.psulvsb_icp(None, P, 4, P, 4, None, C.byref(good), R, t, None, P, None, None) == capi.ERR_INVALID  # work
    assert L.psulvsb_icp(None, P, 4, P, 4, None, C.byref(good), R, t, P, None, None, None) == capi.ERR_INVALID  # result
    assert L.psulvsb_icp_workspace_bytes(-1, 5) == 0
    assert L.psulvsb_icp_workspace_bytes(50000, 50000) >= 50000 * (32 + 4 + 4 + 4) + 50000 * 4
    assert L.psulvsb_icp_workspace_bytes(1000, 7) == L.psulvsb_icp_workspace_bytes(1000, 7)
    if L.psulvsb_device_count() == 0:
        assert L.psulvsb_icp_host(P, 4, P, 4, None, C.byref(good), R, t, C.byref(res), None,
                                  corr.ctypes.data) == capi.ERR_NO_DEVICE
        assert L.psulvsb_icp(None, P, 4, P, 4, None, C.byref(good), R, t, P, P, None, None) == capi.ERR_NO_DEVICE
        assert b"no CUDA device" in L.psulvsb_last_error()
        from psulvsb_b200 import icp

        with pytest.raises(capi.PsulvsbError):
            icp.icp(pts, pts, np.eye(3), np.zeros(3), 0.1)


def test_icp_structs_match_the_header(tmp_path):
    src = tmp_path / "sizes.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "psulvsb.h"\n'
                   "int main(void) {\n"
                   '  printf("%zu %zu %zu\\n", sizeof(psulvsb_icp_params_t), sizeof(psulvsb_icp_result_t), '
                   "sizeof(psulvsb_icp_iteration_t));\n"
                   '  printf("%zu %zu %zu %zu\\n", offsetof(psulvsb_icp_params_t, max_iterations), '
                   "offsetof(psulvsb_icp_result_t, fitness), offsetof(psulvsb_icp_result_t, status), "
                   "offsetof(psulvsb_icp_iteration_t, n_correspondences));\n"
                   "  return 0;\n}\n")
    exe = str(tmp_path / "sizes")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe])
    sizes, offs = [list(map(int, line.split())) for line in subprocess.check_output([exe], text=True).splitlines()]
    assert sizes == [C.sizeof(capi.IcpParams), C.sizeof(capi.IcpResult), C.sizeof(capi.IcpIteration)]
    assert offs == [capi.IcpParams.max_iterations.offset, capi.IcpResult.fitness.offset, capi.IcpResult.status.offset,
                    capi.IcpIteration.n_correspondences.offset]


def test_correspondence_kernel_does_not_spill(tmp_path):
    """k9_icp_correspond keeps its 27-cell walk and its per-CTA sums in registers (sm_100a, -Xptxas -v)."""
    nvcc = "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    r = subprocess.run([nvcc, "-O3", "-std=c++17", "-fmad=false", "-gencode", "arch=compute_100a,code=sm_100a",
                        "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-c", os.path.join(CSRC, "k9_icp.cu"), "-o",
                        str(tmp_path / "k9_icp.o")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    found = 0
    lines = r.stderr.splitlines()
    for i, line in enumerate(lines):
        if "Function properties for" in line and "k9_icp_correspond" in line:
            found += 1
            m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", lines[i + 1])
            assert m and m.groups() == ("0", "0", "0"), lines[i:i + 3]
    assert found == 2                                           # point-to-point and point-to-plane
