"""The correspondence stage on the GPU against the numpy restatement (oracle/features.py): radius normals, FPFH
descriptors, the two-way descriptor nearest neighbour, the matcher's lists and tuple test, and registration from raw
clouds end to end (Python and the C++ example)."""
import os
import subprocess

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from oracle import features as OF
from psulvsb_b200 import capi, features, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bunny():
    return np.load(os.path.join(ROOT, "tests", "golden", "bunny_res3.npz"))["vertices"].astype(np.float64) * 10


def rigid(seed):
    R, _ = synth.random_rigid(np.random.default_rng(seed))
    return R, np.array([0.4, -0.3, 0.2])


def test_radius_normals_vs_restatement(bunny):
    _, got = features.fpfh(bunny, 0.08, 0.15)
    want, _ = OF.radius_normals(bunny, 0.08)
    assert np.array_equal(np.isnan(got[0]), np.isnan(want[0]))
    ok = ~np.isnan(want[0])
    assert np.allclose(np.linalg.norm(got[:, ok], axis=0), 1.0, atol=1e-9)
    cos = np.abs((got[:, ok] * want[:, ok]).sum(axis=0))
    assert (cos > 1 - 1e-6).mean() > 0.995
    assert ((got[:, ok] * want[:, ok]).sum(axis=0) > 0)[cos > 1 - 1e-6].all()


@pytest.mark.parametrize("cloud,rn,rf", [("bunny", 0.08, 0.15), ("bunny", 0.1, 0.25), ("surface", 0.03, 0.05)])
def test_fpfh_vs_restatement(bunny, cloud, rn, rf):
    P = bunny if cloud == "bunny" else synth.make_surface(20000, 3)
    got, _ = features.fpfh(P, rn, rf)
    want, _, fragile = OF.fpfh(P, rn, rf)
    l1 = np.abs(got.astype(np.float64) - want).sum(axis=1)
    assert l1[~fragile].max(initial=0) <= 1e-3, (np.argmax(np.where(fragile, 0, l1)), l1[~fragile].max())
    assert (l1 <= 1e-3).mean() >= 0.99


def test_fpfh_is_deterministic_and_host_equals_device(bunny):
    import torch

    from psulvsb_b200 import stages

    a, na = features.fpfh(bunny, 0.08, 0.15)
    b, nb = features.fpfh(bunny, 0.08, 0.15)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(na, nb, equal_nan=True)
    d, dn = features.fpfh_device(stages.to_device_points(bunny), 0.08, 0.15)
    torch.cuda.synchronize()
    assert np.array_equal(d.cpu().numpy().view(np.uint32), a.view(np.uint32))
    assert np.array_equal(dn.cpu().numpy().T, na, equal_nan=True)
    e, _ = features.fpfh(np.zeros((3, 0)), 0.08, 0.15)
    assert e.shape == (0, 33)


def test_fpfh_rigid_invariance(bunny):
    R, t = rigid(8)
    a, _ = features.fpfh(bunny, 0.08, 0.15)
    b, _ = features.fpfh(R @ bunny + t[:, None], 0.08, 0.15, viewpoint=t)
    assert (np.abs(a - b).sum(axis=1) <= 1e-3).mean() >= 0.99


@pytest.mark.parametrize("ns,nt", [(1, 1), (1, 7), (9, 1), (1001, 777), (2049, 4099)])
def test_feature_nn_vs_restatement(bunny, ns, nt):
    f, _ = features.fpfh(bunny, 0.08, 0.15)
    rng = np.random.default_rng(ns * 7 + nt)
    fs = f[rng.integers(0, f.shape[0], ns)]
    ft = f[rng.integers(0, f.shape[0], nt)]          # repeated descriptors: exact ties, lowest index wins
    ft[::3] += rng.normal(0, 0.5, ft[::3].shape).astype(np.float32)
    a, b = features.nearest_neighbours(fs, ft)
    wa, wb, fa, fb = OF.nearest_neighbours(fs, ft)
    assert np.array_equal(a[~fa], wa[~fa]) and np.array_equal(b[~fb], wb[~fb])
    D = OF.descriptor_distances(fs, ft)
    assert np.array_equal(D[np.arange(ns), a], D.min(axis=1))    # fragile or not, the pick is a minimum
    assert np.array_equal(D[b, np.arange(nt)], D.min(axis=0))


def test_match_lists_and_tuple_test_vs_restatement():
    src = synth.make_surface(3000, 5)
    R, t = rigid(9)
    perm = np.random.default_rng(10).permutation(3000)
    tgt = (R @ src + t[:, None])[:, perm]
    tgt += np.random.default_rng(11).normal(0, 0.003, tgt.shape)   # noisy: imperfect lists
    fs, _ = features.fpfh(src, 0.06, 0.1)
    ft, _ = features.fpfh(tgt, 0.06, 0.1, viewpoint=t)
    nn_t, nn_s = features.nearest_neighbours(fs, ft)
    for cross in (True, False):
        got = features.match(src, tgt, fs, ft, crosscheck=cross)
        assert np.array_equal(got, OF.match_list(nn_t, nn_s, cross))
    corr = OF.match_list(nn_t, nn_s, True)
    for seed, scale in ((0, 0.95), (7, 0.9)):
        got = features.match(src, tgt, fs, ft, crosscheck=True, tuple_test=True, tuple_scale=scale, seed=seed)
        want, fragile = OF.tuple_test(src, tgt, corr, scale, seed)
        assert got.shape[0] % 3 == 0 and got.shape[0] <= 3000
        if not fragile:
            assert np.array_equal(got, want)


def test_end_to_end_bunny_python(bunny):
    R, t = rigid(12)
    n = bunny.shape[1]
    perm = np.random.default_rng(13).permutation(n)
    tgt = (R @ bunny + t[:, None])[:, perm]
    fs, _ = features.fpfh(bunny, 0.08, 0.15)
    ft, _ = features.fpfh(tgt, 0.08, 0.15, viewpoint=t)
    pairs = features.match(bunny, tgt, fs, ft, crosscheck=True)
    true = np.argsort(perm)[pairs[:, 0]] == pairs[:, 1]
    assert true.mean() >= 0.9, true.mean()
    extent = np.linalg.norm(np.ptp(bunny, axis=1))
    kw = dict(noise_bound=0.01 * extent, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005,
              wallclock_cap_s=0.0, seed=1)
    h = capi.Handle(0)
    sol, _ = h.solve(capi.default_params(**kw), capi.HostProblem(bunny[:, pairs[:, 0]], tgt[:, pairs[:, 1]]))
    assert sol.valid
    assert synth.rotation_error(sol.R, R) <= np.deg2rad(1.0)
    assert np.linalg.norm(sol.t - t) <= 0.02 * extent


def test_example_binary_registers_the_bunny(tmp_path):
    from tests.test_cpp_facade import write_bunny_ply

    exe = str(tmp_path / "psulvsb_fpfh")
    libdir = os.path.dirname(capi.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
                           "-I", os.path.join(ROOT, "tests", "shim"), os.path.join(ROOT, "examples", "psulvsb_fpfh.cc"),
                           "-o", exe, "-L", libdir, "-l:libpsulvsb_b200.so", "-Wl,-rpath," + libdir])
    ply = str(tmp_path / "bunny.ply")
    write_bunny_ply(ply)
    r = subprocess.run([exe, ply, "10", "0.08", "0.15"], capture_output=True, text=True, timeout=300)
    print(r.stdout)
    assert r.returncode == 0 and "valid=1" in r.stdout, r.stdout + r.stderr
    rot = float(r.stdout.split("rotation_error_deg=")[1].split()[0])
    assert rot <= 1.0


def test_fpfh_snippet_solves(tmp_path):
    from tests.test_features import build_fpfh_snippet

    r = subprocess.run([build_fpfh_snippet(tmp_path), "3000"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "valid=1" in r.stdout, r.stdout + r.stderr
