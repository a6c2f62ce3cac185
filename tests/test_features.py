"""CPU-side checks of the correspondence stage (FPFH descriptors, descriptor nearest neighbours, matcher): the numpy
restatement (oracle/features.py) on hand-built cases, the C ABI's errors without a device, the C++ facade's call
sequence, and the packed FP32 loop of the nearest-neighbour kernel."""
import ctypes as C
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from oracle import features as F
from oracle import oracle as O
from psulvsb_b200 import capi, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
up = np.array([0.0, 0.0, 1.0], dtype=np.float32)


def feats(p, n_p, q, n_q):
    f = F.pair_features(np.array([p], np.float32), np.array([n_p], np.float32), np.array([q], np.float32),
                        np.array([n_q], np.float32))
    return float(f[0][0]), float(f[1][0]), float(f[2][0]), bool(f[3][0])


def test_pair_features_swap_branch_and_skips():
    # |a1| = 0 < |a2|: the roles swap, d is negated and f3 = -a2
    s2 = math.sqrt(0.5)
    f1, f2, f3, ok = feats([0, 0, 0], up, [1, 0, 0], [s2, 0, s2])
    assert ok and f3 == pytest.approx(-s2, abs=1e-6)
    # no swap: f3 = a1
    f1, f2, f3, ok = feats([0, 0, 0], [s2, 0, s2], [1, 0, 0], up)
    assert ok and f3 == pytest.approx(s2, abs=1e-6)
    # coincident points and a normal parallel to d are skipped, so is a NaN normal
    assert not feats([0, 0, 0], up, [0, 0, 0], up)[3]
    assert not feats([0, 0, 0], up, [0, 0, 1], up)[3]
    assert not feats([0, 0, 0], [np.nan] * 3, [1, 0, 0], up)[3]
    # two parallel normals on a plane: f1 = atan2(0, 1) = 0, f2 = 0, f3 = 0
    f1, f2, f3, ok = feats([0, 0, 0], up, [1, 1, 0], up)
    assert ok and (f1, f2, f3) == (0.0, 0.0, 0.0)


def test_bin_edges():
    args = F.bin_args(np.float32([-math.pi, np.float32(math.pi)]), np.float32([-1, 1]), np.float32([0, 1]))
    bins = np.clip(np.floor(args).astype(int), 0, 10)
    assert bins[:, 0].tolist() == [0, 10] and bins[:, 1].tolist() == [0, 10]   # upper edges clamp to the last bin
    assert bins[:, 2].tolist() == [5, 10]


def test_isolated_point_and_nan_normals():
    pts = np.array([[0, 0.01, 0.02, 0.0, 5.0], [0, 0.0, 0.01, 0.02, 5.0], [0, 0.001, 0.0, 0.002, 5.0]])
    f, normals, _ = F.fpfh(pts, 0.05, 0.05)
    assert np.isnan(normals[:, 4]).all() and not np.isnan(normals[:, :4]).any()
    assert (f[4] == 0).all()                                      # isolated: all-zero descriptor
    for h in range(3):
        assert np.allclose(f[:4, h * 11:(h + 1) * 11].sum(axis=1), 100.0, atol=1e-4)
    # two points only: fewer than 3 neighbours -> NaN normals -> every pair skipped -> zero descriptors
    f2, n2, _ = F.fpfh(pts[:, :2], 0.05, 0.05)
    assert np.isnan(n2).all() and (f2 == 0).all()


def test_restated_descriptors_are_rotation_invariant():
    P = synth.make_surface(3000, 2)
    R, _ = synth.random_rigid(np.random.default_rng(4))
    t = np.array([0.5, -1.0, 0.25])
    f0, _, _ = F.fpfh(P, 0.08, 0.12)
    f1, _, _ = F.fpfh(R @ P + t[:, None], 0.08, 0.12, viewpoint=t)   # the viewpoint moves with the cloud
    l1 = np.abs(f1 - f0).sum(axis=1)
    assert (l1 <= 1e-3).mean() >= 0.99


def test_nn_ties_go_to_the_lowest_index():
    fs = np.zeros((3, 33), np.float32)
    ft = np.zeros((4, 33), np.float32)
    fs[1, 0] = 1.0
    ft[2, 0] = 1.0
    ft[3, 0] = 1.0
    a, b, _, fr_t = F.nearest_neighbours(fs, ft)
    assert a.tolist() == [0, 2, 0]
    assert b.tolist() == [0, 0, 1, 1]
    d = F.descriptor_distances(fs, ft)
    assert d[1, 2] == 0 and d[0, 2] == 1


def test_list_orders():
    nn_t = np.array([1, 0, 1, 2])       # source -> target
    nn_s = np.array([1, 2, 0])          # target -> source
    assert F.match_list(nn_t, nn_s, True).tolist() == [[1, 0], [2, 1]]
    # one-way: (i, nn_t(i)) for i in {0, 1, 2} (the sources some target picked) ascending, then (nn_s(j), j)
    assert F.match_list(nn_t, nn_s, False).tolist() == [[0, 1], [1, 0], [2, 1], [1, 0], [2, 1], [0, 2]]


def test_tuple_test_on_a_fixed_stream():
    rng = np.random.default_rng(0)
    src = rng.uniform(-1, 1, (3, 40))
    tgt = src.copy()
    tgt[:, 30:] = rng.uniform(-1, 1, (3, 10))          # 10 wrong pairs
    corr = np.stack([np.arange(40), np.arange(40)], axis=1)
    pairs, _ = F.tuple_test(src, tgt, corr, 0.95, 11)
    assert pairs.shape == (3000, 2)                    # 4000 trials, more than 1000 pass
    draws = F.tuple_draws(11, 0, 5, 40)
    assert draws[0, 0] == O.rand31(11, F.DOMAIN_TUPLE, 0, 0) % 40
    assert draws[4, 2] == O.rand31(11, F.DOMAIN_TUPLE, 0, 14) % 40
    s32, t32 = src.T.astype(np.float32), tgt.T.astype(np.float32)
    kept = []
    for tri in F.tuple_draws(11, 0, 4000, 40):        # trial by trial, in order
        ok = True
        for e in range(3):
            a, b = tri[e], tri[(e + 1) % 3]
            li, lj = np.linalg.norm(s32[a] - s32[b]), np.linalg.norm(t32[a] - t32[b])
            ok = ok and li * np.float32(0.95) < lj < li / np.float32(0.95)
        if ok:
            kept.extend(tri)
        if len(kept) == 3000:
            break
    assert pairs[:, 0].tolist() == kept
    small, _ = F.tuple_test(src[:, :2], tgt[:, :2], corr[:2], 0.95, 11)
    assert small.shape == (0, 2)                       # a degenerate triangle never passes


def test_entries_refuse_bad_arguments_and_need_a_device():
    L = capi.lib()
    pts = np.zeros((3, 4))
    f = np.zeros((4, 33), np.float32)
    nn = np.zeros(4, np.int32)
    n = C.c_longlong(0)
    P, FS, NN = pts.ctypes.data, f.ctypes.data, nn.ctypes.data
    for bad in (0.0, -1.0, float("nan"), float("inf")):
        assert L.psulvsb_fpfh_host(P, 4, bad, 0.1, None, None, FS) == capi.ERR_INVALID
        assert L.psulvsb_fpfh_host(P, 4, 0.1, bad, None, None, FS) == capi.ERR_INVALID
        assert L.psulvsb_fpfh(None, P, 4, bad, 0.1, None, P, None, FS) == capi.ERR_INVALID
    assert L.psulvsb_fpfh_host(None, 4, 0.1, 0.1, None, None, FS) == capi.ERR_INVALID
    assert L.psulvsb_fpfh(None, P, 4, 0.1, 0.1, None, None, None, FS) == capi.ERR_INVALID
    assert L.psulvsb_feature_nn(None, None, 4, FS, 4, NN, NN) == capi.ERR_INVALID
    assert L.psulvsb_match_host(P, 4, P, 4, FS, FS, 1, 0, 0.95, 0, NN, 2, None) == capi.ERR_INVALID
    assert L.psulvsb_match_host(P, 4, None, 4, FS, FS, 1, 0, 0.95, 0, NN, 2, C.byref(n)) == capi.ERR_INVALID
    assert L.psulvsb_fpfh_workspace_bytes(50000) >= 50000 * (16 + 16 + 33 * 4)
    if L.psulvsb_device_count() == 0:
        assert L.psulvsb_fpfh_host(P, 4, 0.1, 0.2, None, None, FS) == capi.ERR_NO_DEVICE
        assert L.psulvsb_fpfh(None, P, 4, 0.1, 0.2, None, P, None, FS) == capi.ERR_NO_DEVICE
        assert L.psulvsb_feature_nn(None, FS, 4, FS, 4, NN, NN) == capi.ERR_NO_DEVICE
        assert L.psulvsb_match_host(P, 4, P, 4, FS, FS, 1, 1, 0.95, 0, NN, 2, C.byref(n)) == capi.ERR_NO_DEVICE
        assert b"no CUDA device" in L.psulvsb_last_error()
        from psulvsb_b200 import features

        with pytest.raises(capi.PsulvsbError):
            features.fpfh(pts, 0.1, 0.2)
        with pytest.raises(capi.PsulvsbError):
            features.match(pts, pts, f, f)


def build_fpfh_snippet(tmp_path):
    exe = str(tmp_path / "fpfh_snippet")
    libdir = os.path.dirname(capi.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
                           "-I", os.path.join(ROOT, "tests", "shim"), os.path.join(ROOT, "tests", "cpp", "fpfh_snippet.cc"),
                           "-o", exe, "-L", libdir, "-l:libpsulvsb_b200.so", "-Wl,-rpath," + libdir])
    return exe


def test_fpfh_facade_compiles_links_and_fails_loudly_without_gpu(tmp_path):
    exe = build_fpfh_snippet(tmp_path)
    if capi.lib().psulvsb_device_count() > 0:
        pytest.skip("GPU present: covered by the gpu-marked test")
    r = subprocess.run([exe, "500"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 3 and "no CUDA device" in r.stdout, r.stdout + r.stderr


def test_feature_nn_loop_is_packed():
    """The descriptor distance loop runs on packed FP32: FADD2 for two columns' differences, FFMA2 for their squares."""
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", capi.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    ops, name = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
        elif name and "k8_feature_nn" in name:
            for op in ("FFMA2", "FADD2", "FFMA"):
                if re.search(r"\b%s\b" % op, line):
                    ops[op] = ops.get(op, 0) + 1
    assert ops.get("FFMA2", 0) >= 32 and ops.get("FFMA2", 0) > ops.get("FFMA", 0), ops
    assert ops.get("FADD2", 0) >= 32, ops


def exact_fma32(a, b, c):
    """float32(a * b + c) rounded once (round half to even), from exact rationals: the reference for fmaf."""
    from fractions import Fraction

    x = Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))
    if x == 0:
        return np.float32(0.0)
    m, e = abs(x), 0
    while m >= 2:
        m, e = m / 2, e + 1
    while m < 1:
        m, e = m * 2, e - 1
    q = abs(x) / Fraction(2) ** (e - 23)          # the 24-bit significand, scaled to an integer part
    r = math.floor(q)
    if q - r > Fraction(1, 2) or (q - r == Fraction(1, 2) and r % 2):
        r += 1
    return np.float32(math.copysign(float(r * Fraction(2) ** (e - 23)), x))


def test_fma32_rounds_once():
    y = 2.0 ** -10
    # a * b + c lands a quarter float64 ulp off a float32 midpoint: float64 rounding alone would hit the midpoint
    # and round half-to-even the wrong way
    cases = [(1 + y, 2.0 ** -24 * (1 - y + y * y), 1.0, 1 + 2.0 ** -23),                   # 1 + 2^-24 + 2^-54
             (1 - y, 2.0 ** -24 * (1 + y + y * y), 1 + 2.0 ** -23, 1 + 2.0 ** -23),        # 1 + 3 2^-24 - 2^-54
             (-(1 + y), 2.0 ** -24 * (1 - y + y * y), -1.0, -(1 + 2.0 ** -23))]
    for a, b, c, want in cases:
        a, b, c = np.float32(a), np.float32(b), np.float32(c)
        assert F.fma32(a, b, c) == np.float32(want) == exact_fma32(a, b, c)
        assert np.float32(float(a) * float(b) + float(c)) != np.float32(want)   # the naive double rounding is wrong
    rng = np.random.default_rng(0)
    a = rng.normal(0, 1, 3000).astype(np.float32)
    b = (rng.normal(0, 1, 3000) * 10.0 ** rng.integers(-8, 8, 3000)).astype(np.float32)
    c = (rng.normal(0, 1, 3000) * 10.0 ** rng.integers(-8, 8, 3000)).astype(np.float32)
    got = F.fma32(a, b, c)
    assert all(got[i] == exact_fma32(a[i], b[i], c[i]) for i in range(3000))
    # the k-NN normals' distance: fmaf(dz, dz, fmaf(dy, dy, dx * dx))
    d = rng.normal(0, 1, (3, 500)).astype(np.float32)
    from oracle import prefilter as OP

    P = np.concatenate([np.zeros((3, 1)), d], axis=1).astype(np.float32)
    got = OP.knn_sqdist32(P, np.array([0]))[0, 1:]
    want = [exact_fma32(z, z, exact_fma32(y, y, np.float32(x * x))) for x, y, z in d.T]
    assert np.array_equal(got, np.array(want, dtype=np.float32))
    # descriptor distances take the same path; an overflow is inf
    big = np.full((1, 33), 1e20, np.float32)
    assert np.isinf(F.descriptor_distances(big, -big)).all()


def test_knn_restatement_ties_and_fragile_rule():
    from oracle import prefilter as OP

    vp = (0.3, 0.2, 5.0)
    base = np.array([[0.0, 1.0, 0.0, 0.0], [0.0, 0.0, 1.0, 0.0], [0.0, 0.0, 0.0, 1.0]])
    # point 0's 2nd, 3rd and 4th neighbours tie exactly at d^2 = 1: k = 3 keeps the lower indices 1 and 2, so the
    # normal is the plane z = 0's; an exact tie is not fragile
    nv, frag = OP.knn_pca_normals(base, k=3, viewpoint=vp, return_fragile=True)
    assert np.allclose(nv[:, 0], [0, 0, 1]) and not frag[0]
    # point 3 a hair further (d^2 = 1 + 2^-22 in FP32, 2.4e-7 relative): the same pick, but fragile
    near = base.copy()
    near[2, 3] = 1 + 2.0 ** -23
    nv, frag = OP.knn_pca_normals(near, k=3, viewpoint=vp, return_fragile=True)
    assert np.allclose(nv[:, 0], [0, 0, 1]) and frag[0]
    # 1e-5 relative further: not fragile
    far = base.copy()
    far[2, 3] = 1 + 1e-5
    assert not OP.knn_pca_normals(far, k=3, viewpoint=vp, return_fragile=True)[1][0]
    # the same cloud in another order: the two lowest tied indices, now (0, 0, 1) and (0, 1, 0), set the plane
    swapped = base[:, [0, 3, 2, 1]]
    nv = OP.knn_pca_normals(swapped, k=3, viewpoint=vp)
    assert np.allclose(nv[:, 0], [1, 0, 0])               # plane x = 0
    # n < k uses all n points; n < 3 is NaN; the default call returns the normals only
    assert OP.knn_pca_normals(base, k=20).shape == (3, 4)
    assert np.isnan(OP.knn_pca_normals(base[:, :2], k=20)).all()
    assert np.isnan(OP.knn_pca_normals(base[:, :1], k=3)).all()


def test_vectorised_philox_matches_the_oracle():
    rng = np.random.default_rng(2)
    blocks = np.concatenate([np.arange(0, 1000, dtype=np.uint64), rng.integers(0, 2 ** 62, 1000, dtype=np.uint64),
                             np.arange(2 ** 30 - 500, 2 ** 30 + 500, dtype=np.uint64),
                             np.arange(2 ** 32 - 300, 2 ** 32 + 300, dtype=np.uint64),
                             np.array([2 ** 64 - 1], dtype=np.uint64)])
    for seed in (0, 11, (7 << 32) | 5):
        got = F.philox_blocks(seed, F.DOMAIN_TUPLE, 0, blocks)
        want = np.stack([O.philox(seed, F.DOMAIN_TUPLE, 0, int(b)) for b in blocks])
        assert np.array_equal(got, want)
    assert np.array_equal(F.philox_blocks(3, 2, 9, blocks[:50]), np.stack([O.philox(3, 2, 9, int(b))
                                                                           for b in blocks[:50]]))
    # draws of trials whose 3t + k crosses 2^32 (blocks above 2^32 / 4)
    t0 = (2 ** 32) // 3 - 5
    d = F.tuple_draws(11, t0, 10, 1000)
    for u in range(10):
        for k in range(3):
            assert d[u, k] == O.rand31(11, F.DOMAIN_TUPLE, 0, 3 * (t0 + u) + k) % 1000


@pytest.mark.parametrize("offset", [0.0, 1e3])
def test_neighbours_match_brute_force(offset):
    """The k-d tree query (radius widened by 1e-4) finds every pair the FP32 distance test accepts."""
    rng = np.random.default_rng(3)
    P = rng.uniform(0, 1, (3, 300)) + offset
    p32 = P.T.astype(np.float32)
    for r in (0.05, 0.2, 0.6):
        ii, jj, d2, _, _ = F.neighbours(P, r)
        d = np.stack([F.sqdist32(np.repeat(p32[i:i + 1], 300, 0), p32) for i in range(300)])
        bi, bj = np.nonzero(d <= np.float32(r * r))
        assert np.array_equal(ii, bi) and np.array_equal(jj, bj)
        assert np.array_equal(d2, d[bi, bj])
