"""GPU parity tests of the four CUDA stages against the CPU oracle, through the C ABI.

Bars (BASELINE.json north_star): adjacency masks / inlier sets / sample index sequences bit-exact;
floating-point outputs within the tolerance written next to each assert.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def P():
    import psulvsb_b200  # noqa: F401
    from psulvsb_b200 import capi, stages, synth

    if capi.lib().psulvsb_device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback")
    return {"capi": capi, "stages": stages, "synth": synth}


@pytest.fixture(scope="module")
def O():
    from oracle import oracle

    return oracle


def test_philox_stream_matches_oracle(P, O):
    st = P["stages"]
    for seed, dom, ev, first in [(0, 1, 0, 0), (0xDEADBEEFCAFEF00D, 2, 7, 5), (42, 3, 0xFFFFFFFF, 2**33 + 3)]:
        got = st.philox_fill(seed, dom, ev, first, 1000)
        want = np.array([O.rand31(seed, dom, ev, first + k) for k in range(1000)], dtype=np.uint32)
        assert np.array_equal(got, want)


@pytest.mark.parametrize("n,count", [(10, 10), (1000, 100), (1000, 1000), (65536, 20000), (627562, 62756), (7, 1),
                                     (147457, 14000), (150000, 75000), (2000000, 200000), (98304, 30000),
                                     # two-word bucket lists (cfg-B's L sample and basic subset): long windows over
                                     # long ranges; and a range that needs more than 256 one-word buckets
                                     (20_700_000, 2_070_000), (2_070_000, 621_000), (24_000_000, 300_000)])
def test_sampler_replays_rejection_sampling(P, O, n, count):
    st = P["stages"]
    for seed, dom, ev in [(1, 1, 0), (99, 2, 13)]:
        got, consumed = st.sample(seed, dom, ev, n, count)
        want, want_consumed = O.sample_without_replacement(seed, dom, ev, n, count)
        assert np.array_equal(got, want)          # same index sequence, bit-exact
        assert consumed == want_consumed          # same stream position afterwards


def test_sampler_list_overflow_falls_back_to_the_walk(P, O):
    """The per-bucket draw lists have room for the mean + 10 sigma of the uniform draws; should one ever overflow, the
    bucket pass walks the whole window instead.  Forced here by filling the lists only to 100 entries."""
    P["capi"].debug_set("sample_list_cap_test", 100)
    st = P["stages"]
    try:
        for n, count in [(627562, 62756), (150000, 75000)]:
            got, consumed = st.sample(7, 1, 3, n, count)
            want, want_consumed = O.sample_without_replacement(7, 1, 3, n, count)
            assert np.array_equal(got, want) and consumed == want_consumed
    finally:
        P["capi"].debug_set("reset", 0)
    got, consumed = st.sample(7, 1, 3, 627562, 62756)          # and the lists work again afterwards (counters were reset)
    want, want_consumed = O.sample_without_replacement(7, 1, 3, 627562, 62756)
    assert np.array_equal(got, want) and consumed == want_consumed


def test_sampler_small_budget_reports_failure(P):
    got, consumed = P["stages"].sample(5, 1, 0, 1000, 1000, max_draws=1200)
    assert consumed == 0


def _upper(mask_full):
    return np.triu(mask_full, 1)


def test_k1_golden_fixed_scale_inliers(P, golden):
    """The reference's own known answer for the length-consistency test (registration-test.cc:286-291)."""
    st = P["stages"]
    reg, meta = golden["reg"], golden["meta"]
    src, dst = reg["objectIn"], reg["sceneIn"]
    n = src.shape[1]
    r = st.consistency_mask(src, dst, meta["fixed_scale_beta"], symmetrize=True)
    full = st.unpack_mask(r["mask"], n)
    off = ~np.eye(n, dtype=bool)
    assert np.array_equal(full[off], reg["fixed_scale_inliers"].astype(np.uint8))
    assert int(full.sum()) == 4016
    assert np.array_equal(r["row_counts"].cpu().numpy(), np.triu(full, 1).sum(axis=1))


@pytest.mark.parametrize("n,seed,beta,outl", [(33, 0, 0.1, "fpfh"), (257, 1, 0.1, "fpfh"), (1000, 2, 0.1, "gross"),
                                             (2049, 3, 0.02, "fpfh"), (5000, 4, 0.1, "fpfh")])
def test_k1_mask_bit_exact_vs_oracle(P, O, n, seed, beta, outl):
    st, synth = P["stages"], P["synth"]
    pair = synth.make_pair(n, 0.9, seed, outliers=outl)
    r = st.consistency_mask(pair["src"], pair["dst"], beta)
    got = st.unpack_mask(r["mask"], n)
    want = _upper(O.consistency_mask(pair["src"], pair["dst"], beta))
    assert np.array_equal(got, want)                       # every bit, incl. zero lower triangle / diagonal
    assert np.array_equal(r["row_counts"].cpu().numpy(), want.sum(axis=1))
    # the FP64 re-evaluated band is small (counted and reported, north_star)
    assert r["border"] <= 0.02 * n * (n - 1) / 2 + 64
    edges, offsets = st.compact_edges(r["mask"], r["row_counts"], n, r["stride"])
    pi, pj = O.reduced_set(pair["src"], pair["dst"], beta)
    e = edges.cpu().numpy()
    assert np.array_equal(e[:, 0], pi) and np.array_equal(e[:, 1], pj)   # reference order (row-major, i<j)


def test_k1_threshold_band_is_resolved_in_fp64(P, O):
    """Pairs placed within 1e-9 relative of the threshold on either side must match the FP64 oracle."""
    st = P["stages"]
    rng = np.random.default_rng(5)
    n, beta = 512, 0.1
    src = rng.uniform(-1.5, 1.5, (3, n))
    dst = src.copy()
    # make |t_0 - t_k| = |s_0 - s_k| + beta (1 + eps_k): move dst_k radially away from dst_0
    for k in range(1, n):
        d = src[:, k] - src[:, 0]
        L = np.linalg.norm(d)
        eps = (rng.integers(-20, 21)) * 1e-10
        dst[:, k] = dst[:, 0] + d / L * (L + beta * (1 + eps))
    r = st.consistency_mask(src, dst, beta)
    got = st.unpack_mask(r["mask"], n)
    want = _upper(O.consistency_mask(src, dst, beta))
    assert np.array_equal(got, want)
    assert r["border"] >= n - 1   # all of row 0 sits inside the band


def test_k1_short_line_vectors_and_diagonal_words(P, O):
    """Pairs with a + b <= beta^2 (both line vectors shorter than beta: the sign of the square-root-free form is not
    the answer there) next to ordinary ones, at sizes where every row's diagonal word and the arrays' last word are
    only partly live (odd n, n % 32 != 0): every bit against the FP64 oracle."""
    st = P["stages"]
    rng = np.random.default_rng(17)
    for n in (95, 1301):
        beta = 0.1
        src = rng.uniform(-1.5, 1.5, (3, n))
        k = n // 3                                        # a third of the points sit in clumps narrower than beta
        src[:, :k] = src[:, [0]] + rng.uniform(-0.03, 0.03, (3, k))
        src[:, k:2 * k:2] = src[:, [k]] + rng.uniform(-0.04, 0.04, (3, len(range(k, 2 * k, 2))))
        dst = src + rng.uniform(-0.02, 0.02, (3, n))
        dst[:, 2 * k:] = rng.uniform(-2.0, 2.0, (3, n - 2 * k))
        perm = rng.permutation(n)                         # clumps spread over the rows / mask words
        src, dst = np.ascontiguousarray(src[:, perm]), np.ascontiguousarray(dst[:, perm])
        r = st.consistency_mask(src, dst, beta)
        got = st.unpack_mask(r["mask"], n)
        want = _upper(O.consistency_mask(src, dst, beta))
        assert np.array_equal(got, want)
        assert np.array_equal(r["row_counts"].cpu().numpy(), want.sum(axis=1))
        assert want[:, :].sum() > k * (k - 1) // 4        # the clumps are there: their pairs are all consistent


@pytest.mark.parametrize("variant", [1, 2, 4])
def test_k1_rows_per_thread_variants_agree_with_the_oracle(P, O, variant):
    """The launcher picks 1, 2 or 4 rows per thread by the amount of work; every variant has its own row-to-warp
    mapping along the diagonal: all of them bit for bit, on sizes with partly live diagonal / last words, whole and
    as row ranges."""
    st, synth, capi = P["stages"], P["synth"], P["capi"]
    capi.debug_set("k1_variant", variant)
    try:
        for n, seed in ((1301, 21), (2049, 22)):
            pair = synth.make_pair(n, 0.9, seed)
            want = _upper(O.consistency_mask(pair["src"], pair["dst"], 0.1))
            r = st.consistency_mask(pair["src"], pair["dst"], 0.1)
            assert np.array_equal(st.unpack_mask(r["mask"], n), want)
            assert np.array_equal(r["row_counts"].cpu().numpy(), want.sum(axis=1))
            a = st.consistency_mask(pair["src"], pair["dst"], 0.1, 0, 517)
            b = st.consistency_mask(pair["src"], pair["dst"], 0.1, 517, n)
            merged = torch.cat([a["mask"][:517], b["mask"][517:]])
            assert np.array_equal(st.unpack_mask(merged, n), want)
    finally:
        capi.debug_set("reset", 0)


def test_k1_row_sharding_and_symmetrize(P, O):
    st, synth = P["stages"], P["synth"]
    n, beta = 777, 0.1
    pair = synth.make_pair(n, 0.9, 11)
    whole = st.consistency_mask(pair["src"], pair["dst"], beta)
    a = st.consistency_mask(pair["src"], pair["dst"], beta, 0, 300)
    b = st.consistency_mask(pair["src"], pair["dst"], beta, 300, n)
    merged = torch.cat([a["mask"][:300], b["mask"][300:]])
    assert torch.equal(merged, whole["mask"])
    assert torch.equal(torch.cat([a["row_counts"][:300], b["row_counts"][300:]]), whole["row_counts"])
    sym = st.consistency_mask(pair["src"], pair["dst"], beta, symmetrize=True)
    assert np.array_equal(st.unpack_mask(sym["mask"], n), O.consistency_mask(pair["src"], pair["dst"], beta))


def _edges_for(P, O, n, seed, beta=0.1, frac=0.1):
    synth = P["synth"]
    pair = synth.make_pair(n, 0.8, seed)
    pi, pj = O.reduced_set(pair["src"], pair["dst"], beta)
    rng = np.random.default_rng(seed)
    sel = rng.permutation(len(pi))[: max(int(len(pi) * frac), 12)]
    return pair, np.stack([pi[sel], pj[sel]], axis=1).astype(np.int32)


@pytest.mark.parametrize("n,seed,warm", [(400, 0, False), (1500, 1, False), (1500, 2, True), (3000, 3, False)])
def test_gnc_tls_rotation_vs_oracle(P, O, n, seed, warm):
    st = P["stages"]
    pair, e = _edges_for(P, O, n, seed)
    sv = pair["src"][:, e[:, 1]] - pair["src"][:, e[:, 0]]
    tv = pair["dst"][:, e[:, 1]] - pair["dst"][:, e[:, 0]]
    R_init = None
    if warm:
        ax = np.array([0.3, -0.2, 0.9])
        ax /= np.linalg.norm(ax)
        K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
        R_init = pair["R"] @ (np.eye(3) + np.sin(0.02) * K + (1 - np.cos(0.02)) * K @ K)
    Rw, inl_w, its_w, cost_w = O.gnc_tls(sv, tv, 0.1, 100, 1.4, 0.005, R_init)
    d_src, d_dst = st.to_device_points(pair["src"]), st.to_device_points(pair["dst"])
    Rg, inl_g, its_g, cost_g, n_inl = st.gnc_tls_rotation(d_src, d_dst, torch.from_numpy(e).cuda(), 0.1, 100, 1.4, 0.005,
                                                         R_init)
    assert its_g == its_w
    assert np.abs(Rg - Rw).max() < 1e-9                       # bar: 1e-5 rad
    assert np.array_equal(inl_g, inl_w)                       # inlier set bit-exact
    assert n_inl == int(inl_w.sum())
    assert abs(cost_g - cost_w) <= 1e-9 * max(1.0, abs(cost_w))


@pytest.mark.parametrize("K", [1, 2, 3, 5, 12, 32])
def test_gnc_tiny_subsets_replay_the_reference_arithmetic_bit_for_bit(P, O, K):
    """A basic subset of ONE line vector gives H = w x y^T of rank 1: R = V U^T is then decided by how the SVD completes
    the null space from 1-ulp entries, so only the reference's own arithmetic reproduces it.  Subsets of up to 32 line
    vectors run through a single thread that replays the oracle's loop (sequential sums, two-sided Jacobi, no FMA):
    rotation, cost, iteration count and inlier mask must be IDENTICAL, cold and warm started, also when the weights
    become fractional (consistent pairs with a length difference near beta) and when all line vectors are parallel."""
    st = P["stages"]
    rng = np.random.default_rng(100 + K)
    for trial in range(12):
        n = 2 * K
        src = rng.uniform(-1.5, 1.5, (3, n))
        ang = rng.uniform(0.1, 3.0)
        ax = rng.standard_normal(3)
        ax /= np.linalg.norm(ax)
        Kx = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
        Rt = np.eye(3) + np.sin(ang) * Kx + (1 - np.cos(ang)) * Kx @ Kx
        dst = Rt @ src + rng.uniform(-0.04, 0.04, (3, n))
        if trial % 3 == 1:                       # stretch some targets: length differences near beta = 0.1
            dst[:, 1::2] += 0.085 * (dst[:, 1::2] - dst[:, 0::2]) / np.linalg.norm(dst[:, 1::2] - dst[:, 0::2], axis=0)
        if trial % 4 == 3:                       # every line vector parallel: rank 1 whatever K is
            d = src[:, 1] - src[:, 0]
            src[:, 1::2] = src[:, 0::2] + d[:, None] * rng.uniform(0.5, 2.0, K)
            dst = Rt @ src
        e = np.stack([np.arange(0, n, 2), np.arange(1, n, 2)], axis=1).astype(np.int32)
        sv = src[:, e[:, 1]] - src[:, e[:, 0]]
        tv = dst[:, e[:, 1]] - dst[:, e[:, 0]]
        R_init = None
        if trial % 2:
            R_init = Rt @ (np.eye(3) + np.sin(0.05) * Kx + (1 - np.cos(0.05)) * Kx @ Kx)
        Rw, inl_w, its_w, cost_w = O.gnc_tls(sv, tv, 0.1, 100, 1.4, 0.005, R_init)
        Rg, inl_g, its_g, cost_g, n_inl = st.gnc_tls_rotation(st.to_device_points(src), st.to_device_points(dst),
                                                             torch.from_numpy(e).cuda(), 0.1, 100, 1.4, 0.005, R_init)
        assert its_g == its_w
        assert np.array_equal(Rg, Rw), (K, trial, np.abs(Rg - Rw).max())       # bit for bit
        assert np.array_equal(inl_g, inl_w) and n_inl == int(inl_w.sum())
        assert cost_g == cost_w or (np.isinf(cost_g) and np.isinf(cost_w))


def test_gnc_tls_golden_rotation_only(P, O, golden):
    """rotation-solver-test.cc:221-250: rotation_only_src.csv rotated by expected_R, tol 1e-5 rad."""
    st = P["stages"]
    src = golden["reg"]["rotation_only_src"]
    if src.shape[0] != 3:
        src = src.T
    Rexp = np.array(golden["meta"]["expected_R_rotation_only"]).reshape(3, 3)
    gp = golden["meta"]["gnc_tls_params"]
    dst = Rexp @ src
    n = src.shape[1]
    # line vectors = consecutive points (the test feeds the solver raw vectors; use origin-anchored edges)
    pts_s = np.concatenate([np.zeros((3, 1)), src], axis=1)
    pts_d = np.concatenate([np.zeros((3, 1)), dst], axis=1)
    e = np.stack([np.zeros(n, dtype=np.int32), np.arange(1, n + 1, dtype=np.int32)], axis=1)
    Rg, inl, its, cost, n_inl = st.gnc_tls_rotation(st.to_device_points(pts_s), st.to_device_points(pts_d),
                                                    torch.from_numpy(e).cuda(), gp["noise_bound"], gp["max_iterations"],
                                                    gp["gnc_factor"], gp["cost_threshold"])
    assert P["synth"].rotation_error(Rg, Rexp) < 1e-5


@pytest.mark.parametrize("cluster,parking", [(1, True), (4, True), (8, True), (4, False), (24, True), (37, False)])
def test_gnc_batch_parks_sleeping_line_vectors_exactly(P, O, cluster, parking):
    """The shape of one engine tick of cfg-A (K = 22 000 line vectors, 95 % FPFH-style outliers per job).  From the
    tenth iteration on most line vectors sit at weight 0 with a margin the remaining rotation drift cannot consume;
    the kernel parks them (k3_rotation.cu).  Nothing is approximated: rotation, iteration count and the inlier mask --
    reported by ORIGINAL index although the positions were permuted -- must match the oracle's plain loop.  Cluster
    sizes above 8 select the kernel's grid mode (that many CTAs per registration, cooperative launch, partial results
    combined through global memory)."""
    st, synth = P["stages"], P["synth"]
    pair = synth.make_pair(5000, 0.95, 3, outliers="fpfh")
    pi, pj = O.reduced_set(pair["src"], pair["dst"], 0.1)
    rng = np.random.default_rng(cluster)
    B, K = 3, 22000
    edges = np.empty((B, K, 2), dtype=np.int32)
    for b in range(B):
        sel = rng.permutation(len(pi))[:K]
        edges[b, :, 0], edges[b, :, 1] = pi[sel], pj[sel]
    Rg, inl, its, n_inl = st.gnc_tls_rotation_batch(st.to_device_points(pair["src"]), st.to_device_points(pair["dst"]),
                                                    torch.from_numpy(edges).cuda(), 0.1, 100, 1.4, 0.005, cluster=cluster,
                                                    parking=parking)
    for b in range(B):
        sv = pair["src"][:, edges[b, :, 1]] - pair["src"][:, edges[b, :, 0]]
        tv = pair["dst"][:, edges[b, :, 1]] - pair["dst"][:, edges[b, :, 0]]
        Rw, inl_w, its_w, _ = O.gnc_tls(sv, tv, 0.1, 100, 1.4, 0.005)
        assert its[b] == its_w and its_w > 20
        assert np.abs(Rg[b] - Rw).max() < 1e-9
        assert np.array_equal(inl[b], inl_w) and n_inl[b] == int(inl_w.sum())
        assert P["synth"].rotation_error(Rg[b], pair["R"]) < 0.02


@pytest.mark.parametrize("margin", ["1e-9", "1e-4"])
def test_gnc_parking_wakes_line_vectors_up_again(P, O, margin, request):
    """The parking threshold is a performance knob: with a tiny one, line vectors are parked with almost no margin,
    the rotation drift reaches their wake-up values within an iteration or two and the active range is reopened
    again and again.  The result must not change."""
    P["capi"].debug_set("gnc_deep_margin", float(margin))
    request.addfinalizer(lambda: P["capi"].debug_set("reset", 0))
    st, synth = P["stages"], P["synth"]
    pair = synth.make_pair(5000, 0.95, 11, outliers="fpfh")
    pi, pj = O.reduced_set(pair["src"], pair["dst"], 0.1)
    rng = np.random.default_rng(5)
    B, K = 2, 16000
    edges = np.empty((B, K, 2), dtype=np.int32)
    for b in range(B):
        sel = rng.permutation(len(pi))[:K]
        edges[b, :, 0], edges[b, :, 1] = pi[sel], pj[sel]
    for cluster in (1, 4, 20):
        Rg, inl, its, n_inl = st.gnc_tls_rotation_batch(st.to_device_points(pair["src"]), st.to_device_points(pair["dst"]),
                                                        torch.from_numpy(edges).cuda(), 0.1, 100, 1.4, 0.005,
                                                        cluster=cluster)
        for b in range(B):
            sv = pair["src"][:, edges[b, :, 1]] - pair["src"][:, edges[b, :, 0]]
            tv = pair["dst"][:, edges[b, :, 1]] - pair["dst"][:, edges[b, :, 0]]
            Rw, inl_w, its_w, _ = O.gnc_tls(sv, tv, 0.1, 100, 1.4, 0.005)
            assert its[b] == its_w
            assert np.abs(Rg[b] - Rw).max() < 1e-9
            assert np.array_equal(inl[b], inl_w)


def test_kabsch_batch_vs_oracle(P, O):
    st = P["stages"]
    pair, e = _edges_for(P, O, 800, 4, frac=0.2)
    rng = np.random.default_rng(0)
    k, H = 8, 300
    sets = rng.integers(0, len(e), (H, k)).astype(np.int32)
    R, t = st.kabsch_batch(st.to_device_points(pair["src"]), st.to_device_points(pair["dst"]),
                           torch.from_numpy(e).cuda(), torch.from_numpy(sets).cuda(), k)
    R = R.cpu().numpy()
    for h in range(0, H, 7):
        ee = e[sets[h]]
        sv = pair["src"][:, ee[:, 1]] - pair["src"][:, ee[:, 0]]
        tv = pair["dst"][:, ee[:, 1]] - pair["dst"][:, ee[:, 0]]
        Rw = O.svd_rot(sv, tv, np.ones(k))
        Rg = R[h].reshape(3, 3, order="F")
        assert np.allclose(Rg @ Rg.T, np.eye(3), atol=1e-12) and np.linalg.det(Rg) > 0
        assert P["synth"].rotation_error(Rg, Rw) < 1e-7


def test_kabsch_rank2_is_unique_and_matches_oracle(P, O):
    """Two line vectors: H has rank 2, sigma_3 = 0, and R = V diag(1, 1, +-1) U^T is still unique (the third
    singular pair is fixed by orthogonality and the determinant rule, utils.h:131-133).  Basic subsets of two
    line vectors occur on small reduced sets, so this must agree with the oracle like the full-rank case."""
    st = P["stages"]
    pair, e = _edges_for(P, O, 400, 5, frac=0.2)
    rng = np.random.default_rng(1)
    k, H = 2, 400
    sets = np.stack([rng.permutation(len(e))[:k] for _ in range(H)]).astype(np.int32)
    R, _ = st.kabsch_batch(st.to_device_points(pair["src"]), st.to_device_points(pair["dst"]),
                           torch.from_numpy(e).cuda(), torch.from_numpy(sets).cuda(), k)
    R = R.cpu().numpy()
    worst = 0.0
    for h in range(H):
        ee = e[sets[h]]
        sv = pair["src"][:, ee[:, 1]] - pair["src"][:, ee[:, 0]]
        tv = pair["dst"][:, ee[:, 1]] - pair["dst"][:, ee[:, 0]]
        Rw = O.svd_rot(sv, tv, np.ones(k))
        Rg = R[h].reshape(3, 3, order="F")
        assert np.allclose(Rg @ Rg.T, np.eye(3), atol=1e-12) and np.linalg.det(Rg) > 0
        worst = max(worst, float(np.abs(Rg - Rw).max()))
    assert worst < 1e-9, worst


@pytest.mark.parametrize("n,with_last,grid", [(34, False, 0), (300, False, 0), (300, True, 0), (2500, True, 0),
                                              (6000, False, 0), (6000, True, 0), (3000, True, 0.01), (1300, False, 0.02)])
def test_tls_translation_vs_oracle(P, O, n, with_last, grid):
    """Max-stabbing translation against the oracle's sorted sweep.  Up to 1024 measurements the device counts all pairs,
    above it sorts the axis and finds every candidate's members by binary search with the same rounded predicates
    (solve_dev.cuh); `grid` > 0 snaps the measurements to a lattice, so that many candidates tie in depth and many
    endpoints coincide."""
    st = P["stages"]
    rng = np.random.default_rng(n)
    src = rng.uniform(-1, 1, (3, n))
    t_true = np.array([0.3, -0.7, 1.1])
    dst = src + t_true[:, None] + rng.uniform(-0.04, 0.04, (3, n))
    if grid > 0:
        src = np.round(src / grid) * grid
        dst = np.round(dst / grid) * grid
    bad = rng.permutation(n)[: n // 2]
    dst[:, bad] += rng.uniform(-3, 3, (3, len(bad)))
    flags = np.ones(n, dtype=np.uint8)
    flags[rng.permutation(n)[: n // 5]] = 0
    sel = flags.astype(bool)
    last = (t_true + 0.01) if with_last else None
    t_w, _ = O.tls_translation(src[:, sel], dst[:, sel], 0.05, 1.0, last)
    t_g, npts = st.tls_translation(st.to_device_points(src), st.to_device_points(dst), torch.from_numpy(flags).cuda(),
                                   1.0, np.eye(3), 0.05, last)
    assert npts == int(sel.sum())
    assert np.abs(t_g - t_w).max() < 1e-12     # bar: 1e-5 units


def test_tls_translation_golden(P, O, golden):
    """translation-solver-test.cc fixtures through the device max-stabbing == oracle's."""
    st = P["stages"]
    reg = golden["reg"]
    v1, v2 = reg["translation_v1"], reg["translation_v2"]
    t_w, _ = O.tls_translation(v1, v2, 0.05, 1.0, None)
    flags = np.ones(v1.shape[1], dtype=np.uint8)
    t_g, _ = st.tls_translation(st.to_device_points(v1), st.to_device_points(v2), torch.from_numpy(flags).cuda(), 1.0,
                                np.eye(3), 0.05, None)
    assert np.abs(t_g - t_w).max() < 1e-12


def _hypotheses(pair, H, seed):
    rng = np.random.default_rng(seed)
    hyp = np.zeros((H, 12))
    for h in range(H):
        ax = rng.standard_normal(3)
        ax /= np.linalg.norm(ax)
        ang = rng.uniform(0, 0.02) if h % 3 == 0 else rng.uniform(0, np.pi)
        K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
        dR = np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K
        R = dR @ pair["R"]
        t = pair["t"] + (rng.uniform(-0.01, 0.01, 3) if h % 3 == 0 else rng.uniform(-1, 1, 3))
        hyp[h, :9] = R.ravel(order="F")
        hyp[h, 9:] = t
    return hyp


def test_score_one_bit_exact(P, O):
    st = P["stages"]
    pair = P["synth"].make_pair(3000, 0.7, 21)
    hyp = _hypotheses(pair, 4, 0)
    d_src, d_dst = st.to_device_points(pair["src"]), st.to_device_points(pair["dst"])
    for h in range(4):
        R, t = hyp[h, :9].reshape(3, 3, order="F"), hyp[h, 9:]
        cnt_w, inl_w, res_w = O.score(pair["src"], pair["dst"], 1.0, R, t, 0.04)
        cnt_g, inl_g, res_g = st.score_one(d_src, d_dst, 1.0, R, t, 0.04)
        assert np.array_equal(res_g, res_w)      # FP64, same operation order, no FMA: bit-exact
        assert np.array_equal(inl_g, inl_w) and cnt_g == cnt_w


@pytest.mark.parametrize("n,H", [(1000, 1), (5000, 1500), (2049, 1025)])
def test_score_batch_counts_bit_exact(P, O, n, H):
    st = P["stages"]
    pair = P["synth"].make_pair(n, 0.6, 31)
    hyp = _hypotheses(pair, H, 1)
    r = st.consistency_mask(pair["src"], pair["dst"], 0.1, 0, 1)   # only for the packed tiles / centres
    d_hyp = torch.from_numpy(hyp).cuda()
    tau = 0.04
    counts, best, border = st.score_batch(r["f_src"], r["f_dst"], r["d_src"], r["d_dst"], d_hyp, 1.0, tau, r["bound"],
                                          r["centres"], hyp_begin=100)
    torch.cuda.synchronize()
    counts = counts.cpu().numpy()
    want = np.array([O.score(pair["src"], pair["dst"], 1.0, hyp[h, :9].reshape(3, 3, order="F"), hyp[h, 9:], tau)[0]
                     for h in range(H)])
    assert np.array_equal(counts, want)           # inlier counts bit-exact vs the FP64 oracle
    c, hid = st.decode_best(int(best.item()))
    assert c == want.max() and hid == 100 + int(np.argmax(want))   # first best hypothesis wins


def test_errors_are_reported_not_thrown(P):
    capi = P["capi"]
    L = capi.lib()
    rc = L.psulvsb_consistency_mask(None, None, None, None, None, 10, 0.1, 1.0, None, 1, None, None)
    assert rc == capi.ERR_INVALID and b"NULL" in L.psulvsb_last_error()
    h = capi.Handle(0)
    p = capi.default_params(estimate_scaling=1)
    # coincident source points with distinct targets: the length ratio is infinite, which would regrow the
    # reference's histogram mid-stream (registration.cc:714-718) -> reported, not guessed
    src = np.zeros((3, 4))
    dst = np.arange(12, dtype=np.float64).reshape(3, 4)
    with pytest.raises(capi.PsulvsbError) as ei:
        h.solve(p, capi.HostProblem(src, dst))
    assert ei.value.code == capi.ERR_UNSUPPORTED


def test_greedy_clique_on_planted_graphs(P, O):
    """Clique escalation (registration.cc:1000-1085): the oracle's exact branch and bound stands for PMC.  On
    registration-like graphs (one planted clique over a sparse random background) the greedy clique must be a
    clique, maximal, and as large as the exact one."""
    st = P["stages"]
    rng = np.random.default_rng(3)
    for n, k, p_bg in [(40, 8, 0.05), (200, 25, 0.05), (600, 60, 0.03), (50, 1, 0.0)]:
        members = np.sort(rng.permutation(n)[:k])
        A = rng.uniform(0, 1, (n, n)) < p_bg
        A = np.triu(A, 1)
        A[np.ix_(members, members)] = np.triu(np.ones((k, k), dtype=bool), 1)
        ei, ej = np.nonzero(A)
        edges = np.stack([ei, ej], axis=1).astype(np.int32)
        got, size = st.greedy_clique(edges, n)
        assert size == len(got)
        if len(edges):
            got_x, size_x, proven = st.max_clique(edges, n)   # the exact search confirms it
            assert proven and size_x == size and np.array_equal(got_x, got)
            assert np.array_equal(got_x, O.max_clique(n, edges))   # same members as the oracle (canonical clique)
        full = A | A.T
        for a in got:                                    # a clique ...
            for b in got:
                assert a == b or full[a, b]
        if len(got):                                     # ... that is maximal
            common = np.all(full[got], axis=0)
            common[got] = False
            assert not common.any()
        exact = O.max_clique(n, edges) if len(edges) else np.array([], dtype=np.int32)
        if len(edges):
            assert size == len(exact)                    # same size as the exact maximum clique
            if k >= 8:
                assert np.array_equal(got, members)      # and it is the planted one
        else:
            assert size == 0


def _is_clique(edges, n, got):
    full = np.zeros((n, n), dtype=bool)
    full[edges[:, 0], edges[:, 1]] = True
    full |= full.T
    return all(a == b or full[a, b] for a in got for b in got)


@pytest.mark.parametrize("n,p_edge,seed", [(60, 0.15, 1), (300, 0.05, 2), (1000, 0.02, 3), (2500, 0.02, 4),
                                           (400, 0.2, 5), (150, 0.5, 6)])
def test_exact_clique_on_random_graphs(P, O, n, p_edge, seed):
    """No-consensus inlier graphs (what the (1.0, 1.0) round sees when a registration is failing) are sparse random
    graphs where a greedy clique is often one vertex short of the maximum.  The exact improvement search must
    reach the size of the oracle's exact branch and bound (PMC's stand-in) and say so (proven)."""
    st = P["stages"]
    rng = np.random.default_rng(seed)
    A = np.triu(rng.uniform(0, 1, (n, n)) < p_edge, 1)
    ei, ej = np.nonzero(A)
    edges = np.stack([ei, ej], axis=1).astype(np.int32)
    exact = O.max_clique(n, edges)
    got, size, proven = st.max_clique(edges, n)
    assert size == len(got) and _is_clique(edges, n, got)
    assert proven and size == len(exact)
    # members too: both sides return the lexicographically smallest clique of the maximum size
    assert np.array_equal(np.sort(got), np.asarray(exact))
    g_got, g_size = st.greedy_clique(edges, n)
    assert g_size == len(g_got) <= size and _is_clique(edges, n, g_got)
    got2, size2, _ = st.max_clique(edges, n)            # deterministic: same members on a second run
    assert np.array_equal(got, got2) and size2 == size


def test_exact_clique_reports_unproven_on_wide_neighbourhoods(P, O):
    """A dense graph whose neighbourhoods exceed the 512-vertex local matrix: the search declines (proven = 0) and the
    greedy clique stands -- still a valid maximal clique."""
    st = P["stages"]
    rng = np.random.default_rng(9)
    n = 1600
    A = np.triu(rng.uniform(0, 1, (n, n)) < 0.8, 1)
    ei, ej = np.nonzero(A)
    edges = np.stack([ei, ej], axis=1).astype(np.int32)
    got, size, proven = st.max_clique(edges, n)
    assert not proven and size == len(got) >= 10 and _is_clique(edges, n, got)


def test_solver_reaches_the_clique_escalation(P, O):
    """Inputs on which the two-level RANSAC escalates three times (rates (1.0, 1.0), registration.cc:1377-1388)
    and falls back to the inlier-graph clique: the device path must run it (no CPU fallback) and end where the
    oracle (exact clique) ends."""
    capi, synth = P["capi"], P["synth"]
    h = capi.Handle(0)
    kw = dict(noise_bound=0.05, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005, wallclock_cap_s=0.0)
    hits = 0
    for n, ratio, seed in [(100, 0.9, 4), (100, 0.9, 5), (60, 0.9, 2)]:
        pair = synth.make_pair(n, ratio, seed, outliers="fpfh")
        so, _ = O.solve(O.default_params(seed=seed, **kw), pair["src"], pair["dst"])
        sg, _ = h.solve(capi.default_params(seed=seed, **kw), capi.HostProblem(pair["src"], pair["dst"]))
        assert so.escalations == 3
        assert sg.status == 0 and sg.escalations == 3 and bool(sg.valid) == bool(so.valid)
        assert sg.local_iters == so.local_iters and sg.host_rounds == so.host_rounds
        if sg.final_inlier_count == so.final_inlier_count:
            hits += 1
            assert synth.rotation_error(sg.R, O.solution_R(so)) < 1e-5
            assert np.abs(sg.t - O.solution_t(so)).max() < 1e-5
    assert hits >= 2


def test_knn_pca_normals_vs_restatement(P, golden):
    """What the reference driver asks PCL for (PSULVSB.cc:35-85: k = 20 nearest neighbours, smallest-eigenvalue
    eigenvector, flipped towards the origin) on the reference's bunny vertices, against the numpy restatement."""
    import os

    from oracle import prefilter as OP
    from psulvsb_b200 import io

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    v = np.load(os.path.join(root, "tests", "golden", "bunny_res3.npz"))["vertices"].astype(np.float64)
    sub = v[:, :600]
    got = io.estimate_normals(sub, k=20)
    want = OP.knn_pca_normals(sub, k=20)
    assert np.allclose(np.linalg.norm(got, axis=0), 1.0, atol=1e-9)
    cos = np.abs((got * want).sum(axis=0))
    assert (cos > 1 - 1e-6).mean() > 0.995          # same normal up to neighbourhood ties / degenerate planes
    same_side = ((got * want).sum(axis=0) > 0)
    assert same_side[cos > 1 - 1e-6].all()           # and the same orientation (flipped towards the viewpoint)
    # a rigid motion of the cloud rotates the normals' LINES with it (orientation depends on the viewpoint)
    R = np.array([[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0]])
    moved = io.estimate_normals(R @ sub + np.array([[0.3], [0.1], [-0.2]]), k=20)
    assert (np.abs(((R @ got) * moved).sum(axis=0)) > 1 - 1e-5).mean() > 0.97


def test_k1_large_n_sampled_rows_and_invariants(P, O):
    """Size-independent checks at a size the O(N^2) oracle cannot sweep in full: N = 30 000 (4.5e8 pairs).
    (1) 40 random rows bit-exact against the oracle's ScaleInliersSelector on those rows' line vectors;
    (2) popcount(mask) == sum(row_counts) == number of compacted edges; (3) a rigid motion of BOTH clouds
    leaves every pair's lengths unchanged up to rounding, so the mask may differ only on pairs inside the
    counted FP64 band."""
    st = P["stages"]
    n, beta = 30000, 0.1
    pair = P["synth"].make_pair(n, 0.99, 77, side=10.0)
    r = st.consistency_mask(pair["src"], pair["dst"], beta)
    counts = r["row_counts"].cpu().numpy().astype(np.int64)
    rng = np.random.default_rng(1)
    rows = np.sort(rng.permutation(n - 1)[:40])
    m = r["mask"][torch.from_numpy(rows).cuda()].cpu().numpy().view(np.uint32)
    bits = np.unpackbits(m.view(np.uint8), axis=1, bitorder="little")[:, :n]
    for k, i in enumerate(rows):
        js = np.arange(i + 1, n)
        sv = pair["src"][:, js] - pair["src"][:, [i]]
        tv = pair["dst"][:, js] - pair["dst"][:, [i]]
        want = O.scale_inliers(sv, tv, beta)
        assert np.array_equal(bits[k, i + 1:], want), i
        assert not bits[k, : i + 1].any()
        assert counts[i] == int(want.sum())
    edges, offsets = st.compact_edges(r["mask"], r["row_counts"], n, r["stride"])
    assert edges.shape[0] == int(counts.sum())
    e = edges.cpu().numpy()
    assert np.all(e[:, 0] < e[:, 1])
    key = e[:, 0].astype(np.int64) * n + e[:, 1]
    assert np.all(np.diff(key) > 0)                      # reference order: row-major over the upper triangle
    assert r["border"] < 1e-4 * n * (n - 1) / 2
