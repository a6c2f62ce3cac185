"""The unknown-scale stage 1 on the device (csrc/k1_ratio.cu through psulvsb_ratio_reduced_set, the solve's own code)
against the numpy restatement oracle/ratio.py: every pair bin bit for bit, the final MaxScale, the peak bin and
height, and the reduced set in order -- at the shapes where it can go wrong: bins past the shared-memory histogram,
a peak at bin 0 or at the last bin, ties at the maximum height, histogram growth, thousands of pairs above the
initial MaxScale, refusals, the capacity check, batches and a whole scale-1000 solve."""
import ctypes as C

import numpy as np
import pytest

from oracle import ratio as RR
from tests.test_ratio import growth_problem, lattice_problem, pair_index

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def env():
    import psulvsb_b200  # noqa: F401
    from oracle import oracle
    from psulvsb_b200 import capi, stages, synth

    if capi.lib().psulvsb_device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback")
    return {"capi": capi, "stages": stages, "synth": synth, "O": oracle, "h": capi.Handle(0)}


def check(env, src, dst):
    r = RR.reduced_set(src, dst)
    assert r["status"] == RR.OK
    g = env["stages"].ratio_reduced_set(src, dst, pair_bins=True)
    assert np.array_equal(g["pair_bins"], r["pair_bins"])
    assert g["max_scale"] == r["max_scale"]
    assert (g["peak_bin"], g["peak_height"]) == (r["peak_bin"], r["peak_height"])
    assert g["n_edges"] == len(r["edges"]) and np.array_equal(g["edges"], r["edges"])
    return r


def whole_target_scaled(synth, n, outlier_ratio, seed, scale, outliers="gross"):
    """Units that differ: the whole target (outliers included) multiplied by `scale`."""
    p = synth.make_pair(n, outlier_ratio, seed, outliers=outliers)
    return p["src"], np.asfortranarray(p["dst"] * scale)


@pytest.mark.parametrize("scale", [1e-3, 0.03, 0.6, 2.5, 50.0, 102.3, 102.5, 1000.0, 9999.99])
def test_scale_sweep(env, scale):
    """Ratios >= 102.4 fall in bins >= 2048 (global atomics); below ~0.05 the peak is bin 0 (no peak - 1 class);
    9999.99 without noise puts every pair in the last bin (no peak + 1 class)."""
    synth = env["synth"]
    peaks, high_bins = set(), 0
    for n in [2, 3, 4, 33, 257, 1000, 3000]:
        if scale == 9999.99:
            p = synth.make_pair(n, 0.0, n, sigma=0.0, outliers="gross")
            src, dst = p["src"], np.asfortranarray(p["dst"] * scale)
        else:
            src, dst = whole_target_scaled(synth, n, 0.3, n, scale)
        if RR.reduced_set(src, dst)["status"] != RR.OK:  # (n = 3000 at scale 1000: MaxScale would pass 2e6)
            with pytest.raises(env["capi"].PsulvsbError) as e:
                env["stages"].ratio_reduced_set(src, dst)
            assert e.value.code == env["capi"].ERR_UNSUPPORTED and "outgrow" in str(e.value)
            continue
        r = check(env, src, dst)
        peaks.add(r["peak_bin"] - (int(r["max_scale"] * 20) - 1))
        high_bins += int((r["pair_bins"] >= 2048).sum())
    if scale <= 0.03:
        assert peaks == {-199999}                      # peak at bin 0
    if scale == 9999.99:
        assert peaks == {0}                            # peak at the last bin
    if scale >= 2.5:
        assert high_bins > 0


def test_max_height_ties(env):
    """"The first bin to reach the maximum" among tied bins is neither the lowest nor the highest index in general."""
    rng = np.random.default_rng(5)
    middle = 0
    for _ in range(300):
        src, dst = lattice_problem(rng, int(rng.integers(4, 13)))
        r = check(env, src, dst)
        tied = np.flatnonzero(np.bincount(r["pair_bins"]) == r["peak_height"])
        middle += tied.size >= 3 and tied[0] < r["peak_bin"] < tied[-1]
    assert middle >= 3


@pytest.mark.parametrize("positions", [
    [(3, 250)],
    [(0, 1), (17, 18), (400, 999)],
    [(1, 2), (4, 999), (5, 8), (64, 65), (200, 731), (500, 501), (997, 998)],
])
def test_crafted_growth(env, positions):
    """Near-coincident source pairs at chosen pair positions (row starts, row ends, the last rows): 1, 3 and 7 growths
    (7 is the most that stays <= 2e6), plus a ratio between 1e4 and the MaxScale in force that must not grow it."""
    n = 1000
    src, dst = growth_problem(n, positions, seed=len(positions))
    a, b = 150, 600  # pair (150, 600) comes after the first growth: X = 1.5e4 < MaxScale (> 2e4)
    src[:, b] = src[:, a] + np.array([0.0, 0.0, 1e-6])
    dst[:, b] = dst[:, a] + np.array([1.5e4 * 1e-6, 0.0, 0.0])
    r = check(env, src, dst)
    assert [l for l, _ in r["break_points"]] == [pair_index(p, q, n) for p, q in positions]
    assert 1e4 < RR.pair_ratios(src, dst)[pair_index(a, b, n)] < r["break_points"][0][1]


@pytest.mark.parametrize("n,outliers,whole", [(1000, "gross", True), (3000, "fpfh", True), (3000, "gross", False)])
def test_many_growth_candidates(env, n, outliers, whole):
    """Metres against millimetres: far more than 1024 pairs above 1e4, final MaxScale < 2e6."""
    synth = env["synth"]
    p = synth.make_pair(n, 0.5, 7, outliers=outliers)
    dst = p["dst"] * 1000.0
    if not whole:  # only the inliers rescaled
        inl = p["inlier_mask"]
        dst = p["dst"].copy()
        dst[:, inl] = 1000.0 * (p["R"] @ p["src"][:, inl]) + (p["dst"][:, inl] - p["R"] @ p["src"][:, inl])
    dst = np.asfortranarray(dst)
    assert (RR.pair_ratios(p["src"], dst) > 1e4).sum() > 1024
    r = check(env, p["src"], dst)
    assert r["break_points"] and r["max_scale"] < 2e6


def test_refusals(env):
    capi, stages, h = env["capi"], env["stages"], env["h"]
    base = env["synth"].make_pair(50, 0.3, 1)
    params = capi.default_params(estimate_scaling=1, noise_bound=0.05, wallclock_cap_s=0.0)

    def both_refuse(src, dst, words):
        with pytest.raises(capi.PsulvsbError) as e:
            stages.ratio_reduced_set(src, dst)
        with pytest.raises(capi.PsulvsbError) as f:
            h.solve(params, capi.HostProblem(src, dst))
        assert e.value.code == f.value.code == capi.ERR_UNSUPPORTED
        assert words in str(e.value) and str(e.value) == str(f.value)

    src, dst = base["src"].copy(), base["dst"].copy()
    src[:, 30] = src[:, 12]                                 # coincident sources, distinct targets
    both_refuse(src, dst, "infinite length ratio")
    src, dst = growth_problem(50, [(1, 2), (4, 49), (5, 8), (9, 12), (13, 20), (21, 22), (30, 38), (40, 41)])
    assert RR.reduced_set(src, dst)["status"] == RR.SCALE_TOO_LARGE  # the 8th growth passes 2e6
    both_refuse(src, dst, "outgrow the supported MaxScale")
    src, dst = base["src"].copy(), base["dst"].copy()
    src[:, 30], dst[:, 30] = src[:, 12], dst[:, 12]         # a duplicated correspondence: 0 / 0 is NaN, not refused
    r = check(env, src, dst)
    assert r["pair_bins"][pair_index(12, 30, 50)] == 0


def test_capacity(env):
    capi = env["capi"]
    L = capi.lib()
    src, dst = whole_target_scaled(env["synth"], 257, 0.3, 3, 102.3)
    r = RR.reduced_set(src, dst)
    d_src, d_dst = env["stages"].to_device_points(src), env["stages"].to_device_points(dst)
    ne, ms, pk = C.c_ulonglong(0), C.c_double(0.0), (C.c_uint * 2)()
    st = torch.cuda.current_stream().cuda_stream
    capi.check(L.psulvsb_ratio_reduced_set(st, d_src.data_ptr(), d_dst.data_ptr(), 257, None, None, 0, C.byref(ne),
                                           C.byref(ms), pk))
    assert ne.value == len(r["edges"]) and ms.value == r["max_scale"] and pk[1] == r["peak_bin"]
    edges = torch.full((ne.value, 2), -1, dtype=torch.int32, device="cuda")
    ne.value = 0
    rc = L.psulvsb_ratio_reduced_set(st, d_src.data_ptr(), d_dst.data_ptr(), 257, None, edges.data_ptr(),
                                     len(r["edges"]) - 1, C.byref(ne), None, None)
    assert rc == capi.ERR_CAPACITY and ne.value == len(r["edges"])
    assert b"capacity" in L.psulvsb_last_error()
    assert (edges.cpu().numpy() == -1).all()               # nothing written
    capi.check(L.psulvsb_ratio_reduced_set(st, d_src.data_ptr(), d_dst.data_ptr(), 257, None, edges.data_ptr(),
                                           ne.value, C.byref(ne), None, None))
    assert np.array_equal(edges.cpu().numpy(), r["edges"])


def test_batch_equals_individual_solves(env):
    """Each job of an unknown-scale batch has its own MaxScale and histogram offset."""
    capi, synth = env["capi"], env["synth"]
    pairs = [whole_target_scaled(synth, 1000, 0.5, 7, 1000.0), whole_target_scaled(synth, 257, 0.3, 257, 1000.0),
             whole_target_scaled(synth, 400, 0.0, 4, 1000.0), whole_target_scaled(synth, 600, 0.3, 6, 1000.0),
             whole_target_scaled(synth, 120, 0.3, 8, 1000.0)]
    scales = [RR.reduced_set(s, d)["max_scale"] for s, d in pairs]
    assert len(set(scales)) == len(scales) and 10000.0 in scales
    probs = [capi.HostProblem(s, d) for s, d in pairs]
    seeds = [3, 4, 5, 6, 7]
    params = capi.default_params(noise_bound=50.0, score_noise_bound=10.0, inloop_noise_bound=50.0, estimate_scaling=1,
                                 rotation_cost_threshold=0.005, wallclock_cap_s=0.0)
    batch = env["h"].solve_batch(params, probs, seeds)
    for (s, d), prob, seed, b in zip(pairs, probs, seeds, batch):
        params.seed = seed
        one, _ = env["h"].solve(params, prob)
        assert b.status == 0 and one.status == 0
        assert b.n_reduced == one.n_reduced == len(RR.reduced_set(s, d)["edges"])
        assert np.array_equal(np.array(b.rotation[:]), np.array(one.rotation[:]))
        assert np.array_equal(np.array(b.translation[:]), np.array(one.translation[:]))
        assert b.scale == one.scale and b.valid == one.valid
        assert b.final_inlier_count == one.final_inlier_count and b.local_iters == one.local_iters


def test_scale_1000_solve_matches_oracle(env):
    capi, O, synth = env["capi"], env["O"], env["synth"]
    p = synth.make_pair(1000, 0.5, 7, outliers="gross")
    dst = np.asfortranarray(p["dst"] * 1000.0)
    kw = dict(noise_bound=50.0, score_noise_bound=10.0, inloop_noise_bound=50.0, cbar2=1.0, estimate_scaling=1,
              rotation_cost_threshold=0.005, wallclock_cap_s=0.0, seed=7)
    so, to = O.solve(O.default_params(**kw), p["src"], dst)
    sg, tg = env["h"].solve(capi.default_params(**kw), capi.HostProblem(p["src"], dst), trace_cap=4096)
    assert sg.status == 0
    assert sg.n_reduced == so.n_reduced == len(RR.reduced_set(p["src"], dst)["edges"])
    assert len(tg["local"]) == len(to["local"])
    for a, b in zip(tg["local"], to["local"]):
        for f in ["host_round", "n_sampled_lines", "n_sampled_points", "basic_choose", "gnc_iterations", "rot_inliers",
                  "n_rot_points", "similar", "curr_count", "best_count", "local_r"]:
            assert getattr(a, f) == getattr(b, f), (f, a.local_iter, getattr(a, f), getattr(b, f))
        assert abs(a.scale - b.scale) <= 1e-12 * abs(b.scale)
    assert sg.final_inlier_count == so.final_inlier_count
    assert np.array_equal(tg["final_inliers"], to["final_inliers"])
    assert abs(sg.scale - so.scale) <= 1e-12 * abs(so.scale)
    assert synth.rotation_error(sg.R, O.solution_R(so)) < 1e-5
    assert np.abs(sg.t - O.solution_t(so)).max() < 1e-5 * 1000.0
    assert abs(sg.scale - 1000.0) < 0.02 * 1000.0 and synth.rotation_error(sg.R, p["R"]) < 0.05
