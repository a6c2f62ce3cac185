"""The sampler's on-chip pass (csrc/k2_sampler.cu): one CTA per job walks the draw window in draw order against a
shared-memory bitmap of the values accepted so far.  It must give the rejection sampler's index sequence and stream
position bit for bit, like the bucket passes it replaces for n <= 2^20 and windows <= 2^20 draws: at the budget and one
above it, at chunk (4096-draw) boundaries, under heavy in-chunk duplication and its overflow walk, at cfg-A's L
sample rates, and when the draw budget runs out.  A batch with escalated windows next to normal ones (the escalation's
long window stays with the bucket passes in the same launch) must solve as each registration does alone."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

CHUNK = 4096  # draws per chunk of the on-chip walk
BUDGET = 1 << 20  # largest n (and window) it takes


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


def check(P, O, seed, dom, ev, n, count):
    got, consumed = P["stages"].sample(seed, dom, ev, n, count)
    want, want_consumed = O.sample_without_replacement(seed, dom, ev, n, count)
    assert np.array_equal(got, want), (n, count)
    assert consumed == want_consumed, (n, count, consumed, want_consumed)
    return consumed


@pytest.mark.parametrize("n", [BUDGET, BUDGET + 1])
def test_at_the_budget_and_one_above(P, O, n):
    for count in [n // 10, n // 2]:
        check(P, O, 3, 1, 5, n, count)


def test_counts_ending_on_a_chunk_boundary_and_one_past(P, O):
    """The count-th accepted draw is the last draw of a chunk; then one more accepted draw needs the next chunk."""
    n, seed, dom, ev = 900_000, 11, 1, 2
    for chunks in [1, 3]:
        hit = None
        for count in range(chunks * CHUNK, chunks * CHUNK - 400, -1):  # (~chunks^2 * 9 repeats among the draws)
            if O.sample_without_replacement(seed, dom, ev, n, count)[1] == chunks * CHUNK:
                hit = count
                break
        assert hit is not None
        assert check(P, O, seed, dom, ev, n, hit) == chunks * CHUNK
        assert check(P, O, seed, dom, ev, n, hit + 1) > chunks * CHUNK


@pytest.mark.parametrize("n", [1, 2, 10, 1000, CHUNK, 5000])
def test_heavy_in_chunk_duplication(P, O, n):
    """count = n with n <= a few chunks: most draws repeat a value of their own chunk, the duplicate table overflows."""
    for seed in [1, 77]:
        check(P, O, seed, 2, 9, n, n)


@pytest.mark.parametrize("n,count", [(5000, 4000), (627_562, 62_756), (65_536, 20_000), (20_000, 20_000)])
def test_list_overflow_walk(P, O, n, count):
    """A duplicate table of one loser: every chunk with two in-chunk duplicates takes the one-warp walk."""
    P["capi"].debug_set("sample_list_cap_test", 1)
    try:
        check(P, O, 5, 1, 1, n, count)
    finally:
        P["capi"].debug_set("reset", 0)


def test_bucket_list_overflow_above_the_budget(P, O):
    """Above the on-chip budget the bucket passes and their list-overflow walk are unchanged."""
    P["capi"].debug_set("sample_list_cap_test", 100)
    try:
        check(P, O, 7, 1, 3, 2_070_000, 621_000)
    finally:
        P["capi"].debug_set("reset", 0)


@pytest.mark.parametrize("rate", [0.1, 0.2, 0.5, 1.0])
def test_cfg_a_l_sample(P, O, rate):
    """cfg-A's L sample (~687 000 reduced edges); rate 1.0 is the escalation's window, drawn by the bucket passes."""
    n = 687_000
    check(P, O, 0x5EED, 1, 4, n, int(n * rate))


@pytest.mark.parametrize("n,count,max_draws", [(1000, 1000, 1200), (100_000, 50_000, 60_000), (700_000, 70_000, 70_000)])
def test_budget_exhaustion_reports_failure(P, n, count, max_draws):
    _, consumed = P["stages"].sample(9, 1, 0, n, count, max_draws=max_draws)
    assert consumed == 0


def test_batch_with_escalations_matches_lone_solves(P):
    """Registrations that escalate to the (1.0, 1.0) rate pair (their samples go to the bucket passes) next to ones that
    do not, in one chunk: each must come out as it does alone.  (A lone registration may get another GNC-TLS launch
    shape than the chunk, which reorders FP64 sums: the poses agree to 1e-12, everything counted agrees exactly.)"""
    capi, synth = P["capi"], P["synth"]
    kw = dict(noise_bound=0.05, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005, wallclock_cap_s=0.0)
    pairs = [synth.make_pair(2000, 0.95, 61), synth.make_pair(1000, 0.99, 71, outliers="gross"),
             synth.make_pair(3000, 0.9, 63), synth.make_pair(1500, 0.995, 73)]
    probs = [capi.HostProblem(p["src"], p["dst"]) for p in pairs]
    h = capi.Handle(0)
    batch = h.solve_batch(capi.default_params(seed=7, **kw), probs, seeds=[7, 8, 9, 10])
    escalations = 0
    for k, prob in enumerate(probs):
        alone, _ = h.solve(capi.default_params(seed=7 + k, **kw), prob)
        for f in ["status", "valid", "n_line_vectors", "n_reduced", "final_inlier_count", "host_rounds", "local_iters",
                  "final_C", "escalations", "refined"]:
            assert getattr(batch[k], f) == getattr(alone, f), (k, f, getattr(batch[k], f), getattr(alone, f))
        assert np.abs(batch[k].R - alone.R).max() < 1e-12 and np.abs(batch[k].t - alone.t).max() < 1e-12
        escalations += alone.escalations
    assert escalations > 0
