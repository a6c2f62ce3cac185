"""4-byte against 8-byte reduced-set edges (csrc/edge_fmt.cuh): the engine picks 4-byte edges for a chunk whose working
sets all have at most 65 536 points.  The "edge_wide" switch forces 8-byte edges; every solve here must come out the
same both ways, step by step: the reduced-set size, the number of sampled points (the endpoint flags of the L sample),
the control flow, inlier sets and poses.  The sizes straddle the limit: C = 65 536 (4-byte), C = 65 537 (8-byte), a
self-update working set that outgrows it while C does not, and a chunk that mixes sizes (8-byte for all of it)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

PKW = dict(noise_bound=0.05, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005, wallclock_cap_s=0.0)


@pytest.fixture(scope="module")
def env():
    import psulvsb_b200  # noqa: F401
    from psulvsb_b200 import capi, synth

    if capi.lib().psulvsb_device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback")
    return {"capi": capi, "synth": synth, "h": capi.Handle(0)}


def problem(env, pair, pre=None):
    capi = env["capi"]
    if pre is None:
        return capi.HostProblem(pair["src"], pair["dst"])
    return capi.HostProblem(pre["src_reduce"], pre["dst_reduce"], pair["src"], pair["dst"], pre["keep_mask"],
                            pre["reduce_map"])


def solve(env, prob, seed, wide, **kw):
    capi = env["capi"]
    args = dict(PKW)
    args.update(kw)
    capi.debug_set("edge_wide", 1 if wide else 0)
    try:
        return env["h"].solve(capi.default_params(seed=seed, **args), prob, trace_cap=4096)
    finally:
        capi.debug_set("reset", 0)


def same_solution(a, b):
    for f in ["status", "valid", "n_line_vectors", "n_reduced", "final_inlier_count", "host_rounds", "local_iters",
              "final_C", "escalations", "refined"]:
        assert getattr(a, f) == getattr(b, f), (f, getattr(a, f), getattr(b, f))
    assert np.array_equal(a.R, b.R) and np.array_equal(a.t, b.t) and a.scale == b.scale


def same_run(sa, ta, sb, tb):
    same_solution(sa, sb)
    assert len(ta["local"]) == len(tb["local"]) and len(ta["host"]) == len(tb["host"])
    for a, b in zip(ta["local"], tb["local"]):
        for f in ["host_round", "local_iter", "n_sampled_lines", "n_sampled_points", "basic_choose", "gnc_iterations",
                  "rot_inliers", "n_rot_points", "similar", "curr_count", "best_count", "local_r"]:
            assert getattr(a, f) == getattr(b, f), (f, a.local_iter, getattr(a, f), getattr(b, f))
        assert list(a.R) == list(b.R) and list(a.t) == list(b.t)
    for a, b in zip(ta["host"], tb["host"]):
        for f in ["host_round", "curr_count", "best_host", "new_corr_count", "inlier_map_size", "host_r"]:
            assert getattr(a, f) == getattr(b, f), (f, getattr(a, f), getattr(b, f))
    assert np.array_equal(ta["final_inliers"], tb["final_inliers"])
    assert np.array_equal(ta["inlier_counter"], tb["inlier_counter"])


@pytest.mark.parametrize("n", [65536, 65537])
def test_narrow_and_wide_edges_agree_at_the_limit(env, n):
    pair = env["synth"].make_pair(n, 0.99, 4243, side=20.0)
    prob = problem(env, pair)
    sn, tn = solve(env, prob, 31, wide=False)
    sw, tw = solve(env, prob, 31, wide=True)
    assert sn.status == 0 and sn.n_reduced > 0
    same_run(sn, tn, sw, tw)
    assert sum(1 for a in tn["local"] if a.n_sampled_points > 0) > 0


@pytest.mark.parametrize("n,ratio,seed", [(3000, 0.9, 13), (80000, 0.99, 17)])
def test_self_update_agrees(env, n, ratio, seed):
    """3000: a 4-byte list that the self-update appends to; 80 000: C0 ~ 24 000 but the working set may grow to
    ~ 69 000 points, past the 16-bit indices, so the list is 8-byte although C fits."""
    synth = env["synth"]
    pair = synth.make_pair(n, ratio, seed, side=20.0 if n > 10000 else 1.0)
    pre = synth.prefilter(pair, seed)
    ccap = int((pre["keep_mask"] == 1).sum() + (pre["keep_mask"] == 0).sum())
    assert (ccap > 65536) == (n > 10000) and pre["src_reduce"].shape[1] < 65536
    prob = problem(env, pair, pre)
    sn, tn = solve(env, prob, seed, wide=False)
    sw, tw = solve(env, prob, seed, wide=True)
    assert sn.status == 0
    same_run(sn, tn, sw, tw)
    assert sum(a.new_corr_count for a in tn["host"]) > 0


def test_unknown_scale_agrees(env):
    synth = env["synth"]
    pair = synth.make_pair(1500, 0.9, 5)
    pair["dst"] = np.asfortranarray(pair["dst"] * 1.7)
    prob = problem(env, pair)
    sn, tn = solve(env, prob, 5, wide=False, estimate_scaling=1)
    sw, tw = solve(env, prob, 5, wide=True, estimate_scaling=1)
    assert sn.status == 0
    same_run(sn, tn, sw, tw)


def test_mixed_chunk_matches_individual_solves(env):
    """A chunk with one working set above 65 536 points takes 8-byte edges for all its registrations; the small ones
    must come out as they do alone (4-byte).  (A lone registration may get another GNC-TLS launch shape than the
    chunk, which reorders FP64 sums: the poses agree to 1e-12, everything counted agrees exactly.)"""
    capi, synth = env["capi"], env["synth"]
    pairs = [synth.make_pair(2000, 0.95, 61), synth.make_pair(65537, 0.99, 62, side=20.0), synth.make_pair(3000, 0.9, 63)]
    probs = [problem(env, p) for p in pairs]
    params = capi.default_params(seed=7, **PKW)
    batch = env["h"].solve_batch(params, probs, seeds=[7, 8, 9])
    for k, prob in enumerate(probs):
        alone, _ = env["h"].solve(capi.default_params(seed=7 + k, **PKW), prob)
        for f in ["status", "valid", "n_line_vectors", "n_reduced", "final_inlier_count", "host_rounds", "local_iters",
                  "final_C", "escalations", "refined"]:
            assert getattr(batch[k], f) == getattr(alone, f), (k, f, getattr(batch[k], f), getattr(alone, f))
        assert np.abs(batch[k].R - alone.R).max() < 1e-12 and np.abs(batch[k].t - alone.t).max() < 1e-12
