"""CPU checks of oracle/score.py, the numpy restatement of stage 4's FP32 fast path and launch shape
(csrc/k4_score.cu) that tests/test_gpu_score_edges.py compares the device with: against a literal per-point loop, the
soundness of the error band against the pinned FP64 oracle over a dynamic-range sweep, and the slice picker on worked
values."""
import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from oracle import oracle as O
from oracle import score as S
from oracle.features import fma32
from psulvsb_b200.stages import centre_and_bound

F = np.float32


def loop_fast(src, dst, hyp_row, scale, tau, centres, bound):
    """score_batch_kernel's prologue and scalar chain for one hypothesis, point by point -> (u list, eps)."""
    cs, cd = centres
    R = [[float(hyp_row[c * 3 + r]) for c in range(3)] for r in range(3)]
    Rf = [[F(scale * R[r][c]) for c in range(3)] for r in range(3)]
    tp = [scale * (R[r][0] * cs[0] + R[r][1] * cs[1] + R[r][2] * cs[2] + float(hyp_row[9 + r])) - cd[r]
          for r in range(3)]
    tf = [F(x) for x in tp]
    G = max(0.0, *[abs(x) for x in tp]) + (1.0 + 1.7320508 * abs(scale)) * float(F(bound * 1.0000002))
    e = (64.0 * S.MU * tau * (G + tau) + 640.0 * ((S.MU * G) * (S.MU * G))) * 1.0001
    eps = F(F(e) + F(1e-37))
    tau2 = F(tau * tau)
    us = []
    for j in range(src.shape[1]):
        p = [F(float(src[c, j]) - cs[c]) for c in range(3)]
        q = [F(float(dst[c, j]) - cd[c]) for c in range(3)]
        d = []
        for r in range(3):
            acc = F(tf[r] - q[r])                  # one rounding: fma(q, -1, tf)
            for c in (2, 1, 0):
                acc = fma32(Rf[r][c], p[c], acc)[()]
            d.append(acc)
        u = fma32(d[0], d[0], -tau2)[()]
        u = fma32(d[1], d[1], u)[()]
        us.append(fma32(d[2], d[2], u)[()])
    return np.array(us, dtype=F), eps


def _hand_cases():
    rng = np.random.default_rng(3)
    src = rng.uniform(-1, 1, (3, 7))
    hyp = np.zeros((2, 12))
    R = S.rotation([1, 2, 3], 0.7)
    hyp[:, :9] = R.ravel(order="F")
    hyp[1, 9:] = [0.01, -0.02, 0.005]
    dst = R @ src + rng.uniform(-0.03, 0.03, (3, 7))
    yield "odd n", src, dst, hyp, 1.0, 0.04
    pts = rng.uniform(-2, 2, (3, 5))
    ident = np.zeros((1, 12))
    ident[0, [0, 4, 8]] = 1.0
    yield "tau = 0, exact-zero residuals", pts, pts.copy(), ident, 1.0, 0.0
    on = np.zeros((3, 3))
    on_dst = np.array([[0.5, 0.0, 0.0], [0.0, 0.5, 0.0], [0.0, 0.0, -0.5]])
    yield "points exactly at tau", on, on_dst, ident, 1.0, 0.5
    yield "negative scale", src, -2.5 * (R @ src) + rng.uniform(-0.03, 0.03, (3, 7)), hyp, -2.5, 0.05


@pytest.mark.parametrize("case", list(range(4)))
def test_restatement_matches_a_scalar_loop(case):
    name, src, dst, hyp, s, tau = list(_hand_cases())[case]
    centres, bound = centre_and_bound(src, dst)
    f = S.fast_path(src, dst, hyp, s, tau, centres, bound)
    for h in range(hyp.shape[0]):
        u, eps = loop_fast(src, dst, hyp[h], s, tau, centres, bound)
        assert np.array_equal(f["u"][h].view(np.uint32), u.view(np.uint32)), name
        assert f["eps"][h] == eps, name
        assert np.array_equal(f["band"][h], ~(np.abs(u) > eps)), name
        assert f["count"][h] == int(np.signbit(u).sum()), name
        # the exact count is the fast count corrected on the band points
        cnt, inl, _ = O.score(src, dst, s, hyp[h, :9].reshape(3, 3, order="F"), hyp[h, 9:], tau)
        fast = np.signbit(u)
        assert np.array_equal(fast[~f["band"][h]], inl.astype(bool)[~f["band"][h]]), name
        assert f["count"][h] + int(inl[f["band"][h]].sum()) - int(fast[f["band"][h]].sum()) == cnt, name
    if name.startswith("tau = 0"):
        # d = p - q = 0 exactly: u = fma(0, 0, -0) = +0, outside the sign test but inside the band
        assert np.all(f["u"] == 0) and not np.signbit(f["u"]).any() and f["band"].all()
    if name.startswith("points exactly"):
        assert np.all(f["u"][0] == 0) and f["band"][0].all()
        assert O.score(src, dst, s, np.eye(3), np.zeros(3), tau)[0] == 3


SWEEP = [(spread, tau, s) for spread in (1.0, 1e3, 1e5, 1e6, 1e7) for tau in (1e-4, 1e-2, 1.0)
         for s in (1e-3, 1.0, 1e3)]


def _unsound_units(spread, tau, s, **band):
    """(h, j) units whose fast sign disagrees with the FP64 oracle while lying outside the band, and G / tau."""
    src, dst, hyp = S.planted_problem(600, spread, tau, s, 7)
    centres, bound = centre_and_bound(src, dst)
    f = S.fast_path(src, dst, hyp, s, tau, centres, bound, **band)
    bad = 0
    for h in range(hyp.shape[0]):
        inl = O.score(src, dst, s, hyp[h, :9].reshape(3, 3, order="F"), hyp[h, 9:], tau)[1].astype(bool)
        bad += int(((np.signbit(f["u"][h]) != inl) & ~f["band"][h]).sum())
    Rf, tf, eps, _ = S.hypothesis_constants(hyp, s, tau, *centres, bound)
    g_over_tau = (np.abs(tf.astype(np.float64)).max() + (1 + 3 ** 0.5 * s) * bound) / tau
    return bad, g_over_tau


@pytest.mark.parametrize("spread,tau,s", SWEEP)
def test_band_is_sound_over_the_dynamic_range(spread, tau, s):
    """Every unit whose FP32 sign is wrong lies inside the band, for G / tau from about 10^2 to 10^17."""
    bad, _ = _unsound_units(spread, tau, s)
    assert bad == 0


def test_band_without_the_quadratic_term_misses_wrong_signs():
    """The sweep has teeth: with eps = 64 mu tau (G + tau) alone (the releases before the (mu G)^2 term), true
    inliers come out of FP32 far outside the band once G / tau reaches a few 10^9, and are counted as outliers."""
    failing = []
    for spread, tau, s in SWEEP:
        bad, g = _unsound_units(spread, tau, s, quadratic=0.0)
        if bad:
            failing.append((spread, tau, s))
            assert g > 1e9
    assert (1e5, 1e-4, 1.0) in failing and (1e6, 1e-4, 1.0) in failing and (1e7, 1e-4, 1e3) in failing
    assert (1e7, 1e-2, 1.0) in failing


def test_band_overflow_sends_every_point_to_fp64():
    """tau^2 beyond FP32 (tau = 1e20), or a band beyond it (coordinates of 1e27): eps = inf, every unit is a band
    unit and the count is the FP64 one."""
    for spread, tau in ((1.0, 1e20), (1e27, 1.0)):
        src, dst, hyp = S.planted_problem(50, spread, tau, 1.0, 2)
        centres, bound = centre_and_bound(src, dst)
        f = S.fast_path(src, dst, hyp, 1.0, tau, centres, bound)
        assert np.isinf(f["eps"]).all() and f["band"].all() and f["border_count"] == 100


def test_slice_picker_on_worked_values():
    # the cfg-D sweep on 148 SMs: 98 tiles in 13 slices of 8 fill 45 waves of 296 CTAs to 0.9994 (25 slices of 4:
    # 87 waves, 0.9941)
    assert S.slices(50000, 1 << 20, 148) == (1024, 13, 4096)
    # fewer than 4 tiles: one slice of all of them
    assert S.slices(1, 1, 148) == (1, 1, 512)
    assert S.slices(1025, 1, 148) == (1, 1, 1536)
    assert S.slices(2047, 4097, 148) == (5, 1, 2048)
    # 9 tiles and one CTA of hypotheses: a single wave, so the most slices win -> 3 slices of 4 tiles, the last
    # holding one point
    assert S.slices(4097, 1, 148) == (1, 3, 2048)
    # the 65 535-slice limit: with slots to spare, more slices always win, down to the limit
    assert S.slices(4 * 65535 * 512, 1, 40000) == (1, 65535, 2048)
    assert S.slices((4 * 65535 + 1) * 512, 1, 40000) == (1, 52429, 2560)
