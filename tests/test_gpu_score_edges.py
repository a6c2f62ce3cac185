"""Stage 4 (psulvsb_score_batch, csrc/k4_score.cu) at its edges: every count against the pinned FP64 oracle and the
border counter (units re-scored in FP64) against oracle/score.py's restatement of the FP32 fast path, over the error
band, a dynamic-range sweep, the launch shapes the slice picker produces on this device, the fused argmax, and the
argument and degenerate-input paths."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

KEY_MASK = (1 << 64) - 1


@pytest.fixture(scope="module")
def P():
    import psulvsb_b200  # noqa: F401
    from oracle import oracle, score
    from psulvsb_b200 import capi, stages

    if capi.lib().psulvsb_device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback")
    return {"capi": capi, "st": stages, "O": oracle, "S": score, "L": capi.lib(),
            "sms": torch.cuda.get_device_properties(0).multi_processor_count}


class Problem:
    """Device copies of one problem: FP64 points, the centred float4 tiles, the hypotheses."""

    def __init__(self, P, src, dst, hyp, scale, tau):
        st = P["st"]
        self.P, self.src, self.dst, self.hyp, self.s, self.tau = P, src, dst, np.asarray(hyp, np.float64), scale, tau
        self.n, self.H = src.shape[1], self.hyp.shape[0]
        (self.cs, self.cd), self.bound = st.centre_and_bound(src, dst)
        self.d_src, self.d_dst = st.to_device_points(src), st.to_device_points(dst)
        self.f_src, self.f_dst = st.pack_points(self.d_src, self.cs), st.pack_points(self.d_dst, self.cd)
        self.d_hyp = torch.from_numpy(np.ascontiguousarray(self.hyp)).cuda()

    def call(self, counts, best, border, hyp_begin=0, n=None, n_hyp=None, d_hyp=None, f_src=None, tau=None, s=None,
             stream=None):
        L = self.P["L"]
        ptr = lambda t: None if t is None else (t if isinstance(t, int) else t.data_ptr())  # noqa: E731
        stream = torch.cuda.current_stream().cuda_stream if stream is None else stream
        return L.psulvsb_score_batch(
            stream, ptr(self.f_src if f_src is None else f_src), ptr(self.f_dst), ptr(self.d_src), ptr(self.d_dst),
            self.n if n is None else n, ptr(self.d_hyp if d_hyp is None else d_hyp), self.H if n_hyp is None else n_hyp,
            hyp_begin, self.s if s is None else s, self.tau if tau is None else tau, self.bound,
            (C.c_double * 3)(*self.cs), (C.c_double * 3)(*self.cd), ptr(counts), ptr(best), ptr(border))

    def run(self, hyp_begin=0):
        counts = torch.full((self.H,), -1, dtype=torch.int32, device="cuda")
        best = torch.zeros(1, dtype=torch.int64, device="cuda")
        border = torch.zeros(1, dtype=torch.int64, device="cuda")
        assert self.call(counts, best, border, hyp_begin) == 0, self.P["L"].psulvsb_last_error()
        torch.cuda.synchronize()
        return counts.cpu().numpy().astype(np.int64), int(best.item()) & KEY_MASK, int(border.item())

    def want(self):
        O = self.P["O"]
        counts = np.array([O.score(self.src, self.dst, self.s, self.hyp[h, :9].reshape(3, 3, order="F"),
                                   self.hyp[h, 9:], self.tau)[0] for h in range(self.H)], dtype=np.int64)
        return counts, self.fast()

    def fast(self, block=256):
        """Restatement in blocks of hypotheses -> (border count, band [H, n])."""
        S = self.P["S"]
        bands = [S.fast_path(self.src, self.dst, self.hyp[h:h + block], self.s, self.tau, (self.cs, self.cd),
                             self.bound)["band"] for h in range(0, self.H, block)]
        band = np.concatenate(bands, axis=0)
        return int(band.sum()), band

    def check(self, hyp_begin=0):
        counts, best, border = self.run(hyp_begin)
        want, (want_border, band) = self.want()
        bad = np.flatnonzero(counts != want)
        assert bad.size == 0, f"counts differ at {bad[:8]}: {counts[bad[:8]]} vs {want[bad[:8]]}"
        assert border == want_border
        assert best == self.P["S"].best_key(want, hyp_begin)
        return counts, best, border, band


def hypotheses_around(hyp0, H, tau, scale, seed):
    """H hypotheses: the true one and copies with t moved by up to 2 tau / |s| (counts differ, many points stay next to
    the threshold)."""
    rng = np.random.default_rng(seed)
    hyp = np.repeat(np.asarray(hyp0, np.float64).reshape(1, 12), H, axis=0)
    hyp[1:, 9:] += rng.uniform(-2, 2, (H - 1, 3)) * tau / abs(scale)
    return hyp


# ---------------------------------------------------------------------------------------------------------------------
def test_the_band_is_exercised(P):
    S = P["S"]
    src, dst, hyp = S.planted_problem(3000, 1.0, 0.05, 1.0, 11)
    counts, best, border, band = Problem(P, src, dst, hyp, 1.0, 0.05).check()
    assert border > 0 and border == band.sum()


def test_tau_zero_and_points_exactly_on_tau(P):
    S = P["S"]
    rng = np.random.default_rng(5)
    src = rng.uniform(-2, 2, (3, 1001))
    dst = src.copy()
    dst[:, ::3] += rng.uniform(-1e-3, 1e-3, (3, dst[:, ::3].shape[1]))   # a third are not exact
    ident = np.zeros((3, 12))
    ident[:, [0, 4, 8]] = 1.0
    ident[1, 9] = 2.0 ** -30
    ident[2, :9] = S.rotation([0, 0, 1], 1e-7).ravel(order="F")
    counts, _, border, band = Problem(P, src, dst, ident, 1.0, 0.0).check()
    assert counts[0] == 1001 - dst[:, ::3].shape[1] and band[0].sum() >= counts[0]
    # three points exactly at tau = 0.5 (all values exact in binary)
    on_dst = np.array([[0.5, 0.0, 0.0], [0.0, 0.5, 0.0], [0.0, 0.0, -0.5]])
    counts, _, border, _ = Problem(P, np.zeros((3, 3)), on_dst, ident[:1], 1.0, 0.5).check()
    assert counts[0] == 3 and border == 3


SWEEP = [(spread, tau, s) for spread in (1.0, 1e3, 1e5, 1e6, 1e7) for tau in (1e-4, 1e-2, 1.0)
         for s in (1e-3, 1.0, 1e3)] + [(1e-19, 1e-20, 1.0)]


@pytest.mark.parametrize("spread,tau,s", SWEEP)
def test_dynamic_range_sweep(P, spread, tau, s):
    """G / tau from about 10^2 to 10^17 (and a subnormal u range at spread 1e-19): counts exact, border counter as
    restated."""
    src, dst, hyp = P["S"].planted_problem(2000, spread, tau, s, 7)
    Problem(P, src, dst, hyp, s, tau).check()


def test_band_overflow_rescoring_everything_in_fp64(P):
    """tau^2 beyond FP32, or a band beyond FP32 (coordinates of 1e27): every unit is re-scored in FP64."""
    for spread, tau in ((1.0, 1e20), (1e27, 1.0)):
        src, dst, hyp = P["S"].planted_problem(700, spread, tau, 1.0, 2)
        counts, _, border, _ = Problem(P, src, dst, hyp, 1.0, tau).check()
        assert border == 2 * 700


# ---------------------------------------------------------------------------------------------------------------------
SHAPES = [(1, 1), (2, 1023), (3, 1024), (511, 1025), (512, 4097), (513, 1), (1025, 1023), (2047, 1025), (4097, 1),
          (4097, 1024)]


def test_launch_shapes(P):
    S = P["S"]
    tau = 0.05
    seen = {"gy1": False, "gy2": False, "partial": False, "boundary": False, "odd_alone": False, "gy3": False}
    shapes = list(SHAPES)
    big = next(n for n in (4097, 20001, 50001, 100001) if S.slices(n, 1025, P["sms"])[1] >= 3)
    shapes.append((big, 1025))
    for i, (n, H) in enumerate(shapes):
        gx, gy, chunk = S.slices(n, H, P["sms"])
        rng = np.random.default_rng(100 + i)
        radii = S.planted_radii(n, tau, rng)
        boundary = [j for j in (chunk - 1, chunk) if j < n]
        radii[boundary] = tau * (1 + 2.0 ** -20)           # band points either side of the first slice boundary
        last_lo = chunk * (gy - 1)
        if n - last_lo == 1:                               # the odd last point alone in its slice: on tau exactly
            radii[n - 1] = tau
        src, dst, hyp0 = S.planted_problem(n, 1.0, tau, 1.0, 200 + i, radii=radii)
        hyp = hypotheses_around(hyp0[0], H, tau, 1.0, 300 + i)
        _, _, _, band = Problem(P, src, dst, hyp, 1.0, tau).check(hyp_begin=7 * i)
        seen["gy1"] |= gy == 1
        seen["gy2"] |= gy >= 2
        seen["gy3"] |= gy >= 3 and n == big
        seen["partial"] |= gy >= 2 and n % chunk != 0
        seen["boundary"] |= gy >= 2 and bool(band[:, boundary].any())
        seen["odd_alone"] |= gy >= 2 and n - last_lo == 1 and bool(band[:, n - 1].any())
    assert all(seen.values()), seen


# ---------------------------------------------------------------------------------------------------------------------
def _tied_problem(P, n, H, ids, seed):
    """The true hypothesis at `ids`, a useless one (t 10^3 away) elsewhere: the largest count is tied at `ids`."""
    S = P["S"]
    src, dst, hyp0 = S.planted_problem(n, 1.0, 0.05, 1.0, seed)
    hyp = np.repeat(hyp0[:1], H, axis=0)
    hyp[:, 9:] += 1e3
    hyp[list(ids), 9:] = hyp0[0, 9:]
    return Problem(P, src, dst, hyp, 1.0, 0.05)


@pytest.mark.parametrize("n", [1000, 4097])
def test_argmax_ties_go_to_the_lowest_id(P, n):
    """Ties across lanes (33, 34 -> threads 8), warps, CTAs (1100) and hypothesis groups (2100, 4096); with n = 4097
    the counts come from several slices and the last slice to finish reduces."""
    S = P["S"]
    ids = [4096, 2100, 1100, 300, 70, 34, 33]
    prob = _tied_problem(P, n, 4097, ids, 3)
    counts, best, _, _ = prob.check(hyp_begin=11)
    c, hid = P["st"].decode_best(best)
    assert hid == 11 + 33 and c == counts.max() and np.flatnonzero(counts == c).tolist() == sorted(ids)
    if n == 4097:
        assert S.slices(n, 4097, P["sms"])[1] >= 2


def test_all_counts_zero_gives_the_first_key(P):
    S = P["S"]
    src, dst, hyp0 = S.planted_problem(1500, 1.0, 0.05, 1.0, 4)
    hyp = np.repeat(hyp0[:1], 1500, axis=0)
    hyp[:, 9:] += 1e3
    counts, best, _, _ = Problem(P, src, dst, hyp, 1.0, 0.05).check(hyp_begin=5)
    assert not counts.any() and best == 0xFFFFFFFF - 5


def test_hypothesis_id_range(P):
    capi = P["capi"]
    src, dst, hyp = P["S"].planted_problem(600, 1.0, 0.05, 1.0, 9)
    prob = Problem(P, src, dst, hyp, 1.0, 0.05)
    largest = 0xFFFFFFFF - prob.H
    counts, best, border, _ = prob.check(hyp_begin=largest)      # ids up to 0xFFFFFFFE
    buf = torch.zeros(prob.H, dtype=torch.int32, device="cuda")
    for hb in (largest + 1, (1 << 64) - 1, (1 << 64) - prob.H):
        assert prob.call(buf, None, None, hyp_begin=hb) == capi.ERR_UNSUPPORTED, hex(hb)
    assert prob.call(buf, None, None, n_hyp=1 << 32) == capi.ERR_UNSUPPORTED


def test_halves_into_one_best_equal_the_whole(P):
    S = P["S"]
    src, dst, hyp0 = S.planted_problem(4097, 1.0, 0.05, 1.0, 12)
    hyp = hypotheses_around(hyp0[0], 3000, 0.05, 1.0, 13)
    prob = Problem(P, src, dst, hyp, 1.0, 0.05)
    counts, best, border = prob.run(hyp_begin=40)
    d_best = torch.zeros(1, dtype=torch.int64, device="cuda")
    d_border = torch.zeros(1, dtype=torch.int64, device="cuda")
    parts = []
    for lo, hi in ((0, 1700), (1700, 3000)):
        c = torch.zeros(hi - lo, dtype=torch.int32, device="cuda")
        assert prob.call(c, d_best, d_border, hyp_begin=40 + lo, n_hyp=hi - lo, d_hyp=prob.d_hyp[lo:hi]) == 0
        parts.append(c)
    torch.cuda.synchronize()
    assert np.array_equal(torch.cat(parts).cpu().numpy(), counts)
    assert int(d_best.item()) & KEY_MASK == best and int(d_border.item()) == border
    # no best / no border counter: the same counts
    c = torch.zeros(3000, dtype=torch.int32, device="cuda")
    assert prob.call(c, None, None, hyp_begin=40) == 0
    torch.cuda.synchronize()
    assert np.array_equal(c.cpu().numpy(), counts)


# ---------------------------------------------------------------------------------------------------------------------
def test_no_points_zeroes_the_counts_and_writes_the_first_key(P):
    capi = P["capi"]
    src, dst, hyp = P["S"].planted_problem(10, 1.0, 0.05, 1.0, 1)
    prob = Problem(P, src, dst, np.repeat(hyp, 700, axis=0), 1.0, 0.05)
    counts = torch.full((prob.H,), -559038737, dtype=torch.int32, device="cuda")   # 0xDEADBEEF
    best = torch.zeros(1, dtype=torch.int64, device="cuda")
    border = torch.full((1,), 77, dtype=torch.int64, device="cuda")
    assert prob.call(counts, best, border, hyp_begin=9, n=0) == 0
    torch.cuda.synchronize()
    assert not counts.cpu().numpy().any()
    assert int(best.item()) == 0xFFFFFFFF - 9 and int(border.item()) == 77
    assert prob.call(counts, best, border, n=-1) == capi.ERR_INVALID


def test_no_hypotheses_writes_nothing(P):
    src, dst, hyp = P["S"].planted_problem(100, 1.0, 0.05, 1.0, 1)
    prob = Problem(P, src, dst, hyp, 1.0, 0.05)
    counts = torch.full((4,), 1234, dtype=torch.int32, device="cuda")
    best = torch.full((1,), 5678, dtype=torch.int64, device="cuda")
    border = torch.full((1,), 91, dtype=torch.int64, device="cuda")
    assert prob.call(counts, best, border, n_hyp=0) == 0
    torch.cuda.synchronize()
    assert counts.cpu().tolist() == [1234] * 4 and int(best.item()) == 5678 and int(border.item()) == 91


def test_bad_arguments_are_refused(P):
    capi = P["capi"]
    src, dst, hyp = P["S"].planted_problem(100, 1.0, 0.05, 1.0, 1)
    prob = Problem(P, src, dst, hyp, 1.0, 0.05)
    counts = torch.zeros(2, dtype=torch.int32, device="cuda")
    assert prob.call(counts, None, None, f_src=prob.f_src.data_ptr() + 4) == capi.ERR_INVALID
    assert prob.call(counts, None, None, tau=float("nan")) == capi.ERR_INVALID
    assert prob.call(counts, None, None, s=float("nan")) == capi.ERR_INVALID
    assert prob.call(counts, None, None, tau=-1.0) == capi.ERR_INVALID


def test_repeated_calls_on_a_side_stream(P):
    S = P["S"]
    src, dst, hyp0 = S.planted_problem(5001, 1.0, 0.05, 1.0, 21)
    prob = Problem(P, src, dst, hypotheses_around(hyp0[0], 2500, 0.05, 1.0, 22), 1.0, 0.05)
    counts, best, border, _ = prob.check()
    side = torch.cuda.Stream()
    for rep in range(3):
        c = torch.full((prob.H,), 0x5A5A5A5A + rep, dtype=torch.int32, device="cuda")
        b = torch.zeros(1, dtype=torch.int64, device="cuda")
        bo = torch.zeros(1, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            assert prob.call(c, b, bo, stream=side.cuda_stream) == 0
        side.synchronize()
        assert np.array_equal(c.cpu().numpy(), counts)
        assert int(b.item()) & KEY_MASK == best and int(bo.item()) == border
