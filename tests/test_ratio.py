"""CPU checks of oracle/ratio.py, the numpy restatement of the unknown-scale stage 1 (registration.cc:687-752) that
tests/test_gpu_ratio.py compares the device kernels with: against a literal loop over the pairs, against the pinned
oracle's reduced-set size, and on hand-built edge cases.  Also the argument checks of psulvsb_ratio_reduced_set,
which come before any device work."""
import ctypes as C
import math

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from oracle import oracle as O
from oracle import ratio as RR
from psulvsb_b200 import capi, synth


def loop_reference(src, dst):
    """registration.cc:687-752 pair by pair in Python floats (FP64, no contraction): (bins, MaxScale, peak, edges)."""
    n = src.shape[1]
    max_scale, hsize = 10000, 200000
    hist = {}
    bins, peak, height = [], 0, 0
    for i in range(n - 1):
        for j in range(i + 1, n):
            sv = [float(src[r, j]) - float(src[r, i]) for r in range(3)]
            tv = [float(dst[r, j]) - float(dst[r, i]) for r in range(3)]
            try:
                X = math.sqrt((tv[0] * tv[0] + tv[1] * tv[1]) + tv[2] * tv[2]) / math.sqrt(
                    (sv[0] * sv[0] + sv[1] * sv[1]) + sv[2] * sv[2])
            except ZeroDivisionError:
                X = math.nan if tv == [0.0, 0.0, 0.0] else math.inf
            if X > max_scale:
                max_scale = math.ceil(max_scale + X)
                hsize = max_scale * 20
            f = math.floor(X / max_scale * hsize) if X == X else None
            h = 0 if f is None else f
            if h == hsize:
                h -= 1
            elif h > hsize or h < 0:
                h = 0
            bins.append(h)
            hist[h] = hist.get(h, 0) + 1
            if hist[h] > height:
                height, peak = hist[h], h
    want = [peak] + ([peak - 1] if peak != 0 else []) + ([peak + 1] if peak != hsize - 1 else [])
    pairs = [(i, j) for i in range(n - 1) for j in range(i + 1, n)]
    edges = [pairs[l] for w in want for l in range(len(pairs)) if bins[l] == w]
    return np.array(bins, dtype=np.uint32), float(max_scale), peak, height, np.array(edges, dtype=np.int64).reshape(-1, 2)


def lattice_problem(rng, n):
    """Small integer lattices: a handful of distinct ratios, so bins tie at the maximum height."""
    while True:
        src = rng.integers(0, 3, (3, n)).astype(np.float64)
        if len({tuple(c) for c in src.T}) == n:
            break
    dst = rng.integers(0, 3, (3, n)).astype(np.float64) * rng.choice([0.5, 1.0, 7.0])
    return src, dst


def growth_problem(n, positions, seed=3, factor=1.01):
    """Rigid pair with the point b of each (a, b) in `positions` (all b distinct) moved next to a: their ratio is
    `factor` times the MaxScale then in force, so each one grows the histogram."""
    pair = synth.make_pair(n, 0.3, seed, outliers="gross")
    src, dst = pair["src"].copy(), pair["dst"].copy()
    cur = 10000.0
    for a, b in positions:
        X = cur * factor
        src[:, b] = src[:, a] + np.array([1e-7, 0.0, 0.0])
        dst[:, b] = dst[:, a] + np.array([0.0, X * 1e-7, 0.0])
        cur = math.ceil(cur + X)
    return np.asfortranarray(src), np.asfortranarray(dst)


def pair_index(a, b, n):
    return a * (2 * n - a - 1) // 2 + (b - a - 1)


def assert_matches_loop(src, dst):
    r = RR.reduced_set(src, dst)
    bins, ms, pk, mh, edges = loop_reference(src, dst)
    assert r["status"] == RR.OK
    assert np.array_equal(r["pair_bins"], bins)
    assert r["max_scale"] == ms and r["peak_bin"] == pk and r["peak_height"] == mh
    assert np.array_equal(r["edges"], edges)
    return r


def test_restatement_matches_the_pair_loop_on_lattice_ties():
    rng = np.random.default_rng(11)
    tied_middle = 0
    for _ in range(60):
        n = int(rng.integers(4, 13))
        src, dst = lattice_problem(rng, n)
        r = assert_matches_loop(src, dst)
        hist = np.bincount(r["pair_bins"])
        tied = np.flatnonzero(hist == r["peak_height"])
        tied_middle += tied.size >= 3 and tied[0] < r["peak_bin"] < tied[-1]
    assert tied_middle > 0


@pytest.mark.parametrize("positions", [[(3, 9)], [(2, 5), (6, 7), (11, 39)], [(1, 2), (4, 39), (5, 8), (9, 12),
                                                                               (13, 20), (21, 22), (30, 38)]])
def test_restatement_matches_the_pair_loop_with_growth(positions):
    src, dst = growth_problem(40, positions)
    r = assert_matches_loop(src, dst)
    assert [l for l, _ in r["break_points"]] == [pair_index(a, b, 40) for a, b in positions]


@pytest.mark.parametrize("n,outl,scale,seed", [(60, "gross", 1.0, 1), (150, "fpfh", 0.6, 2), (300, "gross", 1000.0, 3),
                                               (300, "fpfh", 1000.0, 4), (200, "gross", 0.02, 5), (250, "gross", 80.0, 6)])
def test_restatement_size_matches_the_oracle(n, outl, scale, seed):
    pair = synth.make_pair(n, 0.5, seed, outliers=outl)
    dst = np.asfortranarray(pair["dst"] * scale)
    r = RR.reduced_set(pair["src"], dst)
    assert r["status"] == RR.OK
    kw = dict(noise_bound=0.05 * scale, cbar2=1.0, estimate_scaling=1, rotation_cost_threshold=0.005,
              wallclock_cap_s=0.0, seed=seed)
    so, _ = O.solve(O.default_params(**kw), pair["src"], dst)
    assert so.n_reduced == len(r["edges"])
    if scale == 1000.0:
        assert r["break_points"]          # the scale-1000 cases do grow the histogram


def test_restatement_size_matches_the_oracle_with_crafted_growth():
    src, dst = growth_problem(200, [(3, 9), (20, 21), (40, 199), (77, 150)], seed=9)
    r = RR.reduced_set(src, dst)
    assert len(r["break_points"]) == 4
    so, _ = O.solve(O.default_params(noise_bound=0.05, estimate_scaling=1, wallclock_cap_s=0.0, seed=1), src, dst)
    assert so.n_reduced == len(r["edges"])


def test_ratio_of_exactly_max_scale_goes_to_the_last_bin_without_growth():
    src = np.array([[0.0, 1.0], [0.0, 0.0], [0.0, 0.0]])
    dst = np.array([[0.0, 10000.0], [0.0, 0.0], [0.0, 0.0]])
    r = assert_matches_loop(src, dst)
    assert r["break_points"] == [] and r["max_scale"] == 10000.0
    assert r["pair_bins"].tolist() == [199999] and r["peak_bin"] == 199999
    assert r["edges"].tolist() == [[0, 1]]     # no peak + 1 class at the last bin


def test_duplicated_correspondence_goes_to_bin_zero():
    src = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, 0.0], [0.0, 0.0, 2.0]])
    dst = np.array([[5.0, 5.0, 6.0], [1.0, 1.0, 1.0], [0.0, 0.0, 2.0]])   # pair (0, 1): 0 / 0
    r = assert_matches_loop(src, dst)
    assert np.isnan(RR.pair_ratios(src, dst)[0])
    assert r["pair_bins"][0] == 0 and r["break_points"] == []


def test_growing_pair_is_binned_on_the_new_grid():
    src = np.array([[0.0, 1.0, 1.0 + 1e-3], [0.0, 0.0, 0.0], [0.0, 0.0, 0.0]])
    dst = np.array([[0.0, 1.0, 101.0], [0.0, 0.0, 0.0], [0.0, 0.0, 0.0]])  # pair (1, 2): X = 1e5
    r = assert_matches_loop(src, dst)
    X = RR.pair_ratios(src, dst)
    assert r["break_points"] == [(2, math.ceil(10000.0 + X[2]))]
    ms = r["max_scale"]
    assert r["pair_bins"][2] == math.floor(X[2] / ms * (ms * 20))       # new grid; the old one would clamp it to 0
    assert r["pair_bins"][2] != 0


def test_refusals_are_classified():
    src = np.array([[0.0, 1.0, 0.0], [0.0, 0.0, 0.0], [0.0, 0.0, 0.0]])
    dst = np.array([[0.0, 1.0, 3.0], [0.0, 0.0, 0.0], [0.0, 0.0, 0.0]])  # points 0 and 2 coincide, targets differ
    assert RR.reduced_set(src, dst)["status"] == RR.INFINITE_RATIO
    src = np.array([[0.0, 1e-6], [0.0, 0.0], [0.0, 0.0]])
    dst = np.array([[0.0, 3.0], [0.0, 0.0], [0.0, 0.0]])                  # X = 3e6
    assert RR.reduced_set(src, dst)["status"] == RR.SCALE_TOO_LARGE


def test_entry_point_refuses_bad_arguments_before_device_work():
    L = capi.lib()
    ne, ms, pk = C.c_ulonglong(7), C.c_double(0.0), (C.c_uint * 2)()
    buf = (C.c_double * 12)()
    assert L.psulvsb_ratio_reduced_set(None, None, buf, 4, None, None, 0, C.byref(ne), C.byref(ms), pk) == capi.ERR_INVALID
    assert b"psulvsb_ratio_reduced_set" in L.psulvsb_last_error()
    assert L.psulvsb_ratio_reduced_set(None, buf, buf, 1, None, None, 0, C.byref(ne), C.byref(ms), pk) == capi.ERR_INVALID
    assert L.psulvsb_ratio_reduced_set(None, buf, buf, 4, None, None, 0, None, C.byref(ms), pk) == capi.ERR_INVALID
    assert ne.value == 7
