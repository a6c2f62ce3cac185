"""numpy restatement of the unknown-scale stage 1 (registration.cc:687-752): the length-ratio histogram, its growth
in the middle of the pair loop, the "first bin to reach the maximum height" and the three-bin reduced set.

TEST INFRASTRUCTURE ONLY.  Every value is FP64 in the reference's operation order and numpy never contracts a
multiply-add, so the bin of every pair agrees bit for bit with the device kernels (csrc/k1_ratio.cu, built with
-fmad=false) and with the pinned oracle (oracle/psulvsb_oracle.cpp).
"""
from __future__ import annotations

import numpy as np

MAX_SCALE0 = 10000.0       # registration.cc:688
BIN_SIZE = 20.0            # registration.cc:687
SUPPORTED_MAX_SCALE = 2e6  # the library refuses a larger final MaxScale (a 40 M-bin histogram)

OK, INFINITE_RATIO, SCALE_TOO_LARGE = 0, 1, 3


def pair_ratios(src, dst) -> np.ndarray:
    """X_l = |t_j - t_i| / |s_j - s_i| of every pair i < j, row-major (the reference's l order)."""
    s = np.asarray(src, dtype=np.float64)
    t = np.asarray(dst, dtype=np.float64)
    i, j = np.triu_indices(s.shape[1], 1)
    sv = s[:, j] - s[:, i]
    tv = t[:, j] - t[:, i]
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.sqrt((tv[0] * tv[0] + tv[1] * tv[1]) + tv[2] * tv[2]) / np.sqrt(
            (sv[0] * sv[0] + sv[1] * sv[1]) + sv[2] * sv[2])


def growth(X: np.ndarray):
    """registration.cc:714-718 replayed in pair order -> (break points [(l, MaxScale from pair l on)], final MaxScale).

    A pair can only grow the histogram if its ratio exceeds every earlier one (MaxScale is always >= every ratio
    binned so far), so only those running-maximum records are walked."""
    if X.size == 0:
        return [], MAX_SCALE0
    Xn = np.where(np.isnan(X), -np.inf, X)  # a NaN ratio (0 / 0) never grows anything
    prev = np.concatenate(([-np.inf], np.maximum.accumulate(Xn)[:-1]))
    cand = np.flatnonzero((Xn > prev) & (Xn > MAX_SCALE0))
    cur, bps = MAX_SCALE0, []
    for l in cand:
        x = float(X[l])
        if x > cur:
            cur = float(np.ceil(cur + x))  # MaxScale = ceil(MaxScale + X)
            bps.append((int(l), cur))
    return bps, cur


def bins(X: np.ndarray, bps) -> np.ndarray:
    """registration.cc:697-723: bin of every pair on the grid in force when it is binned (growth happens before)."""
    scale = np.full(X.shape, MAX_SCALE0)
    for l, ms in bps:
        scale[l:] = ms
    hsize = scale * BIN_SIZE                        # H.size() == MaxScale * binsize, exact
    with np.errstate(invalid="ignore", over="ignore"):
        f = np.floor((X / scale) * hsize)
    h = np.where(np.isfinite(f), f, 0.0)            # NaN (0 / 0): the reference files it under bin 0
    h = np.where(h == hsize, hsize - 1, h)          # X == MaxScale: the last bin
    h = np.where((h > hsize) | (h < 0), 0.0, h)
    return h.astype(np.uint32)


def peak(b: np.ndarray, hsize: int):
    """The first bin to reach the running maximum height (strict '>' at registration.cc:725) -> (bin, height).
    Among the bins at the final maximum height that is the one whose last member comes first in pair order."""
    hist = np.bincount(b, minlength=hsize)
    mh = int(hist.max())
    tied = np.flatnonzero(hist == mh)
    last = np.array([np.flatnonzero(b == k)[-1] for k in tied])
    return int(tied[np.argmin(last)]), mh


def reduced_set(src, dst) -> dict:
    """The whole stage -> dict(status, pair_bins, break_points, max_scale, peak_bin, peak_height, edges [K, 2]).
    status INFINITE_RATIO / SCALE_TOO_LARGE: what the library refuses (the reference is undefined there / the
    histogram is too large); the other fields are then absent."""
    X = pair_ratios(src, dst)
    if np.isinf(X).any():
        return {"status": INFINITE_RATIO}
    bps, ms = growth(X)
    if ms > SUPPORTED_MAX_SCALE:
        return {"status": SCALE_TOO_LARGE, "max_scale": ms, "break_points": bps}
    hsize = int(ms * BIN_SIZE)
    b = bins(X, bps)
    pk, mh = peak(b, hsize)
    n = np.asarray(src).shape[1]
    i, j = np.triu_indices(n, 1)
    want = [pk] + ([pk - 1] if pk != 0 else []) + ([pk + 1] if pk != hsize - 1 else [])
    sel = np.concatenate([np.flatnonzero(b == w) for w in want])
    return {"status": OK, "pair_bins": b, "break_points": bps, "max_scale": ms, "peak_bin": pk, "peak_height": mh,
            "edges": np.stack([i[sel], j[sel]], axis=1).astype(np.int64)}
