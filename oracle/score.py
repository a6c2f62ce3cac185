"""numpy restatement of the FP32 fast path of stage 4 (csrc/k4_score.cu, score_batch_kernel) and of its launcher's slice
picker (launch_score_batch).

TEST INFRASTRUCTURE ONLY.  The exact side is the pinned oracle (oracle.oracle.score, FP64 in the reference's order);
this module says what the kernel computes before its FP64 fix-up, operation for operation:
  * the centred float4 tiles: (float)(p - c) per coordinate (common.cuh pack_point);
  * Rf = (float)(s R), tf = (float)(s (R c_src + t) - c_dst), the FP64 values unfused (the library builds with
    -fmad=false, numpy never contracts);
  * d = fma(Rx, px, fma(Ry, py, fma(Rz, pz, tf - q))) per row, tf - q rounded once, then
    u = fma(d2, d2, fma(d1, d1, fma(d0, d0, -tau^2))), all FP32 with one rounding each (features.fma32);
  * the error band eps of DESIGN.md "K4 error band", with the kernel's casts and its 1.0001 and 1e-37f terms.
A point is inside the band when !(|u| > eps); the kernel re-scores exactly those points in FP64 and counts them, so the
border counter is the number of (hypothesis, point) units inside the band, however the points are sliced.
"""
from __future__ import annotations

import numpy as np

from .features import fma32

MU = 5.9604644775390625e-08   # 2^-24
BAND_LINEAR = 64.0            # eps = (BAND_LINEAR mu tau (G + tau) + BAND_QUADRATIC (mu G)^2) * 1.0001 + 1e-37f
BAND_QUADRATIC = 640.0
SB_THREADS, SB_HPT, SB_TP = 256, 4, 512   # threads per CTA, hypotheses per thread, points per tile
FLT_MAX = float(np.finfo(np.float32).max)


def pack(points, centre) -> np.ndarray:
    """3xN FP64 points -> 3xN float32 centred coordinates, as psulvsb_pack_points stores them."""
    p = np.asarray(points, dtype=np.float64)
    c = np.zeros(3) if centre is None else np.asarray(centre, dtype=np.float64)
    return (p - c[:, None]).astype(np.float32)


def hypothesis_constants(hyp, scale, tau, csrc, cdst, coord_bound, quadratic=BAND_QUADRATIC, floor=1e-37):
    """hyp [H, 12] (R column-major, then t) -> (Rf [H, 3, 3] f32, tf [H, 3] f32, eps [H] f32, tau2 f32), as the
    kernel's prologue forms them.  quadratic=0 gives the band of the releases before the (mu G)^2 term (which had no
    overflow rule either); floor is the FP32 term added last."""
    hyp = np.asarray(hyp, dtype=np.float64).reshape(-1, 12)
    s, tau = float(scale), float(tau)
    cs = np.zeros(3) if csrc is None else np.asarray(csrc, dtype=np.float64)
    cd = np.zeros(3) if cdst is None else np.asarray(cdst, dtype=np.float64)
    R = hyp[:, :9].reshape(-1, 3, 3).transpose(0, 2, 1)     # column-major -> [h][r][c]
    with np.errstate(over="ignore", invalid="ignore"):
        Rf = (s * R).astype(np.float32)
        tp = s * (((R[:, :, 0] * cs[0] + R[:, :, 1] * cs[1]) + R[:, :, 2] * cs[2]) + hyp[:, 9:]) - cd
        tf = tp.astype(np.float32)
        tmax = np.abs(tp).max(axis=1)
        cb = float(np.float32(coord_bound * 1.0000002))     # launcher: (float)(coord_bound * 1.0000002)
        G = tmax + (1.0 + 1.7320508 * abs(s)) * cb
        tau2_d = tau * tau
        tau2 = np.float32(tau2_d)
        mg = MU * G
        e = (BAND_LINEAR * MU * tau * (G + tau) + quadratic * (mg * mg)) * 1.0001
        eps = e.astype(np.float32) + np.float32(floor)
        if quadratic:   # tau^2 or eps beyond FP32: every point goes to the FP64 fix-up
            eps = np.where((tau2_d >= FLT_MAX) | ~(e < FLT_MAX), np.float32(np.inf), eps)
    return Rf, tf, eps.astype(np.float32), np.float32(tau2)


def fast_u(P, Q, Rf, tf, tau2) -> np.ndarray:
    """P, Q: 3xN float32 tiles; Rf [H, 3, 3], tf [H, 3] -> u [H, N] float32 of the kernel's FP32 chain."""
    P = np.asarray(P, dtype=np.float32)
    Q = np.asarray(Q, dtype=np.float32)
    d = []
    for r in range(3):
        e = fma32(Q[r][None, :], np.float32(-1.0), tf[:, r][:, None])
        acc = fma32(Rf[:, r, 2][:, None], P[2][None, :], e)
        acc = fma32(Rf[:, r, 1][:, None], P[1][None, :], acc)
        d.append(fma32(Rf[:, r, 0][:, None], P[0][None, :], acc))
    u = fma32(d[0], d[0], -tau2)
    u = fma32(d[1], d[1], u)
    return fma32(d[2], d[2], u)


def fast_path(src, dst, hyp, scale, tau, centres, coord_bound, quadratic=BAND_QUADRATIC, floor=1e-37):
    """-> dict(count [H] fast counts (sign bit of u), u [H, N], band [H, N] = !(|u| > eps), eps [H],
    border_count = number of units inside the band)."""
    cs, cd = (None, None) if centres is None else centres
    P, Q = pack(src, cs), pack(dst, cd)
    Rf, tf, eps, tau2 = hypothesis_constants(hyp, scale, tau, cs, cd, coord_bound, quadratic, floor)
    with np.errstate(over="ignore", invalid="ignore"):
        u = fast_u(P, Q, Rf, tf, tau2)
        band = ~(np.abs(u) > eps[:, None])
    count = np.signbit(u).sum(axis=1).astype(np.int64)
    return {"count": count, "u": u, "band": band, "eps": eps, "border_count": int(band.sum())}


def slices(n: int, n_hyp: int, sm_count: int):
    """launch_score_batch's grid: (gx, gy, chunk_points).  gx = hypothesis groups of SB_THREADS * SB_HPT, gy = point
    slices of chunk_points (a whole number of tiles): slices of >= 4 tiles (fewer only when n has fewer), at most
    65 535 of them, the slice length that fills the last wave of 2 CTAs per SM best (few waves: weighted towards more
    CTAs), ties keep the longer slice."""
    per_cta = SB_THREADS * SB_HPT
    gx = (n_hyp + per_cta - 1) // per_cta
    slots = sm_count * 2
    n_tiles = (n + SB_TP - 1) // SB_TP
    best_tiles, best_eff = n_tiles, -1.0
    t_min = n_tiles if n_tiles < 4 else 4
    for t in range(n_tiles, t_min - 1, -1):
        gy_t = (n_tiles + t - 1) // t
        if gy_t > 65535:
            break
        ctas = gx * gy_t
        waves = (ctas + slots - 1) // slots
        eff = float(ctas) / float(waves * slots)
        if waves < 10:
            eff *= 0.5 + 0.05 * float(waves)
        if eff > best_eff + 1e-9:
            best_eff, best_tiles = eff, t
    chunk = best_tiles * SB_TP
    return gx, (n + chunk - 1) // chunk, chunk


def best_key(counts, hyp_begin: int = 0) -> int:
    """(count << 32) | (0xFFFFFFFF - id) of the first hypothesis with the largest count."""
    counts = np.asarray(counts, dtype=np.int64)
    h = int(np.argmax(counts))
    return (int(counts[h]) << 32) | (0xFFFFFFFF - (hyp_begin + h))


def rotation(axis, angle) -> np.ndarray:
    ax = np.asarray(axis, dtype=np.float64)
    ax = ax / np.linalg.norm(ax)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    return np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * K @ K


def planted_radii(n: int, tau: float, rng, kmax: int = 24) -> np.ndarray:
    """Residuals next to the threshold: tau (1 + 2^-k) and tau (1 - 2^-k) for k = 1..kmax, tau itself and 0, then
    uniform in [0, 3 tau) for the remaining points, in a random order (a random subset of them when n is small)."""
    near = [tau * (1 + 2.0 ** -k) for k in range(1, kmax + 1)] + [tau * (1 - 2.0 ** -k) for k in range(1, kmax + 1)]
    base = np.array(near + [tau, 0.0])
    return rng.permutation(np.concatenate([base, rng.uniform(0, 3 * tau, max(0, n - base.size))]))[:n]


def planted_problem(n: int, spread: float, tau: float, scale: float, seed: int, radii=None):
    """Source points uniform in [-spread, spread]^3, dst = s (R p + t) + r_j (random unit direction) with the planted
    residuals r_j, and two hypotheses: the true (R, t) and the true R with t moved by 0.3 tau / s along x, which moves
    the planted residuals off their values.  -> (src, dst, hyp [2, 12])."""
    rng = np.random.default_rng(seed)
    src = rng.uniform(-spread, spread, (3, n))
    R = rotation(rng.standard_normal(3), rng.uniform(0.3, 3.0))
    t = rng.uniform(-0.4, 0.4, 3) * spread
    dirs = rng.standard_normal((3, n))
    dirs /= np.linalg.norm(dirs, axis=0)
    r = planted_radii(n, tau, rng) if radii is None else np.asarray(radii, dtype=np.float64)
    dst = scale * (R @ src + t[:, None]) + dirs * r
    hyp = np.zeros((2, 12))
    hyp[:, :9] = R.ravel(order="F")
    hyp[0, 9:] = t
    hyp[1, 9:] = t + np.array([0.3 * tau / abs(scale), 0.0, 0.0])
    return src, dst, hyp
