"""Synthetic correspondence generators for the PSULVSB hot path (SURVEY.md section 8d).

Mirrors what the reference's experiment driver does to build its inputs
(examples/teaser_cpp_ply/PSULVSB.cc:256-286 random rigid transform; :190-222 noise + outliers;
:87-188 keep_mask / reduce_map pre-filter, here emulated) with fixed seeds instead of
srand(time(NULL)).  Pure numpy, host side; nothing here runs on the timed path.
"""
from __future__ import annotations

import numpy as np


def random_rigid(rng: np.random.Generator):
    """Random axis, angle U[0, pi), |t| = 3 U[0,1)  (PSULVSB.cc:259-278)."""
    ax = rng.standard_normal(3)
    ax /= np.linalg.norm(ax)
    ang = rng.uniform(0, np.pi)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    R = np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * (K @ K)
    t = rng.standard_normal(3)
    t *= 3.0 * rng.uniform(0, 1) / np.linalg.norm(t)
    return R, t


def make_pair(n: int, outlier_ratio: float, seed: int, *, side: float = 3.0, sigma: float = 0.01,
              outliers: str = "fpfh", src_points: np.ndarray | None = None):
    """One fragment pair: returns dict(src 3xN, dst 3xN, R, t, inlier_mask[N]).

    outliers: "fpfh"  -- dst replaced by a uniform point of the target bounding box (hard case)
              "gross" -- dst += +-U[5,10] per axis (PSULVSB.cc:200-220)
    """
    rng = np.random.default_rng(seed)
    if src_points is None:
        src = rng.uniform(-side / 2, side / 2, (3, n))
    else:
        src = np.array(src_points, dtype=np.float64)
        n = src.shape[1]
    R, t = random_rigid(rng)
    dst = R @ src + t[:, None] + rng.uniform(-sigma, sigma, (3, n))
    n_out = int(n * outlier_ratio)
    out_idx = rng.permutation(n)[:n_out]
    if outliers == "gross":
        mag = rng.uniform(5.0, 10.0, (3, n_out))
        sgn = np.where(rng.uniform(0, 1, (3, n_out)) <= 0.5, -1.0, 1.0)
        dst[:, out_idx] += mag * sgn
    elif outliers == "fpfh":
        lo = dst.min(axis=1, keepdims=True)
        hi = dst.max(axis=1, keepdims=True)
        dst[:, out_idx] = lo + (hi - lo) * rng.uniform(0, 1, (3, n_out))
    else:
        raise ValueError(outliers)
    inl = np.ones(n, dtype=bool)
    inl[out_idx] = False
    return {"src": np.asfortranarray(src), "dst": np.asfortranarray(dst), "R": R, "t": t, "inlier_mask": inl}


def prefilter(pair: dict, seed: int, *, keep_inlier: float = 0.6, keep_outlier: float = 0.3,
              discard_outlier: float = 0.2):
    """Emulated normal-angle histogram pre-filter (PSULVSB.cc:87-188): keep_mask in {-1,0,1},
    reduce_map[M] (original -> reduced column, -1 when absent), reduced src/dst (3xC)."""
    rng = np.random.default_rng(seed ^ 0x5EED)
    inl = pair["inlier_mask"]
    M = inl.size
    u = rng.uniform(0, 1, M)
    keep = np.where(inl, u < keep_inlier, u < keep_outlier)
    mask = np.zeros(M, dtype=np.int32)
    mask[keep] = 1
    far = (~inl) & (~keep) & (rng.uniform(0, 1, M) < discard_outlier)
    mask[far] = -1
    reduce_map = np.full(M, -1, dtype=np.int32)
    idx = np.flatnonzero(mask == 1)
    reduce_map[idx] = np.arange(idx.size, dtype=np.int32)
    return {
        "keep_mask": mask,
        "reduce_map": reduce_map,
        "src_reduce": np.asfortranarray(pair["src"][:, idx]),
        "dst_reduce": np.asfortranarray(pair["dst"][:, idx]),
    }


def rotation_error(Ra: np.ndarray, Rb: np.ndarray) -> float:
    c = (np.trace(Ra.T @ Rb) - 1.0) / 2.0
    return float(abs(np.arccos(np.clip(c, -1.0, 1.0))))


def make_surface(n: int, seed: int) -> np.ndarray:
    """n points (3xn) on the seeded smooth surface z = 0.3 sin(2x) cos(3y) + 0.1 x y over [0, 2]^2: the synthetic
    cloud of the FPFH tests and benchmark (about 20 neighbours within r = 0.08 at n = 5 000)."""
    rng = np.random.default_rng(seed)
    x, y = rng.uniform(0.0, 2.0, n), rng.uniform(0.0, 2.0, n)
    return np.stack([x, y, 0.3 * np.sin(2 * x) * np.cos(3 * y) + 0.1 * x * y])
