"""Numpy restatement of the robust kernels of point-to-plane ICP and generalized ICP (DESIGN.md section 11, "Robust
kernels"; csrc/k9_icp.cu's `robust_weight`, `robust_row_terms`, `whiten_beta` and `whitening`): test infrastructure
only.

The loop, evaluation, correspondences and stop rule are oracle/icp.py's; the unit normals, m = R_k n_s-hat and the 6x6
solve are tests/gicp_restatement.py's.  Given the same transform bits, `p2l_terms` and `gicp_terms` reproduce the
kernel's per-correspondence J^T J and J^T r bit for bit: every product, sum, square root and division is one elementwise
IEEE FP64 operation in the kernel's order.  The sums over the correspondences are in numpy's order, so the systems and
updates agree with the kernel's to the last few bits only.

A loss is (type, k) or an object with `type` and `k` (psulvsb_b200.icp.HuberLoss and the others).
"""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

from oracle import icp as OI
from tests import gicp_restatement as G

L2, HUBER, CAUCHY, GM, TUKEY = range(5)
SQRT2, TWO_SQRT2, INV_SQRT2 = 1.4142135623730951, 2.8284271247461903, 0.7071067811865476


def _tk(loss):
    return (loss[0], float(loss[1])) if isinstance(loss, tuple) else (loss.type, float(loss.k))


def weight(loss, r):
    """rho(r) elementwise, in robust_weight's order (an overflow to inf gives the weight 0, as on the device)."""
    kind, k = _tk(loss)
    r = np.asarray(r, dtype=np.float64)
    with np.errstate(over="ignore"):
        return _weight(kind, k, r)


def _weight(kind, k, r):
    if kind == HUBER:
        return k / np.maximum(np.abs(r), k)
    if kind == CAUCHY:
        q = r / k
        return 1.0 / (1.0 + q * q)
    if kind == GM:
        s = k + r * r
        return k / (s * s)
    if kind == TUKEY:
        t = np.minimum(1.0, np.abs(r) / k)
        u = 1.0 - t * t
        return u * u
    return np.ones_like(r)


def row_terms(p, d, o, loss):
    """One weighted point-to-plane row per column: r = d . o, J = [p' x o, o], u = rho(r) J; (h [21, K] = u_a J_e, upper
    triangle row by row; g [6, K] = u_a r)."""
    r = (d[0] * o[0] + d[1] * o[1]) + d[2] * o[2]
    J = [p[1] * o[2] - p[2] * o[1], p[2] * o[0] - p[0] * o[2], p[0] * o[1] - p[1] * o[0], o[0], o[1], o[2]]
    rho = weight(loss, r)
    u = [rho * J[a] for a in range(6)]
    h = [u[a] * J[e] for a in range(6) for e in range(a, 6)]
    return np.stack(h), np.stack([u[a] * r for a in range(6)])


def p2l_terms(p, q, n, loss):
    """Robust point-to-plane terms of the correspondences (columns of p' = T_k P, q, the target normals n)."""
    d = [p[0] - q[0], p[1] - q[1], p[2] - q[2]]
    return row_terms(p, d, n, loss)


def beta(w, lam):
    """w / ((2 sqrt2 a)(sqrt2 + a)), a = sqrt(2 - w lambda)."""
    a = np.sqrt(2.0 - w * lam)
    return w / ((TWO_SQRT2 * a) * (SQRT2 + a))


def whitening(m, n, w):
    """W = (2 I - w (m m^T + n n^T))^-1/2 in closed form, as (W00, W01, W02, W11, W12, W22) columnwise; a zero column
    of m or n drops that normal."""
    m, n = np.asarray(m, dtype=np.float64), np.asarray(n, dtype=np.float64)
    K = m.shape[1]
    hm, hn = (m != 0.0).any(axis=0), (n != 0.0).any(axis=0)
    both = hm & hn
    neg = ((m[0] * n[0] + m[1] * n[1]) + m[2] * n[2]) < 0.0
    plus, minus = m + n, m - n
    v1 = np.where(both, np.where(neg, minus, plus), np.where(hm, m, n))
    v2 = np.where(both, np.where(neg, plus, minus), 0.0)
    lam1 = ((v1[0] * v1[0] + v1[1] * v1[1]) + v1[2] * v1[2]) * 0.5
    lam2 = ((v2[0] * v2[0] + v2[1] * v2[1]) + v2[2] * v2[2]) * 0.5
    with np.errstate(invalid="ignore", divide="ignore"):
        b1 = np.where(both, beta(w, np.where(both, lam1, 0.0)), np.where(hm | hn, 2.0 * beta(w, np.ones(K)), 0.0))
        b2 = np.where(both, beta(w, np.where(both, lam2, 0.0)), 0.0)
    return tuple(((INV_SQRT2 if i == j else 0.0) + (b1 * v1[i]) * v1[j]) + (b2 * v2[i]) * v2[j]
                 for i, j in ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)))


def gicp_terms(p, q, m, n, w, loss):
    """Robust GICP terms: the rows of W = C^-1/2 as point-to-plane rows of d = p' - q, added in order 0, 1, 2."""
    W00, W01, W02, W11, W12, W22 = whitening(m, n, w)
    d = [p[0] - q[0], p[1] - q[1], p[2] - q[2]]
    h, g = row_terms(p, d, np.stack([W00, W01, W02]), loss)
    for o in (np.stack([W01, W11, W12]), np.stack([W02, W12, W22])):
        hr, gr = row_terms(p, d, o, loss)
        h, g = h + hr, g + gr
    return h, g


def system(Pp, Q, corr, loss, *, normals=None, src_normals=None, tgt_normals=None, R_k=None, epsilon=None):
    """(H upper triangle [21], g [6]) summed over the correspondences of the evaluation at T_k: point-to-plane with the
    target `normals`, or GICP with src_normals, tgt_normals, R_k and epsilon."""
    sel = np.flatnonzero(corr >= 0)
    j = corr[sel]
    if epsilon is None:
        h, g = p2l_terms(Pp[:, sel], Q[:, j], np.asarray(normals, dtype=np.float64)[:, j], loss)
    else:
        m = G.rotate(R_k, G.unit_normals(np.asarray(src_normals, dtype=np.float64)[:, sel]))
        n = G.unit_normals(np.asarray(tgt_normals, dtype=np.float64)[:, j])
        h, g = gicp_terms(Pp[:, sel], Q[:, j], m, n, 1.0 - epsilon, loss)
    return h.sum(axis=1), g.sum(axis=1)


def update(Pp, Q, corr, loss, **objective):
    """(R_u, t_u), or None below the minimum count (6 point-to-plane, 3 GICP) or when solve6 fails."""
    if int((corr >= 0).sum()) < (6 if objective.get("epsilon") is None else 3):
        return None
    x = G.solve6(*system(Pp, Q, corr, loss, **objective))
    return None if x is None else (OI.euler_zyx(x), x[3:].copy())


def step_check(P, Q, d, R_k, t_k, loss, *, normals=None, src_normals=None, tgt_normals=None, epsilon=None, tree=None):
    """What the evaluation of trace record T_k must produce (oracle/icp.py's step_check with the robust update)."""
    Pp = OI.transform(P, R_k, t_k)
    corr, d2 = OI.correspond(Pp, Q, d, normals if epsilon is None else None, tree)
    n, fitness, rmse = OI.evaluate(corr, d2)
    if epsilon is None:
        U = update(Pp, Q, corr, loss, normals=normals)
    else:
        U = update(Pp, Q, corr, loss, src_normals=src_normals, tgt_normals=tgt_normals, R_k=R_k, epsilon=epsilon)
    return {"corr": corr, "d2": d2, "n_corr": n, "fitness": fitness, "inlier_rmse": rmse,
            "next": None if U is None else OI.compose(U, R_k, t_k)}


def icp(P, Q, R0, t0, d, loss, *, normals=None, src_normals=None, tgt_normals=None, epsilon=None, max_iterations=30,
        relative_fitness=1e-6, relative_rmse=1e-6):
    """The free-running loop of oracle/icp.py's icp with the robust update: point-to-plane with the target `normals`,
    or GICP with src_normals, tgt_normals and epsilon."""
    P, Q = np.asarray(P, dtype=np.float64), np.asarray(Q, dtype=np.float64)
    R, t = np.array(R0, dtype=np.float64), np.array(t0, dtype=np.float64)
    out = {"R": R, "t": t, "fitness": 0.0, "inlier_rmse": 0.0, "n_corr": 0, "iterations": 0, "status": OI.NO_UPDATE,
           "corr": np.full(P.shape[1], -1, dtype=np.int64), "trace": [(R, t, 0.0, 0.0, 0)]}
    if P.shape[1] == 0 or Q.shape[1] == 0:
        return out
    keep = np.flatnonzero(OI.candidate_mask(Q, normals if epsilon is None else None))
    tree = cKDTree(Q[:, keep].T) if keep.size else None
    out["trace"] = []
    prev, k = None, 0
    while True:
        s = step_check(P, Q, d, R, t, loss, normals=normals, src_normals=src_normals, tgt_normals=tgt_normals,
                       epsilon=epsilon, tree=tree)
        cur = (s["fitness"], s["inlier_rmse"])
        out.update(R=R, t=t, fitness=cur[0], inlier_rmse=cur[1], n_corr=s["n_corr"], corr=s["corr"], iterations=k)
        out["trace"].append((R, t, cur[0], cur[1], s["n_corr"]))
        status = OI.stop(k, prev, cur, max_iterations, relative_fitness, relative_rmse)
        if status is None and s["next"] is None:
            status = OI.NO_UPDATE
        if status is not None:
            out["status"] = status
            return out
        R, t = s["next"]
        prev, k = cur, k + 1
