"""Numpy restatement of colored ICP (DESIGN.md section 11, "Colored ICP"; csrc/k8_features.cu's k8_color_gradients
and csrc/k9_icp.cu's `colored_terms`): test infrastructure only.

The loop, evaluation, correspondences and stop rule are oracle/icp.py's (point-to-plane: a target with a non-finite
normal is no candidate); the weights are tests/robust_icp_restatement.py's and the 6x6 solve tests/gicp_restatement.py's.
Given the same transform bits and the same gradients, `terms` reproduces the kernel's per-correspondence J^T J and
J^T r bit for bit: every product, sum, square root and division is one elementwise IEEE FP64 operation in the kernel's
order.  The sums over the correspondences, and the gradient stage's sums over a neighbourhood, run in numpy's order, so
the systems, updates and gradients agree with the kernel's to the last few bits only.

The gradient stage keeps the hybrid neighbourhood of tests/normals_restatement.py (FP32 keys on FPFH's grid).  A loss is
None (L2), (type, k) or an object with `type` and `k`.
"""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

from oracle import icp as OI
from tests import gicp_restatement as G
from tests import normals_restatement as NR
from tests import robust_icp_restatement as RR

MAX_NN = 30            # Open3D's KDTreeSearchParamHybrid(2 d, 30)


def intensity(colors):
    """((r + g) + b) / 3 per column."""
    c = np.asarray(colors, dtype=np.float64)
    return ((c[0] + c[1]) + c[2]) / 3.0


def solve3(A, b):
    """k8_features.cu's solve3, elementwise: (g [3, K], ok [K]); g is meaningful where ok."""
    A00, A01, A02, A11, A12, A22 = A
    with np.errstate(all="ignore"):
        ok = A00 > 0.0
        L00 = np.sqrt(A00)
        L10, L20 = A01 / L00, A02 / L00
        d1 = A11 - L10 * L10
        ok &= d1 > 0.0
        L11 = np.sqrt(d1)
        L21 = (A12 - L20 * L10) / L11
        d2 = (A22 - L20 * L20) - L21 * L21
        ok &= d2 > 0.0
        L22 = np.sqrt(d2)
        y0 = b[0] / L00
        y1 = (b[1] - L10 * y0) / L11
        y2 = ((b[2] - L20 * y0) - L21 * y1) / L22
        g2 = y2 / L22
        g1 = (y1 - L21 * g2) / L11
        g0 = ((y0 - L10 * g1) - L20 * g2) / L00
    g = np.stack([g0, g1, g2])
    return g, ok & np.isfinite(g).all(axis=0)


def gradients(points, colors, normals, radius, max_nn=MAX_NN):
    """(G [3, n], fragile [n]): the colour gradient of every point.  Point i's hybrid neighbourhood keeps nn points (i
    included); with nn >= 4 and a finite normal n, each kept j != i gives the row a = (q_j - ((q_j - q_i).n) n) - q_i,
    b = I_j - I_i, the row (nn - 1) n has b = 0, and A^T A g = A^T b is solved by solve3; else, or when it fails, 0.
    fragile: the hybrid selection's flags (normals_restatement.hybrid_neighbours)."""
    P = np.asarray(points, dtype=np.float64)
    N = np.asarray(normals, dtype=np.float64)
    n = P.shape[1]
    ii, jj, _, frag = NR.hybrid_neighbours(P, radius, max_nn)
    nn = np.bincount(ii, minlength=n)
    I = intensity(colors)
    sel = jj != ii
    i, j = ii[sel], jj[sel]
    Ni, Qi, Qj = N[:, i], P[:, i], P[:, j]
    s = ((Qj[0] - Qi[0]) * Ni[0] + (Qj[1] - Qi[1]) * Ni[1]) + (Qj[2] - Qi[2]) * Ni[2]
    a = [(Qj[r] - s * Ni[r]) - Qi[r] for r in range(3)]
    b = I[j] - I[i]
    pairs = [(r, c) for r in range(3) for c in range(r, 3)]
    A = [np.bincount(i, weights=a[r] * a[c], minlength=n) for r, c in pairs]
    bv = [np.bincount(i, weights=a[r] * b, minlength=n) for r in range(3)]
    w = (nn - 1).astype(np.float64)
    c = [w * N[r] for r in range(3)]
    A = [A[e] + c[r] * c[cc] for e, (r, cc) in enumerate(pairs)]
    g, ok = solve3(A, bv)
    ok &= (nn >= 4) & np.isfinite(N).all(axis=0)
    return np.where(ok, g, 0.0), frag


def _loss(loss):
    return (RR.L2, 1.0) if loss is None else loss


def _scaled_row(p, o, s):
    """J = s [p' x o, o]."""
    return [s * (p[1] * o[2] - p[2] * o[1]), s * (p[2] * o[0] - p[0] * o[2]), s * (p[0] * o[1] - p[1] * o[0]),
            s * o[0], s * o[1], s * o[2]]


def _row(J, r, loss):
    rho = RR.weight(_loss(loss), r)
    u = [rho * J[a] for a in range(6)]
    return np.stack([u[a] * J[e] for a in range(6) for e in range(a, 6)]), np.stack([u[a] * r for a in range(6)])


def terms(p, q, n, g, Is, It, lam, loss=None):
    """Colored ICP's terms of the correspondences (columns of p' = T_k P, q, the target normals n and gradients g, the
    intensities Is and It): the geometric row r = sl (d . n), J = sl [p' x n, n], then the photometric row
    r = sc (Is - (g . d + It)), J = sc [p' x m, m], m = -(g - (g . n) n), each weighted by rho(r); a photometric term
    equal to zero leaves the geometric one as it is.  (h [21, K], g [6, K])."""
    sl, sc = np.sqrt(np.float64(lam)), np.sqrt(1.0 - np.float64(lam))
    d = [p[0] - q[0], p[1] - q[1], p[2] - q[2]]
    h, gg = _row(_scaled_row(p, n, sl), sl * ((d[0] * n[0] + d[1] * n[1]) + d[2] * n[2]), loss)
    gn = (g[0] * n[0] + g[1] * n[1]) + g[2] * n[2]
    m = [-(g[r] - gn * n[r]) for r in range(3)]
    gd = (g[0] * d[0] + g[1] * d[1]) + g[2] * d[2]
    h2, g2 = _row(_scaled_row(p, m, sc), sc * (Is - (gd + It)), loss)
    return np.where(h2 == 0.0, h, h + h2), np.where(g2 == 0.0, gg, gg + g2)


def system(Pp, Q, N, Gt, Is, It, corr, lam, loss=None):
    """(H upper triangle [21], g [6]) summed over the correspondences of the evaluation at T_k."""
    sel = np.flatnonzero(corr >= 0)
    j = corr[sel]
    h, g = terms(Pp[:, sel], Q[:, j], N[:, j], Gt[:, j], Is[sel], It[j], lam, loss)
    return h.sum(axis=1), g.sum(axis=1)


def step_check(P, Q, N, Gt, Cs, Ct, d, R_k, t_k, lam, loss=None, tree=None):
    """What the evaluation of trace record T_k must produce (oracle/icp.py's step_check with colored ICP's update)
    for the target gradients Gt."""
    Pp = OI.transform(P, R_k, t_k)
    corr, d2 = OI.correspond(Pp, Q, d, N, tree)
    n, fitness, rmse = OI.evaluate(corr, d2)
    nxt = None
    if n >= 6:
        x = G.solve6(*system(Pp, Q, N, Gt, intensity(Cs), intensity(Ct), corr, lam, loss))
        if x is not None:
            nxt = OI.compose((OI.euler_zyx(x), x[3:].copy()), R_k, t_k)
    return {"corr": corr, "d2": d2, "n_corr": n, "fitness": fitness, "inlier_rmse": rmse, "next": nxt}


def colored_icp(P, Q, Cs, Ct, N, R0, t0, d, lam=0.968, loss=None, *, Gt=None, max_iterations=30,
                relative_fitness=1e-6, relative_rmse=1e-6):
    """The free-running loop of oracle/icp.py's icp with colored ICP's update; Gt: the target gradients (default: the
    restatement's, radius 2 d and max_nn 30)."""
    P, Q = np.asarray(P, dtype=np.float64), np.asarray(Q, dtype=np.float64)
    R, t = np.array(R0, dtype=np.float64), np.array(t0, dtype=np.float64)
    out = {"R": R, "t": t, "fitness": 0.0, "inlier_rmse": 0.0, "n_corr": 0, "iterations": 0, "status": OI.NO_UPDATE,
           "corr": np.full(P.shape[1], -1, dtype=np.int64), "trace": [(R, t, 0.0, 0.0, 0)]}
    if P.shape[1] == 0 or Q.shape[1] == 0:
        return out
    if Gt is None:
        Gt = gradients(Q, Ct, N, 2.0 * d)[0]
    keep = np.flatnonzero(OI.candidate_mask(Q, N))
    tree = cKDTree(Q[:, keep].T) if keep.size else None
    out["trace"] = []
    prev, k = None, 0
    while True:
        s = step_check(P, Q, N, Gt, Cs, Ct, d, R, t, lam, loss, tree)
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
