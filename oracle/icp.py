"""Numpy restatement of the ICP refinement (DESIGN.md section 11, csrc/k9_icp.cu): test infrastructure only.

Given the same transform bits, `transform` and `correspond` reproduce the kernel's transformed points, squared
distances and correspondences bit for bit (FP64, the kernel's unfused operation order, ties to the lowest target
index).  The sums (rmse, H, J^T J, J^T r) are FP64 in numpy's order, so they and the updates they give agree with the
kernel's to the last few bits only.
"""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

CONVERGED, MAX_ITERATIONS, NO_UPDATE = 0, 1, 2


def transform(P, R, t):
    """((R[r, 0] x + R[r, 1] y) + R[r, 2] z) + t[r], elementwise (R @ P could fuse or reorder)."""
    x, y, z = np.asarray(P, dtype=np.float64)
    return np.stack([((R[r, 0] * x + R[r, 1] * y) + R[r, 2] * z) + t[r] for r in range(3)])


def sqdist(Pp, Q, i, j):
    """((dx dx + dy dy) + dz dz) with d = q_j - p'_i, as the kernel evaluates it."""
    dx, dy, dz = (Q[r, j] - Pp[r, i] for r in range(3))
    return (dx * dx + dy * dy) + dz * dz


def candidate_mask(Q, normals=None):
    """Target points that can be a correspondence (point-to-plane: finite normal)."""
    if normals is None:
        return np.ones(Q.shape[1], dtype=bool)
    return np.isfinite(normals).all(axis=0)


def correspond(Pp, Q, d, normals=None, tree=None):
    """(corr [n_s] int64 target index or -1, d2 [n_s] float64, inf without one).  tree: a cKDTree over the candidate
    targets (candidate_mask) to reuse."""
    Pp = np.asarray(Pp, dtype=np.float64)
    ns = Pp.shape[1]
    keep = np.flatnonzero(candidate_mask(Q, normals))
    corr = np.full(ns, -1, dtype=np.int64)
    d2 = np.full(ns, np.inf)
    if ns == 0 or keep.size == 0:
        return corr, d2
    if tree is None:
        tree = cKDTree(Q[:, keep].T)
    lists = tree.query_ball_point(Pp.T, d * (1 + 1e-9), workers=-1)
    lens = np.fromiter((len(x) for x in lists), dtype=np.int64, count=ns)
    if lens.sum() == 0:
        return corr, d2
    ii = np.repeat(np.arange(ns), lens)
    jj = keep[np.concatenate([np.asarray(x, dtype=np.int64) for x in lists if len(x)])]
    dist = sqdist(Pp, Q, ii, jj)
    ok = dist <= d * d
    ii, jj, dist = ii[ok], jj[ok], dist[ok]
    order = np.lexsort((jj, dist, ii))          # by source, then distance, then target index
    ii, jj, dist = ii[order], jj[order], dist[order]
    first = np.ones(ii.size, dtype=bool)
    first[1:] = ii[1:] != ii[:-1]
    corr[ii[first]] = jj[first]
    d2[ii[first]] = dist[first]
    return corr, d2


def evaluate(corr, d2):
    """(n_corr, fitness, inlier_rmse) of one evaluation."""
    sel = corr >= 0
    n = int(sel.sum())
    fitness = n / corr.size if corr.size else 0.0
    rmse = float(np.sqrt(d2[sel].sum() / n)) if n else 0.0
    return n, fitness, rmse


def kabsch(H):
    """R = V U^T of H = U S V^T, the smallest singular direction flipped when det(U) det(V) < 0 (svd3.cuh)."""
    U, _, Vt = np.linalg.svd(H)
    V = Vt.T
    if np.linalg.det(U) * np.linalg.det(V) < 0:
        V[:, 2] = -V[:, 2]
    return V @ U.T


def update_point_to_point(Pp, Q, corr):
    """Umeyama without scale over the correspondences: (R_u, t_u), or None below 3 correspondences."""
    sel = np.flatnonzero(corr >= 0)
    if sel.size < 3:
        return None
    p, q = Pp[:, sel], Q[:, corr[sel]]
    mu_p, mu_q = p.mean(axis=1), q.mean(axis=1)
    H = (p - mu_p[:, None]) @ (q - mu_q[:, None]).T
    R = kabsch(H)
    return R, mu_q - R @ mu_p


def euler_zyx(x):
    """Rz(x2) Ry(x1) Rx(x0)."""
    ca, sa, cb, sb, cg, sg = np.cos(x[0]), np.sin(x[0]), np.cos(x[1]), np.sin(x[1]), np.cos(x[2]), np.sin(x[2])
    Rx = np.array([[1, 0, 0], [0, ca, -sa], [0, sa, ca]])
    Ry = np.array([[cb, 0, sb], [0, 1, 0], [-sb, 0, cb]])
    Rz = np.array([[cg, -sg, 0], [sg, cg, 0], [0, 0, 1]])
    return Rz @ Ry @ Rx


def update_point_to_plane(Pp, Q, N, corr):
    """Open3D's linearisation: r = (p' - q).n, J = [p' x n, n]; solve J^T J x = -J^T r by Cholesky.  (R_u, t_u), or
    None below 6 correspondences, on a non-positive pivot or a non-finite solution."""
    sel = np.flatnonzero(corr >= 0)
    if sel.size < 6:
        return None
    p, q, n = Pp[:, sel], Q[:, corr[sel]], N[:, corr[sel]]
    r = ((p - q) * n).sum(axis=0)
    J = np.concatenate([np.cross(p.T, n.T).T, n])          # 6 x K
    A, g = J @ J.T, J @ r
    try:
        L = np.linalg.cholesky(A)
    except np.linalg.LinAlgError:
        return None
    x = np.linalg.solve(L.T, np.linalg.solve(L, -g))
    if not np.isfinite(x).all():
        return None
    return euler_zyx(x), x[3:].copy()


def compose(U, R, t):
    """U T: (R_u R, R_u t + t_u)."""
    Ru, tu = U
    return Ru @ R, Ru @ t + tu


def step_check(P, Q, d, R_k, t_k, *, normals=None, point_to_plane=False, tree=None):
    """What the evaluation of the GPU's trace record T_k must produce: corr, d2, n_corr, fitness, inlier_rmse and
    next = T_{k+1} = U T_k (None when no update can be computed)."""
    Pp = transform(P, R_k, t_k)
    corr, d2 = correspond(Pp, Q, d, normals if point_to_plane else None, tree)
    n, fitness, rmse = evaluate(corr, d2)
    U = update_point_to_plane(Pp, Q, normals, corr) if point_to_plane else update_point_to_point(Pp, Q, corr)
    return {"corr": corr, "d2": d2, "n_corr": n, "fitness": fitness, "inlier_rmse": rmse,
            "next": None if U is None else compose(U, R_k, t_k)}


def stop(k, prev, cur, max_iterations, relative_fitness, relative_rmse):
    """The stop rule after evaluation k (prev, cur = (fitness, rmse)): a status, or None to go on."""
    if k > 0 and abs(cur[0] - prev[0]) < relative_fitness and abs(cur[1] - prev[1]) < relative_rmse:
        return CONVERGED
    if k >= max_iterations:
        return MAX_ITERATIONS
    return None


def icp(P, Q, R0, t0, d, *, normals=None, point_to_plane=False, max_iterations=30, relative_fitness=1e-6,
        relative_rmse=1e-6):
    """The free-running loop: dict with R, t, fitness, inlier_rmse, n_corr, iterations, status, corr and trace (one
    (R, t, fitness, inlier_rmse, n_corr) per evaluation)."""
    P, Q = np.asarray(P, dtype=np.float64), np.asarray(Q, dtype=np.float64)
    R, t = np.array(R0, dtype=np.float64), np.array(t0, dtype=np.float64)
    out = {"R": R, "t": t, "fitness": 0.0, "inlier_rmse": 0.0, "n_corr": 0, "iterations": 0, "status": NO_UPDATE,
           "corr": np.full(P.shape[1], -1, dtype=np.int64), "trace": [(R, t, 0.0, 0.0, 0)]}
    if P.shape[1] == 0 or Q.shape[1] == 0:
        return out
    keep = np.flatnonzero(candidate_mask(Q, normals if point_to_plane else None))
    tree = cKDTree(Q[:, keep].T) if keep.size else None
    out["trace"] = []
    prev, k = None, 0
    while True:
        s = step_check(P, Q, d, R, t, normals=normals, point_to_plane=point_to_plane, tree=tree)
        cur = (s["fitness"], s["inlier_rmse"])
        out.update(R=R, t=t, fitness=cur[0], inlier_rmse=cur[1], n_corr=s["n_corr"], corr=s["corr"], iterations=k)
        out["trace"].append((R, t, cur[0], cur[1], s["n_corr"]))
        status = stop(k, prev, cur, max_iterations, relative_fitness, relative_rmse)
        if status is None and s["next"] is None:
            status = NO_UPDATE
        if status is not None:
            out["status"] = status
            return out
        R, t = s["next"]
        prev, k = cur, k + 1
