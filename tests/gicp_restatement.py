"""Numpy restatement of generalized ICP's update (DESIGN.md section 11, "Generalized ICP"; csrc/k9_icp.cu's
`unit_normal`, `gicp_terms` and `solve6`): test infrastructure only.

The loop, evaluation, correspondences (every target point a candidate) and stop rule are oracle/icp.py's.  Given the
same transform bits, `terms` reproduces the kernel's per-correspondence H = A^T M A and g = A^T M d bit for bit: every
product, sum, square root and division is one elementwise IEEE FP64 operation in the kernel's order.  The sums over
the correspondences are in numpy's order, so H, g and the update agree with the kernel's to the last few bits only.
"""
from __future__ import annotations

import numpy as np

from oracle import icp as OI


def unit_normals(N):
    """n / sqrt((x x + y y) + z z) per column; 0 where that squared length is not finite and positive."""
    x, y, z = np.asarray(N, dtype=np.float64)
    s2 = (x * x + y * y) + z * z
    ok = np.isfinite(s2) & (s2 > 0.0)
    s = np.sqrt(np.where(ok, s2, 1.0))
    return np.where(ok, np.stack([x / s, y / s, z / s]), 0.0)


def rotate(R, U):
    """R U in transform_point's unfused order, without a translation."""
    a0, a1, a2 = U
    return np.stack([(R[r, 0] * a0 + R[r, 1] * a1) + R[r, 2] * a2 for r in range(3)])


def cross(a, b):
    """(a1 b2 - a2 b1, a2 b0 - a0 b2, a0 b1 - a1 b0), columnwise."""
    return np.stack([a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]])


def covariance(m, n, w):
    """C = 2 I - w (m m^T + n n^T) as (C00, C01, C02, C11, C12, C22), columnwise; m = 0 or n = 0 drops that term."""
    def entry(r, s):
        return (2.0 if r == s else 0.0) - w * (m[r] * m[s] + n[r] * n[s])
    return tuple(entry(r, s) for r, s in ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)))


def inverse(C):
    """adj(C) / det(C) of the symmetric C: the 3 x 3 rows of M, columnwise."""
    C00, C01, C02, C11, C12, C22 = C
    A00, A01, A02 = C11 * C22 - C12 * C12, C02 * C12 - C01 * C22, C01 * C12 - C02 * C11
    A11, A12, A22 = C00 * C22 - C02 * C02, C01 * C02 - C00 * C12, C00 * C11 - C01 * C01
    det = (C00 * A00 + C01 * A01) + C02 * A02
    M00, M01, M02, M11, M12, M22 = (A / det for A in (A00, A01, A02, A11, A12, A22))
    return [[M00, M01, M02], [M01, M11, M12], [M02, M12, M22]]


def terms(p, q, m, n, w):
    """Per correspondence (columns): h [21, K] (A^T M A, upper triangle row by row) and g [6, K] (A^T M d), A = [-[p']x,
    I3], d = p' - q, M = (2 I - w (m m^T + n n^T))^-1."""
    M = inverse(covariance(m, n, w))
    d = [p[0] - q[0], p[1] - q[1], p[2] - q[2]]
    e = [(M[r][0] * d[0] + M[r][1] * d[1]) + M[r][2] * d[2] for r in range(3)]
    K = [cross(p, np.stack(M[r])) for r in range(3)]                       # row r: p' x M_r
    SK = np.stack([cross(p, np.stack([K[0][b], K[1][b], K[2][b]])) for b in range(3)], axis=1)   # [a, b, K]
    h = []
    for a in range(3):
        h += [SK[a, b] for b in range(a, 3)] + [K[b][a] for b in range(3)]
    h += [M[a][b] for a in range(3) for b in range(a, 3)]
    pe = cross(p, np.stack(e))
    return np.stack(h), np.stack([pe[0], pe[1], pe[2], e[0], e[1], e[2]])


def system(Pp, Q, Ns, Nt, R_k, corr, epsilon):
    """(H upper triangle [21], g [6]) summed over the correspondences of the evaluation at T_k (Pp = T_k P)."""
    sel = np.flatnonzero(corr >= 0)
    j = corr[sel]
    m = rotate(R_k, unit_normals(np.asarray(Ns, dtype=np.float64)[:, sel]))
    n = unit_normals(np.asarray(Nt, dtype=np.float64)[:, j])
    h, g = terms(Pp[:, sel], Q[:, j], m, n, 1.0 - epsilon)
    return h.sum(axis=1), g.sum(axis=1)


def solve6(A, g):
    """k9_icp.cu's solve6 in Python floats: Cholesky of the 21-entry upper triangle A, x with A x = -g; None on a
    non-positive pivot or a non-finite solution."""
    idx = {}
    v = 0
    for a in range(6):
        for e in range(a, 6):
            idx[a, e] = idx[e, a] = v
            v += 1
    A, g = [float(x) for x in A], [float(x) for x in g]
    L = [[0.0] * 6 for _ in range(6)]
    for j in range(6):
        d = A[idx[j, j]]
        for k in range(j):
            d -= L[j][k] * L[j][k]
        if not d > 0.0:
            return None
        L[j][j] = float(np.sqrt(d))
        for i in range(j + 1, 6):
            s = A[idx[i, j]]
            for k in range(j):
                s -= L[i][k] * L[j][k]
            L[i][j] = s / L[j][j]
    y = [0.0] * 6
    for i in range(6):
        s = -g[i]
        for k in range(i):
            s -= L[i][k] * y[k]
        y[i] = s / L[i][i]
    x = [0.0] * 6
    for i in range(5, -1, -1):
        s = y[i]
        for k in range(i + 1, 6):
            s -= L[k][i] * x[k]
        x[i] = s / L[i][i]
    x = np.array(x)
    return x if np.isfinite(x).all() else None


def update(Pp, Q, Ns, Nt, R_k, corr, epsilon):
    """(R_u, t_u) = [Rz(x2) Ry(x1) Rx(x0) | x3..5], or None below 3 correspondences or when solve6 fails."""
    if int((corr >= 0).sum()) < 3:
        return None
    H, g = system(Pp, Q, Ns, Nt, R_k, corr, epsilon)
    x = solve6(H, g)
    return None if x is None else (OI.euler_zyx(x), x[3:].copy())


def step_check(P, Q, Ns, Nt, d, R_k, t_k, epsilon, tree=None):
    """oracle/icp.py's step_check with generalized ICP's update."""
    Pp = OI.transform(P, R_k, t_k)
    corr, d2 = OI.correspond(Pp, Q, d, None, tree)
    n, fitness, rmse = OI.evaluate(corr, d2)
    U = update(Pp, Q, Ns, Nt, R_k, corr, epsilon)
    return {"corr": corr, "d2": d2, "n_corr": n, "fitness": fitness, "inlier_rmse": rmse,
            "next": None if U is None else OI.compose(U, R_k, t_k)}
