"""numpy restatement of the hybrid normals (csrc/k8_features.cu, k8_radius_normals with kCap; DESIGN.md section 10,
"Normals alone"), built on the radius neighbourhoods of oracle/features.py.

TEST INFRASTRUCTURE ONLY.  Point i keeps the max_nn smallest keys (FP32 d^2 bits, j) of its radius neighbourhood (d^2
>= 0, so the bits sort as the numbers do; ties go to the lower index), or the whole neighbourhood when it is no
larger.  Mean, covariance, smallest eigenvector and the flip follow oracle.features.radius_normals, in numpy's order.
Fragile, besides radius_normals' flags (the two smallest eigenvalues within 1e-6 relative, a normal within 1e-7 of
perpendicular to the viewpoint, a neighbour within 1e-6 relative of the radius):
  - a capped point whose max_nn-th and (max_nn + 1)-th d^2 differ, by at most 1e-6 relative: FP32 rounding of a
    coordinate may swap them (an exact tie is decided by the index on both sides).
"""
import numpy as np

from oracle import features as OF


def hybrid_neighbours(points, r, max_nn):
    """(ii, jj, sizes, fragile): the kept pairs sorted by (i, j), the radius neighbourhood's size per point and the
    per-point fragile flag of the selection (near-tie at the cap, or a neighbour near the radius)."""
    P = np.asarray(points, dtype=np.float64)
    n = P.shape[1]
    ii, jj, d2, _, bfrag = OF.neighbours(P, r)
    sizes = np.bincount(ii, minlength=n)
    # rank every candidate of point i by (d^2 bits, j): lexsort's last key is the primary one
    bits = d2.view(np.uint32).astype(np.int64)
    order = np.lexsort((jj, bits, ii))
    start = np.concatenate([[0], np.cumsum(sizes)])
    rank = np.empty(ii.size, dtype=np.int64)
    rank[order] = np.arange(ii.size) - np.repeat(start[:-1], sizes)
    keep = rank < max_nn
    frag = bfrag.copy()
    capped = np.flatnonzero(sizes > max_nn)
    if capped.size:
        srt = d2[order].astype(np.float64)
        last = srt[start[capped] + max_nn - 1]       # the max_nn-th smallest d^2
        nxt = srt[start[capped] + max_nn]            # the first one left out
        frag[capped] |= (nxt != last) & (nxt - last <= 1e-6 * np.maximum(nxt, 1e-30))
    ii, jj = ii[keep], jj[keep]
    o = np.lexsort((jj, ii))
    return ii[o], jj[o], sizes, frag


def hybrid_normals(points, r, max_nn, viewpoint=(0.0, 0.0, 0.0), return_sizes=False):
    """3xn normals of the hybrid neighbourhood (NaN for fewer than 3 kept points) and a per-point fragile flag; with
    return_sizes also the radius neighbourhood's size per point (how many points the cap acted on)."""
    P = np.asarray(points, dtype=np.float64)
    n = P.shape[1]
    ii, jj, sizes, sfrag = hybrid_neighbours(P, r, max_nn)
    cnt = np.bincount(ii, minlength=n)
    mean = np.zeros((n, 3))
    for c in range(3):
        mean[:, c] = np.bincount(ii, weights=P[c, jj], minlength=n)
    ok = cnt >= 3
    mean[ok] /= cnt[ok, None]
    d = P[:, jj].T - mean[ii]
    cov = np.zeros((n, 3, 3))
    for a in range(3):
        for b in range(3):
            cov[:, a, b] = np.bincount(ii, weights=d[:, a] * d[:, b], minlength=n)
    normals = np.full((3, n), np.nan)
    frag = sfrag.copy()
    if ok.any():
        w, v = np.linalg.eigh(cov[ok])
        nv = v[:, :, 0]
        vp = np.asarray(viewpoint, dtype=np.float64)[None, :] - P[:, ok].T
        side = (vp * nv).sum(axis=1)
        nv[side < 0] *= -1
        normals[:, ok] = nv.T
        scale = np.maximum(np.abs(w[:, 2]), 1e-300)
        frag_ok = (np.abs(w[:, 1] - w[:, 0]) <= 1e-6 * scale) | (np.abs(side) <= 1e-7 * np.linalg.norm(vp, axis=1))
        frag[np.flatnonzero(ok)] |= frag_ok
    if return_sizes:
        return normals, frag, sizes
    return normals, frag
