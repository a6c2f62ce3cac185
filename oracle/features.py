"""numpy restatement of the correspondence stage (csrc/k8_features.cu, DESIGN.md section 10): radius normals, FPFH
descriptors, the two-way descriptor nearest neighbour and FGR's matcher (lists and tuple test).

TEST INFRASTRUCTURE ONLY.  It follows the section's definitions, not the kernels' loops: neighbourhoods by k-d tree
(then the same FP32 distance test), sums in numpy's order.  Where a result can legitimately differ from the device
because of summation order or a last-bit difference of acos / atan2, the item is flagged *fragile*:
  - a pair whose bin argument lies within 1e-5 of an integer, or whose |a1| and |a2| differ, by at most 1e-6
    relative + 1e-7 (the swap test);
  - a neighbour with |d^2 - r^2| <= 1e-6 r^2;
  - a normal whose two smallest eigenvalues are within 1e-6 relative, or that lies within 1e-7 of perpendicular to
    the viewpoint direction;
  - a descriptor nearest neighbour whose best and second-best distances differ by less than 1e-6 relative;
  - a tuple trial within 1e-6 relative of a ratio bound.
"""
import math

import numpy as np
from scipy.spatial import cKDTree

BINS = 11
DIM = 33
DOMAIN_TUPLE = 5
MAX_TUPLES = 1000


def _f32(points):
    return np.ascontiguousarray(np.asarray(points, dtype=np.float64).T).astype(np.float32)  # [n, 3]


def sqdist32(p, q):
    """The device's FP32 |q - p|^2: ((dx dx + dy dy) + dz dz), unfused."""
    d = (q - p).astype(np.float32)
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def neighbours(points, r):
    """Directed pairs (i, j), i included among its own neighbours, with FP32 |p_j - p_i|^2 <= float32(r^2), sorted by
    (i, j); plus d^2 (float32) and the boundary-fragile flag of each pair."""
    p32 = _f32(points)
    n = p32.shape[0]
    r2 = np.float32(r * r)
    tree = cKDTree(p32.astype(np.float64))
    lists = tree.query_ball_point(p32.astype(np.float64), r * (1 + 1e-4) + 1e-30)
    ii = np.repeat(np.arange(n), [len(x) for x in lists]) if n else np.zeros(0, dtype=np.int64)
    jj = np.concatenate([np.asarray(x, dtype=np.int64) for x in lists]) if n else np.zeros(0, dtype=np.int64)
    d2 = sqdist32(p32[ii], p32[jj])
    keep = d2 <= r2
    ii, jj, d2 = ii[keep], jj[keep], d2[keep]
    order = np.lexsort((jj, ii))
    ii, jj, d2 = ii[order], jj[order], d2[order]
    frag = np.abs(d2.astype(np.float64) - float(r2)) <= 1e-6 * float(r2)
    # (a pair just outside the radius is as fragile as one just inside)
    out_frag = np.zeros(n, dtype=bool)
    lists_wide = tree.query_ball_point(p32.astype(np.float64), r * (1 + 1e-5) + 1e-30)
    for i, x in enumerate(lists_wide):
        if x:
            dd = sqdist32(np.repeat(p32[i:i + 1], len(x), 0), p32[np.asarray(x)]).astype(np.float64)
            out_frag[i] = bool(np.any(np.abs(dd - float(r2)) <= 1e-6 * float(r2)))
    return ii, jj, d2, frag, out_frag


def radius_normals(points, r, viewpoint=(0.0, 0.0, 0.0)):
    """3xn normals (NaN for fewer than 3 neighbours) and a per-point fragile flag."""
    P = np.asarray(points, dtype=np.float64)
    n = P.shape[1]
    ii, jj, _, _, bfrag = neighbours(P, r)
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
    frag = bfrag.copy()
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
    return normals, frag


def pair_features(p, np_, q, nq):
    """PCL computePairFeatures for arrays of pairs (float32 [m, 3] each): f1, f2, f3, valid, fragile."""
    p, np_, q, nq = (np.asarray(x, dtype=np.float32) for x in (p, np_, q, nq))

    def dot(a, b):
        return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]

    def cross(a, b):
        return np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                         a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], axis=1)

    with np.errstate(invalid="ignore", divide="ignore"):
        d = (q - p).astype(np.float32)
        ln = np.sqrt(dot(d, d))
        valid = ~(np.isnan(np_[:, 0]) | np.isnan(nq[:, 0])) & (ln != 0)
        a1 = dot(np_, d) / ln
        a2 = dot(nq, d) / ln
        swap = np.abs(a1) < np.abs(a2)  # acos(|a1|) > acos(|a2|)
        # one FP32 ulp of a normal moves a1 / a2 by ~1e-7: a swap decision closer than that may go either way (an
        # exact tie, two equal FP32 normals, is decided the same way on both sides)
        big = np.maximum(np.abs(a1), np.abs(a2)).astype(np.float64)
        gap = np.abs(np.abs(a1).astype(np.float64) - np.abs(a2))
        frag = (gap > 0) & (gap <= 1e-6 * big + 1e-7)
        n1 = np.where(swap[:, None], nq, np_)
        n2 = np.where(swap[:, None], np_, nq)
        d = np.where(swap[:, None], -d, d)
        f3 = np.where(swap, -a2, a1).astype(np.float32)
        v = cross(d, n1)
        vn = np.sqrt(dot(v, v))
        valid &= vn != 0
        v = v / vn[:, None]
        w = cross(n1, v)
        f2 = dot(v, n2)
        f1 = np.arctan2(dot(w, n2), dot(n1, n2))
    return f1, f2, f3, valid, frag


def bin_args(f1, f2, f3):
    return np.stack([11.0 * (f1.astype(np.float64) + math.pi) / (2.0 * math.pi),
                     11.0 * (f2.astype(np.float64) + 1.0) / 2.0, 11.0 * (f3.astype(np.float64) + 1.0) / 2.0], axis=1)


def fpfh(points, normal_radius, feature_radius, viewpoint=(0.0, 0.0, 0.0), normals=None):
    """(features n x 33 float32, normals 3xn, fragile [n]) following DESIGN.md section 10."""
    P = np.asarray(points, dtype=np.float64)
    n = P.shape[1]
    nfrag = np.zeros(n, dtype=bool)
    if normals is None:
        normals, nfrag = radius_normals(P, normal_radius, viewpoint)
    p32 = _f32(P)
    n32 = np.asarray(normals, dtype=np.float64).T.astype(np.float32)
    ii, jj, d2, bfrag_pair, bfrag_out = neighbours(P, feature_radius)
    K = np.bincount(ii, minlength=n)
    other = ii != jj
    pi, pj = ii[other], jj[other]
    f1, f2, f3, valid, sfrag = pair_features(p32[pi], n32[pi], p32[pj], n32[pj])
    with np.errstate(invalid="ignore"):
        args = bin_args(f1, f2, f3)
    afrag = np.any(np.abs(args - np.round(args)) <= 1e-5, axis=1)
    pfrag = ((sfrag | afrag) & valid) | nfrag[pi] | nfrag[pj]
    bins = np.clip(np.floor(np.nan_to_num(args, nan=0.0)).astype(np.int64), 0, BINS - 1)
    counts = np.zeros((n, DIM), dtype=np.int64)
    for h in range(3):
        np.add.at(counts, (pi[valid], h * BINS + bins[valid, h]), 1)
    spfh_frag = np.zeros(n, dtype=bool)
    np.logical_or.at(spfh_frag, pi, pfrag)
    np.logical_or.at(spfh_frag, ii, bfrag_pair)
    spfh_frag |= bfrag_out
    # FPFH: neighbours j != i at distance > 0, weight 1 / d^2 (FP64 of the FP32 distance)
    use = other & (d2 > 0)
    fi, fj = ii[use], jj[use]
    Kj = K[fj]
    w = np.where(Kj > 1, (100.0 / np.maximum(Kj - 1, 1)) / d2[use].astype(np.float64), 0.0)
    acc = np.zeros((n, DIM))
    np.add.at(acc, fi, counts[fj].astype(np.float64) * w[:, None])
    out = np.zeros((n, DIM), dtype=np.float32)
    for h in range(3):
        s = acc[:, h * BINS:(h + 1) * BINS].sum(axis=1)
        pos = s > 0
        out[pos, h * BINS:(h + 1) * BINS] = (acc[pos, h * BINS:(h + 1) * BINS] * (100.0 / s[pos])[:, None]).astype(
            np.float32)
    frag = spfh_frag.copy()
    np.logical_or.at(frag, fi, spfh_frag[fj])
    return out, normals, frag


def descriptor_distances(fs, ft):
    """n_s x n_t squared distances as the device forms them: d = a - b in FP32, acc = fma(d, d, acc) for the 33
    dimensions in order (a float64 product is exact, so fma is one float64 add rounded to float32)."""
    fs = np.asarray(fs, dtype=np.float32)
    ft = np.asarray(ft, dtype=np.float32)
    acc = np.zeros((fs.shape[0], ft.shape[0]), dtype=np.float32)
    for k in range(DIM):
        d = (fs[:, k][:, None] - ft[:, k][None, :]).astype(np.float32).astype(np.float64)
        acc = (acc.astype(np.float64) + d * d).astype(np.float32)
    return acc


def nearest_neighbours(fs, ft, block=2048):
    """(nn_src_to_tgt, nn_tgt_to_src, fragile_src, fragile_tgt): ties to the lowest index; fragile = best and
    second-best within 1e-6 relative."""
    fs = np.asarray(fs, dtype=np.float32)
    ft = np.asarray(ft, dtype=np.float32)
    ns, nt = fs.shape[0], ft.shape[0]
    nn_t = np.full(ns, -1, dtype=np.int64)
    fr_s = np.zeros(ns, dtype=bool)
    col_best = np.full(nt, np.inf)
    col_second = np.full(nt, np.inf)
    nn_s = np.full(nt, -1, dtype=np.int64)
    for r0 in range(0, ns, block):
        D = descriptor_distances(fs[r0:r0 + block], ft).astype(np.float64)
        nn_t[r0:r0 + block] = np.argmin(D, axis=1)
        if nt > 1:
            part = np.partition(D, 1, axis=1)
            fr_s[r0:r0 + block] = part[:, 1] - part[:, 0] <= 1e-6 * np.maximum(part[:, 1], 1e-30)
        # running column minimum and second minimum (ties keep the earlier, i.e. lower, row)
        arg = np.argmin(D, axis=0)
        m = D[arg, np.arange(nt)]
        if D.shape[0] > 1:
            sec = np.partition(D, 1, axis=0)[1]
        else:
            sec = np.full(nt, np.inf)
        better = m < col_best
        new_second = np.where(better, np.minimum(col_best, sec), np.minimum(col_second, m))
        nn_s = np.where(better, arg + r0, nn_s)
        col_best = np.where(better, m, col_best)
        col_second = new_second
    fr_t = col_second - col_best <= 1e-6 * np.maximum(col_second, 1e-30)
    return nn_t, nn_s, fr_s, fr_t


def match_list(nn_t, nn_s, crosscheck):
    """FGR's list: mutual pairs (crosscheck), or (i, nn_t(i)) for every i that is some nn_s(j), then (nn_s(j), j)."""
    nn_t = np.asarray(nn_t, dtype=np.int64)
    nn_s = np.asarray(nn_s, dtype=np.int64)
    ns = nn_t.shape[0]
    if crosscheck:
        i = np.flatnonzero(nn_s[nn_t] == np.arange(ns))
        return np.stack([i, nn_t[i]], axis=1)
    marked = np.zeros(ns, dtype=bool)
    marked[nn_s] = True
    i = np.flatnonzero(marked)
    first = np.stack([i, nn_t[i]], axis=1)
    second = np.stack([nn_s, np.arange(nn_s.shape[0])], axis=1)
    return np.concatenate([first, second]).reshape(-1, 2)


def tuple_draws(seed, first_trial, count, ncorr):
    """List positions of trials [first_trial, first_trial + count): rand31(seed; TUPLE, 0, 3t + k) % ncorr."""
    from oracle import oracle as O

    k0 = 3 * first_trial
    k1 = 3 * (first_trial + count)
    blocks = np.stack([O.philox(seed, DOMAIN_TUPLE, 0, b) for b in range(k0 >> 2, ((k1 - 1) >> 2) + 1)])
    words = blocks.reshape(-1)[k0 - 4 * (k0 >> 2):][:k1 - k0] >> 1
    return (words.astype(np.int64) % ncorr).reshape(count, 3)


def tuple_test(src, tgt, corr, scale, seed, chunk=4096):
    """(pairs (3 * kept, 2), fragile_trial_seen): the first min(#passing, 1000) passing trials in trial order."""
    corr = np.asarray(corr, dtype=np.int64).reshape(-1, 2)
    ncorr = corr.shape[0]
    s32, t32 = _f32(src), _f32(tgt)
    s = np.float32(scale)
    kept, fragile = [], False
    for t0 in range(0, 100 * ncorr, chunk):
        cnt = min(chunk, 100 * ncorr - t0)
        r = tuple_draws(seed, t0, cnt, ncorr)
        ok = np.ones(cnt, dtype=bool)
        near = np.zeros(cnt, dtype=bool)
        for e in range(3):
            a, b = r[:, e], r[:, (e + 1) % 3]
            li = np.sqrt(sqdist32(s32[corr[a, 0]], s32[corr[b, 0]]))
            lj = np.sqrt(sqdist32(t32[corr[a, 1]], t32[corr[b, 1]]))
            with np.errstate(invalid="ignore", divide="ignore"):
                lo, hi = (li * s).astype(np.float32), (li / s).astype(np.float32)
                ok &= (lo < lj) & (lj < hi)
                tol = 1e-6 * np.maximum(lj.astype(np.float64), 1e-30)
                near |= (np.abs(lo.astype(np.float64) - lj) <= tol) | (np.abs(hi.astype(np.float64) - lj) <= tol)
        for u in np.flatnonzero(ok | near):
            fragile |= bool(near[u])
            if ok[u]:
                kept.append(r[u])
            if len(kept) >= MAX_TUPLES:
                break
        if len(kept) >= MAX_TUPLES:
            break
    if not kept:
        return np.zeros((0, 2), dtype=np.int64), fragile
    return corr[np.concatenate(kept)], fragile
