"""numpy restatement of the correspondence stage (csrc/k8_features.cu, DESIGN.md section 10): radius normals, FPFH
descriptors, the two-way descriptor nearest neighbour and FGR's matcher (lists and tuple test).

TEST INFRASTRUCTURE ONLY.  It follows the section's definitions, not the kernels' loops: neighbourhoods by k-d tree
(then the same FP32 distance test), sums in numpy's order.  Where a result can legitimately differ from the device
because of summation order or a last-bit difference of acos / atan2, the item is flagged *fragile*:
  - a pair whose bin argument lies within 1e-5 of an integer, or whose |a1| and |a2| differ, by at most 1e-6
    relative + 1e-7 (the swap test); such a pair moves one count of each histogram at most, so a descriptor is
    fragile only when its fragile pairs could move it by more than SOFT_L1 (L1) in all;
  - a neighbour with |d^2 - r^2| <= 1e-6 r^2 (every descriptor it reaches is fragile);
  - a normal whose two smallest eigenvalues are within 1e-6 relative, or that lies within 1e-7 of perpendicular to
    the viewpoint direction;
  - a descriptor nearest neighbour whose best and second-best distances differ, by less than 1e-6 relative;
  - a tuple trial with an edge within 1e-6 relative of a ratio bound while its other edges pass or are as near.
"""
import math

import numpy as np
from scipy import sparse
from scipy.spatial import cKDTree

BINS = 11
DIM = 33
DOMAIN_TUPLE = 5
MAX_TUPLES = 1000
SOFT_L1 = 5e-4   # how far fragile pairs may move a descriptor (L1) before the descriptor counts as fragile


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


def fpfh(points, normal_radius, feature_radius, viewpoint=(0.0, 0.0, 0.0), normals=None, bounds=False):
    """(features n x 33 float32, normals 3xn, fragile [n]) following DESIGN.md section 10.  With bounds, also
    (hard [n], soft_l1 [n]): hard = a fragile neighbour set reaches the descriptor; otherwise the device's
    descriptor lies within soft_l1 (L1, plus rounding) of this one."""
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
    # per histogram h: a pair near a bin edge of feature h, near the swap decision or with a fragile normal
    afrag = np.abs(args - np.round(args)) <= 1e-5
    pfrag = (((sfrag[:, None] | afrag) & valid[:, None]) | (nfrag[pi] | nfrag[pj])[:, None])
    bins = np.clip(np.floor(np.nan_to_num(args, nan=0.0)).astype(np.int64), 0, BINS - 1)
    counts = np.zeros((n, DIM), dtype=np.int64)
    for h in range(3):
        counts[:, h * BINS:(h + 1) * BINS] = np.bincount(
            pi[valid] * BINS + bins[valid, h], minlength=n * BINS).reshape(n, BINS)
    # hard: a neighbour near the radius may join or leave (K and the weights change)
    hard = bfrag_out.copy()
    np.logical_or.at(hard, ii, bfrag_pair)
    # soft: a fragile pair of SPFH_j moves one count of a histogram at most
    nsoft = np.stack([np.bincount(pi, weights=pfrag[:, h], minlength=n) for h in range(3)], axis=1)
    # FPFH: neighbours j != i at distance > 0, weight 1 / d^2 (FP64 of the FP32 distance)
    use = other & (d2 > 0)
    fi, fj = ii[use], jj[use]
    Kj = K[fj]
    w = np.where(Kj > 1, (100.0 / np.maximum(Kj - 1, 1)) / d2[use].astype(np.float64), 0.0)
    W = sparse.csr_matrix((w, (fi, fj)), shape=(n, n))
    acc = np.asarray(W @ counts.astype(np.float64))
    out = np.zeros((n, DIM), dtype=np.float32)
    # moving one count of weight w between two bins of a histogram with sum s moves the output by 200 w / s in L1:
    # a point is fragile when its soft pairs could move it by more than SOFT_L1 in all, or when a hard flag reaches it
    wsoft = W @ nsoft
    moved = np.zeros(n)
    for h in range(3):
        s = acc[:, h * BINS:(h + 1) * BINS].sum(axis=1)
        pos = s > 0
        out[pos, h * BINS:(h + 1) * BINS] = (acc[pos, h * BINS:(h + 1) * BINS] * (100.0 / s[pos])[:, None]).astype(
            np.float32)
        moved += np.where(wsoft[:, h] > 0, 200.0 * wsoft[:, h] / np.maximum(s, 1e-300), 0.0)
    np.logical_or.at(hard, fi, hard[fj])
    frag = hard | (moved > SOFT_L1)
    if bounds:
        return out, normals, frag, hard, moved
    return out, normals, frag


def fma32(a, b, c):
    """The device's fmaf(a, b, c) on float32 arrays, rounded once: a * b is exact in float64, and s = a * b + c in
    float64 is exact up to the tail e that TwoSum recovers.  Rounding s to float32 is then correct unless s lies
    exactly halfway between two float32 values and e != 0 (double rounding): the tail then decides the direction."""
    a, b, c = (np.asarray(x, dtype=np.float32).astype(np.float64) for x in (a, b, c))
    with np.errstate(over="ignore", invalid="ignore"):
        p = a * b
        s = p + c
        bb = s - p
        e = (p - (s - bb)) + (c - bb)
        r = s.astype(np.float32)
        lo = np.where(r.astype(np.float64) > s, np.nextafter(r, np.float32(-np.inf)), r)
        mid = (lo.astype(np.float64) + np.nextafter(lo, np.float32(np.inf)).astype(np.float64)) * 0.5
        tie = np.isfinite(s) & (s == mid) & (e != 0)
    if tie.any():
        r = np.where(tie, np.where(e > 0, np.nextafter(lo, np.float32(np.inf)), lo), r)
    return r


def descriptor_distances(fs, ft):
    """n_s x n_t squared distances as the device forms them: d = a - b in FP32, acc = fma(d, d, acc) for the 33
    dimensions in order (fma32)."""
    fs = np.asarray(fs, dtype=np.float32)
    ft = np.asarray(ft, dtype=np.float32)
    acc = np.zeros((fs.shape[0], ft.shape[0]), dtype=np.float32)
    for k in range(DIM):
        d = (fs[:, k][:, None] - ft[:, k][None, :]).astype(np.float32)
        acc = fma32(d, d, acc)
    return acc


def near_tie(best, second):
    """Best and second-best distances within 1e-6 relative but not equal (descriptor_distances is the device's value
    bit for bit, and an exact tie goes to the lowest index on both sides); no second-best is no tie."""
    with np.errstate(invalid="ignore"):
        return np.isfinite(second) & (second != best) & (second - best <= 1e-6 * np.maximum(second, 1e-30))


def nearest_neighbours(fs, ft, block=2048):
    """(nn_src_to_tgt, nn_tgt_to_src, fragile_src, fragile_tgt): ties to the lowest index; fragile = best and
    second-best within 1e-6 relative (near_tie)."""
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
            fr_s[r0:r0 + block] = near_tie(part[:, 0], part[:, 1])
        # running column minimum and second minimum (ties keep the earlier, i.e. lower, row)
        arg = np.argmin(D, axis=0)
        m = D[arg, np.arange(nt)]
        if D.shape[0] > 1:
            sec = np.partition(D, 1, axis=0)[1]
        else:
            sec = np.full(nt, np.inf)
        better = (m < col_best) | (nn_s < 0)          # (an all-inf column still picks its lowest row)
        new_second = np.where(better, np.minimum(col_best, sec), np.minimum(col_second, m))
        nn_s = np.where(better, arg + r0, nn_s)
        col_best = np.where(better, m, col_best)
        col_second = new_second
    return nn_t, nn_s, fr_s, near_tie(col_best, col_second)


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


def philox_blocks(seed, domain, event, blocks):
    """Philox4x32-10 (oracle.philox) on an array of block counters at once: [len(blocks), 4] uint32."""
    blocks = np.asarray(blocks, dtype=np.uint64)
    m32 = np.uint64(0xFFFFFFFF)
    c0, c1 = blocks & m32, blocks >> np.uint64(32)
    c2 = np.full_like(c0, np.uint64(event) & m32)
    c3 = np.full_like(c0, np.uint64(domain) & m32)
    k0, k1 = int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & m32,
                          (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & m32)
        k0 = (k0 + 0x9E3779B9) & 0xFFFFFFFF
        k1 = (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return np.stack([c0, c1, c2, c3], axis=1).astype(np.uint32)


def tuple_draws(seed, first_trial, count, ncorr):
    """List positions of trials [first_trial, first_trial + count): rand31(seed; TUPLE, 0, 3t + k) % ncorr."""
    k0 = 3 * first_trial
    k1 = 3 * (first_trial + count)
    blocks = philox_blocks(seed, DOMAIN_TUPLE, 0, np.arange(k0 >> 2, ((k1 - 1) >> 2) + 1, dtype=np.uint64))
    words = blocks.reshape(-1)[k0 - 4 * (k0 >> 2):][:k1 - k0] >> 1
    return (words.astype(np.int64) % ncorr).reshape(count, 3)


def tuple_test(src, tgt, corr, scale, seed, chunk=1 << 16):
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
        could = np.ones(cnt, dtype=bool)   # every edge passes or is near a bound: a near edge may decide the trial
        for e in range(3):
            a, b = r[:, e], r[:, (e + 1) % 3]
            li = np.sqrt(sqdist32(s32[corr[a, 0]], s32[corr[b, 0]]))
            lj = np.sqrt(sqdist32(t32[corr[a, 1]], t32[corr[b, 1]]))
            with np.errstate(invalid="ignore", divide="ignore"):
                lo, hi = (li * s).astype(np.float32), (li / s).astype(np.float32)
                ok_e = (lo < lj) & (lj < hi)
                tol = 1e-6 * np.maximum(lj.astype(np.float64), 1e-30)
                # (a repeated draw gives li = lj = 0, which fails exactly on both sides)
                near_e = (lj > 0) & ((np.abs(lo.astype(np.float64) - lj) <= tol) |
                                     (np.abs(hi.astype(np.float64) - lj) <= tol))
            ok &= ok_e
            near |= near_e
            could &= ok_e | near_e
        near &= could
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
