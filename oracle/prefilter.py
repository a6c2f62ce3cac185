"""numpy restatement of the reference driver's normal-angle histogram pre-filter.

TEST INFRASTRUCTURE ONLY.  Follows examples/teaser_cpp_ply/PSULVSB.cc:87-172 (histogram_outlier_removal)
and :174-188 (mask_filter) statement by statement; the reference has no fixture for it, so parity for the
pre-filter is "product vs this restatement" (unpinned by the reference's own tests).
Positions taken where the reference is undefined (same as the product, csrc/host_io.cpp): sigma == 0 -> one
bin; an angle exactly on the upper edge of the last bin goes into the last bin.
"""
import math

import numpy as np


def histogram_outlier_removal(src_normals, tgt_normals):
    n = src_normals.shape[1]
    keep = np.zeros(n, dtype=np.int32)
    all_angles = np.full(n, -1.0)
    remain = []
    o_max, o_min, s = 0.0, float(2**31 - 1), 0.0
    for i in range(n):
        a, b = src_normals[:, i], tgt_normals[:, i]
        za, zb = (a[0] * a[0] + a[1] * a[1]) + a[2] * a[2], (b[0] * b[0] + b[1] * b[1]) + b[2] * b[2]
        if za > 0:
            a = a / math.sqrt(za)
        if zb > 0:
            b = b / math.sqrt(zb)
        c = (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]
        # std::max(-1.0, std::min(1.0, c)) (PSULVSB.cc:100): std::min(1.0, NaN) returns its FIRST argument, so a
        # NaN normal (PCL's answer for a degenerate neighbourhood) yields cos = 1, angle 0 -- it is NOT skipped
        # by the isnan test that follows in the reference
        c = 1.0 if math.isnan(c) else max(-1.0, min(1.0, c))
        ang = math.acos(c) * 180.0 / math.pi
        if math.isnan(ang):
            continue
        remain.append(ang)
        all_angles[i] = ang
        o_min, o_max = min(ang, o_min), max(ang, o_max)
        s += ang
    if not remain:
        return keep, 0
    cnt = float(len(remain))
    mean = s / cnt
    sq = 0.0
    for d in remain:
        sq += (d - mean) ** 2
    sd = math.sqrt(sq / cnt)
    width = 3.49 * sd / cnt ** (1.0 / 3.0)
    ok = width > 0 and math.isfinite(width)
    size = max(1, int(math.ceil((o_max - o_min) / width))) if ok else 1
    hist = [[] for _ in range(size)]
    peak_id, peak_h = 0, 0
    for i in range(n):
        if all_angles[i] == -1:
            continue
        b = int((all_angles[i] - o_min) / width) if ok else 0
        b = min(max(b, 0), size - 1)
        hist[b].append(i)
        if len(hist[b]) > peak_h:
            peak_h, peak_id = len(hist[b]), b
    hmean = sum(float(len(h)) for h in hist) / size
    hvar = 0.0
    for h in hist:
        hvar += (len(h) - hmean) ** 2
    thr = hmean + math.sqrt(hvar / size)
    rem = 0
    for i, h in enumerate(hist):
        if abs(i - peak_id) > 2:
            for j in h:
                keep[j] = -1
        if len(h) > thr:
            for j in h:
                keep[j] = 1
                rem += 1
    return keep, rem


def mask_filter(src, tgt, keep):
    idx = np.flatnonzero(keep == 1)
    rm = np.full(src.shape[1], -1, dtype=np.int32)
    rm[idx] = np.arange(idx.size, dtype=np.int32)
    return np.asfortranarray(src[:, idx]), np.asfortranarray(tgt[:, idx]), rm


def knn_sqdist32(Pf, rows):
    """FP32 squared distances from the points `rows` to all points, as k6_normals.cu forms them:
    fmaf(dz, dz, fmaf(dy, dy, dx * dx)) with d = p_j - p_i."""
    from oracle.features import fma32

    d = [(Pf[c][None, :] - Pf[c][rows][:, None]).astype(np.float32) for c in range(3)]
    return fma32(d[2], d[2], fma32(d[1], d[1], d[0] * d[0]))


def knn_pca_normals(points, k=20, viewpoint=(0.0, 0.0, 0.0), return_fragile=False, block=256):
    """Restatement of what PSULVSB.cc:35-85 asks PCL for: for every point the k nearest neighbours (itself
    included), the eigenvector of the smallest eigenvalue of their covariance, flipped towards the viewpoint.

    As the kernel decides it: the fused FP32 distance (knn_sqdist32), ties to the lower index, all n points when
    n < k, NaN when fewer than 3 points remain.  With return_fragile, also a per-point flag for results that
    summation order may decide: the k-th and (k+1)-th distances within 1e-6 relative (an exact tie is decided the
    same way on both sides), the two smallest eigenvalues within 1e-6 relative, or the normal within 1e-7 of
    perpendicular to the viewpoint direction."""
    P = np.asarray(points, dtype=np.float64)
    n = P.shape[1]
    Pf = P.astype(np.float32)
    out = np.full((3, n), np.nan)
    frag = np.zeros(n, dtype=bool)
    m = min(k, n)
    if m >= 3:
        vp = np.asarray(viewpoint, dtype=np.float64)
        idx = np.zeros((n, m), dtype=np.int64)
        for r0 in range(0, n, block):
            rows = np.arange(r0, min(n, r0 + block))
            d = knn_sqdist32(Pf, rows)
            # key = (distance bits, index): non-negative float32 bits keep their order, the index breaks ties
            key = (d.view(np.uint32).astype(np.uint64) << np.uint64(32)) | np.arange(n, dtype=np.uint64)[None, :]
            if n > m:
                key = np.partition(key, m, axis=1)[:, :m + 1]
            key = np.sort(key, axis=1)
            idx[rows] = (key[:, :m] & np.uint64(0xFFFFFFFF)).astype(np.int64)
            if n > m:
                dk = (key[:, m - 1] >> np.uint64(32)).astype(np.uint32).view(np.float32).astype(np.float64)
                dk1 = (key[:, m] >> np.uint64(32)).astype(np.uint32).view(np.float32).astype(np.float64)
                frag[rows] = (dk1 != dk) & (dk1 - dk <= 1e-6 * dk1)
        nb = P[:, idx].transpose(1, 2, 0)                       # [n, m, 3]
        dev = nb - nb.mean(axis=1, keepdims=True)
        cov = np.einsum("nka,nkb->nab", dev, dev)
        w, v = np.linalg.eigh(cov)
        nv = v[:, :, 0]
        side = ((vp[None, :] - P.T) * nv).sum(axis=1)
        nv[side < 0] *= -1
        out = np.ascontiguousarray(nv.T)
        scale = np.maximum(np.abs(w[:, 2]), 1e-300)
        frag |= (np.abs(w[:, 1] - w[:, 0]) <= 1e-6 * scale)
        frag |= np.abs(side) <= 1e-7 * np.linalg.norm(vp[None, :] - P.T, axis=1)
    return (out, frag) if return_fragile else out
