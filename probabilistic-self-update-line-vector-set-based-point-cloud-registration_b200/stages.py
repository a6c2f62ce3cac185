"""Stage-level entry points of the C ABI on torch CUDA tensors (device pointers + current stream).

torch is plumbing here (device memory, streams); every computation happens in libpsulvsb_b200.so.
Reference loops each stage replaces are cited in include/psulvsb.h.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import capi


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dev(t: torch.Tensor) -> int:
    assert t.is_cuda and t.is_contiguous(), "expected a contiguous CUDA tensor"
    return t.data_ptr()


def to_device_points(pts) -> torch.Tensor:
    """3xN (numpy / tensor) -> device tensor [N,3] float64 == column-major 3xN as the C ABI wants."""
    a = np.ascontiguousarray(np.asarray(pts, dtype=np.float64).T)
    return torch.from_numpy(a).cuda()


def pack_points(d_pts: torch.Tensor, center=None) -> torch.Tensor:
    n = d_pts.shape[0]
    out = torch.empty((n, 4), dtype=torch.float32, device=d_pts.device)
    c = None
    if center is not None:
        c = (C.c_double * 3)(*[float(x) for x in center])
    capi.check(capi.lib().psulvsb_pack_points(_stream(), _dev(d_pts), n, c, _dev(out)))
    return out


def centre_and_bound(*point_sets):
    """Per-set box centres and the common max |coordinate| after centring (host, O(N))."""
    centres, bound = [], 0.0
    for p in point_sets:
        p = np.asarray(p, dtype=np.float64)
        lo, hi = p.min(axis=1), p.max(axis=1)
        centres.append(0.5 * (lo + hi))
        bound = max(bound, float((0.5 * (hi - lo)).max()))
    return centres, bound * (1 + 1e-6) + 1e-30


def consistency_mask(src, dst, beta: float, row_begin: int = 0, row_end: int | None = None, symmetrize: bool = False):
    """Returns dict(mask [n, stride] uint32 (int32 view), row_counts [n], border, stride, tensors...)."""
    src = np.asarray(src, dtype=np.float64)
    dst = np.asarray(dst, dtype=np.float64)
    n = src.shape[1]
    if row_end is None:
        row_end = n
    (cs, cd), bound = centre_and_bound(src, dst)
    d_src, d_dst = to_device_points(src), to_device_points(dst)
    f_src, f_dst = pack_points(d_src, cs), pack_points(d_dst, cd)
    stride = ((n + 31) // 32 + 3) // 4 * 4
    mask = torch.zeros((n, stride), dtype=torch.int32, device="cuda")
    counts = torch.zeros(n, dtype=torch.int32, device="cuda")
    border = torch.zeros(1, dtype=torch.int64, device="cuda")
    capi.check(capi.lib().psulvsb_consistency_mask_rows(_stream(), _dev(f_src), _dev(f_dst), _dev(d_src), _dev(d_dst),
                                                        n, row_begin, row_end, beta, bound, _dev(mask), stride,
                                                        _dev(counts), _dev(border)))
    if symmetrize:
        capi.check(capi.lib().psulvsb_mask_symmetrize(_stream(), _dev(mask), n, stride))
    torch.cuda.synchronize()
    return {"mask": mask, "row_counts": counts, "border": int(border.item()), "stride": stride, "n": n,
            "d_src": d_src, "d_dst": d_dst, "f_src": f_src, "f_dst": f_dst, "bound": bound, "centres": (cs, cd)}


def unpack_mask(mask: torch.Tensor, n: int) -> np.ndarray:
    """[n, stride] packed words -> [n, n] uint8 (bit j of row i = word j>>5, bit j&31)."""
    w = mask.cpu().numpy().view(np.uint32)
    bits = np.unpackbits(w.view(np.uint8), axis=1, bitorder="little")
    return bits[:, :n]


def compact_edges(mask: torch.Tensor, counts: torch.Tensor, n: int, stride: int):
    offsets = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    n_edges = torch.zeros(1, dtype=torch.int64, device="cuda")
    # first pass: sizes only
    capi.check(capi.lib().psulvsb_compact_edges(_stream(), _dev(mask), n, stride, _dev(counts), _dev(offsets), None, 0,
                                                _dev(n_edges)))
    total = int(n_edges.item())
    edges = torch.zeros((max(total, 1), 2), dtype=torch.int32, device="cuda")
    capi.check(capi.lib().psulvsb_compact_edges(_stream(), _dev(mask), n, stride, _dev(counts), _dev(offsets),
                                                _dev(edges), total, _dev(n_edges)))
    torch.cuda.synchronize()
    return edges[:total], offsets


def ratio_reduced_set(src, dst, pair_bins: bool = False):
    """Unknown-scale stage 1 of 3xN FP64 points -> dict(edges [n_edges, 2] int64 in reference order, n_edges,
    max_scale (final MaxScale), peak_bin, peak_height[, pair_bins: n (n - 1) / 2 uint32, row-major pair order])."""
    d_src, d_dst = to_device_points(src), to_device_points(dst)
    n = d_src.shape[0]
    L = capi.lib()
    bins = torch.zeros(max(n * (n - 1) // 2, 1), dtype=torch.int32, device="cuda") if pair_bins else None
    ne, ms, pk = C.c_ulonglong(0), C.c_double(0.0), (C.c_uint * 2)()
    capi.check(L.psulvsb_ratio_reduced_set(_stream(), _dev(d_src), _dev(d_dst), n, _dev(bins) if pair_bins else None,
                                           None, 0, C.byref(ne), C.byref(ms), pk))
    edges = torch.zeros((max(ne.value, 1), 2), dtype=torch.int32, device="cuda")
    capi.check(L.psulvsb_ratio_reduced_set(_stream(), _dev(d_src), _dev(d_dst), n, None, _dev(edges), ne.value,
                                           C.byref(ne), C.byref(ms), pk))
    out = {"edges": edges[:ne.value].cpu().numpy().astype(np.int64), "n_edges": ne.value, "max_scale": ms.value,
           "peak_height": int(pk[0]), "peak_bin": int(pk[1])}
    if pair_bins:
        out["pair_bins"] = bins[:n * (n - 1) // 2].cpu().numpy().view(np.uint32)
    return out


def sample(seed: int, domain: int, event: int, n: int, count: int, max_draws: int = 0):
    out = torch.zeros(max(count, 1), dtype=torch.int32, device="cuda")
    nbytes = capi.lib().psulvsb_sample_workspace_bytes(n, count, max_draws)
    work = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device="cuda")
    status = torch.zeros(1, dtype=torch.int64, device="cuda")
    capi.check(capi.lib().psulvsb_sample(_stream(), seed, domain, event, n, count, max_draws, _dev(out), _dev(work),
                                         _dev(status)))
    torch.cuda.synchronize()
    return out[:count].cpu().numpy().view(np.uint32).astype(np.int64), int(status.item())


def philox_fill(seed: int, domain: int, event: int, first_k: int, count: int) -> np.ndarray:
    out = torch.zeros(max(count, 1), dtype=torch.int32, device="cuda")
    capi.check(capi.lib().psulvsb_philox_fill(_stream(), seed, domain, event, first_k, count, _dev(out)))
    torch.cuda.synchronize()
    return out[:count].cpu().numpy().view(np.uint32)


def gnc_tls_rotation(d_src, d_dst, d_edges, noise_bound, max_iterations=100, gnc_factor=1.4, cost_threshold=0.005,
                     R_init=None, inv_scale=1.0):
    K = d_edges.shape[0]
    w = torch.zeros(max(K, 1), dtype=torch.float64, device="cuda")
    R = torch.zeros(9, dtype=torch.float64, device="cuda")
    inl = torch.zeros(max(K, 1), dtype=torch.uint8, device="cuda")
    info = torch.zeros(4, dtype=torch.int32, device="cuda")
    cost = torch.zeros(1, dtype=torch.float64, device="cuda")
    ri = None
    if R_init is not None:
        ri = torch.from_numpy(np.asfortranarray(np.asarray(R_init, dtype=np.float64)).ravel(order="F").copy()).cuda()
    capi.check(capi.lib().psulvsb_gnc_tls_rotation(_stream(), _dev(d_src), _dev(d_dst), _dev(d_edges), K, inv_scale,
                                                   noise_bound, max_iterations, gnc_factor, cost_threshold,
                                                   _dev(ri) if ri is not None else None, _dev(w), _dev(R), _dev(inl),
                                                   _dev(info), _dev(cost)))
    torch.cuda.synchronize()
    i = info.cpu().numpy()
    return (R.cpu().numpy().reshape(3, 3, order="F"), inl[:K].cpu().numpy(), int(i[0]), float(cost.item()), int(i[1]))


def gnc_tls_rotation_batch(d_src, d_dst, d_edges, noise_bound, max_iterations=100, gnc_factor=1.4, cost_threshold=0.005,
                           cluster: int = 0, lv_scratch: bool = True, parking: bool = True):
    """d_edges: [B, K, 2] int32 on the device, one basic subset per job over the shared points ->
    (R [B, 3, 3], inlier masks [B, K], iterations [B], inlier counts [B])."""
    B, K = int(d_edges.shape[0]), int(d_edges.shape[1])
    w = torch.zeros(B * K, dtype=torch.float64, device="cuda")
    lv = torch.zeros(B * 6 * K, dtype=torch.float64, device="cuda") if lv_scratch else None
    perm = torch.zeros(B * 2 * K, dtype=torch.int32, device="cuda") if (lv_scratch and parking) else None
    R = torch.zeros(B * 9, dtype=torch.float64, device="cuda")
    inl = torch.zeros(B * K, dtype=torch.uint8, device="cuda")
    info = torch.zeros(B * 4, dtype=torch.int32, device="cuda")
    capi.check(capi.lib().psulvsb_gnc_tls_rotation_batch(
        _stream(), _dev(d_src), _dev(d_dst), int(d_src.shape[0]), _dev(d_edges), K, B, noise_bound, max_iterations,
        gnc_factor, cost_threshold, cluster, _dev(w), _dev(lv) if lv is not None else None, K,
        _dev(perm) if perm is not None else None, _dev(R), _dev(inl), _dev(info), None))
    torch.cuda.synchronize()
    i = info.cpu().numpy().reshape(B, 4)
    Rn = R.cpu().numpy().reshape(B, 3, 3).transpose(0, 2, 1)  # column-major -> [b][r][c]
    return Rn, inl.cpu().numpy().reshape(B, K), i[:, 0].copy(), i[:, 1].copy()


def kabsch_batch(d_src, d_dst, d_edges, d_sets, k: int, want_t: bool = True):
    n_hyp = d_sets.numel() // k
    R = torch.zeros((n_hyp, 9), dtype=torch.float64, device="cuda")
    t = torch.zeros((n_hyp, 3), dtype=torch.float64, device="cuda") if want_t else None
    capi.check(capi.lib().psulvsb_kabsch_batch(_stream(), _dev(d_src), _dev(d_dst), _dev(d_edges), _dev(d_sets), k,
                                               n_hyp, _dev(R), _dev(t) if want_t else None))
    return R, t


def tls_translation(d_src, d_dst, d_flags, scale, R, noise, last_best=None):
    n = d_src.shape[0]
    Rd = torch.from_numpy(np.asarray(R, dtype=np.float64).ravel(order="F").copy()).cuda()
    lb = None if last_best is None else torch.from_numpy(np.asarray(last_best, dtype=np.float64).copy()).cuda()
    t = torch.zeros(3, dtype=torch.float64, device="cuda")
    npts = torch.zeros(1, dtype=torch.int32, device="cuda")
    capi.check(capi.lib().psulvsb_tls_translation(_stream(), _dev(d_src), _dev(d_dst), _dev(d_flags), n, scale,
                                                  _dev(Rd), noise, _dev(lb) if lb is not None else None, _dev(t),
                                                  _dev(npts)))
    torch.cuda.synchronize()
    return t.cpu().numpy(), int(npts.item())


def score_batch(f_src, f_dst, d_src, d_dst, d_hyp, scale, tau, bound, centres, hyp_begin: int = 0, d_best=None):
    n = d_src.shape[0]
    n_hyp = d_hyp.shape[0]
    counts = torch.zeros(n_hyp, dtype=torch.int32, device="cuda")
    if d_best is None:
        d_best = torch.zeros(1, dtype=torch.int64, device="cuda")
    border = torch.zeros(1, dtype=torch.int64, device="cuda")
    cs = (C.c_double * 3)(*[float(x) for x in centres[0]])
    cd = (C.c_double * 3)(*[float(x) for x in centres[1]])
    capi.check(capi.lib().psulvsb_score_batch(_stream(), _dev(f_src), _dev(f_dst), _dev(d_src), _dev(d_dst), n,
                                              _dev(d_hyp), n_hyp, hyp_begin, scale, tau, bound, cs, cd, _dev(counts),
                                              _dev(d_best), _dev(border)))
    return counts, d_best, border


def decode_best(packed: int):
    """(count << 32) | (0xFFFFFFFF - hypothesis id) -> (count, id)."""
    packed &= (1 << 64) - 1
    return packed >> 32, 0xFFFFFFFF - (packed & 0xFFFFFFFF)


def score_one(d_src, d_dst, scale, R, t, tau):
    n = d_src.shape[0]
    Rd = torch.from_numpy(np.asarray(R, dtype=np.float64).ravel(order="F").copy()).cuda()
    td = torch.from_numpy(np.asarray(t, dtype=np.float64).copy()).cuda()
    inl = torch.zeros(n, dtype=torch.uint8, device="cuda")
    res = torch.zeros(n, dtype=torch.float64, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    capi.check(capi.lib().psulvsb_score_one(_stream(), _dev(d_src), _dev(d_dst), n, scale, _dev(Rd), _dev(td), tau,
                                            _dev(inl), _dev(res), _dev(cnt)))
    torch.cuda.synchronize()
    return int(cnt.item()), inl.cpu().numpy(), res.cpu().numpy()


def max_clique(edges, n_vertices: int, exact: bool = True):
    """edges: [E, 2] int array -> (sorted clique vertex ids, size, proven).  exact=False: greedy lower bound only."""
    L = capi.lib()
    e = torch.from_numpy(np.ascontiguousarray(edges, dtype=np.int32).reshape(-1, 2)).cuda()
    adj = torch.empty(int(L.psulvsb_max_clique_scratch_words(n_vertices)), dtype=torch.int32, device="cuda")
    flags = torch.zeros(n_vertices, dtype=torch.uint8, device="cuda")
    size = torch.zeros(2, dtype=torch.int32, device="cuda")
    capi.check(L.psulvsb_max_clique(_stream(), _dev(e) if e.numel() else None, e.shape[0], n_vertices, _dev(adj),
                                    _dev(flags), _dev(size), 1 if exact else 0))
    torch.cuda.synchronize()
    sz = size.cpu().numpy()
    return np.flatnonzero(flags.cpu().numpy()), int(sz[0]), bool(sz[1]) if exact else False


def greedy_clique(edges, n_vertices: int):
    got, size, _ = max_clique(edges, n_vertices, exact=False)
    return got, size
