"""Refinement of a registration on the raw clouds: rigid ICP, point-to-point, point-to-plane or generalized ICP, on the
GPU.

What users of TEASER++ run after the global solve (Open3D's registration_icp, PCL's IterativeClosestPoint), through the
C ABI (include/psulvsb.h, csrc/k9_icp.cu; DESIGN.md section 11).  `icp` takes host arrays; `icp_device` takes CUDA
tensors [N, 3] float64 (== column-major 3xN) and runs on the current stream.  `icp_batch` / `icp_batch_device` refine
B independent pairs with shared parameters in one call; pair b's result is bit-identical to `icp` on that pair alone.
`gicp`, `gicp_device`, `gicp_batch` and `gicp_batch_device` are the same four calls with generalized ICP's update
(plane-to-plane; Open3D's registration_generalized_icp); they need the normals of both clouds, for instance the radius
or hybrid normals of `features.normals` / `features.normals_batch` (on the grid, without descriptors), the radius
normals `features.fpfh` returns or the k-NN normals of `stages.estimate_normals`.
Convention: q ~ R p + t.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import capi

CONVERGED, MAX_ITERATIONS, NO_UPDATE = 0, 1, 2


@dataclass
class IcpResult:
    R: np.ndarray                  # 3x3
    t: np.ndarray                  # 3
    fitness: float                 # correspondences / n_src at the final T
    inlier_rmse: float
    n_correspondences: int
    iterations: int                # updates applied
    status: int                    # CONVERGED, MAX_ITERATIONS or NO_UPDATE
    correspondences: object        # [n_src] int32 target index or -1 (numpy; a CUDA tensor from icp_device)
    trace: Optional[dict] = None   # per evaluation k = 0 .. iterations: R [K, 3, 3], t, fitness, inlier_rmse, n_corr


def _cm(a, what) -> np.ndarray:
    a = np.asarray(a, dtype=np.float64)
    if a.ndim != 2 or a.shape[0] != 3:
        raise ValueError(f"{what}: expected a 3xN matrix, got {a.shape}")
    return np.asfortranarray(a)


def _params(d, point_to_plane, max_iterations, relative_fitness, relative_rmse) -> capi.IcpParams:
    p = capi.IcpParams()
    capi.lib().psulvsb_icp_default_params(C.byref(p))
    p.max_correspondence_distance = float(d)
    p.point_to_plane = int(bool(point_to_plane))
    p.max_iterations = int(max_iterations)
    p.relative_fitness = float(relative_fitness)
    p.relative_rmse = float(relative_rmse)
    return p


def _transform(R0, t0):
    R = np.asarray(R0, dtype=np.float64).reshape(3, 3)
    t = np.asarray(t0, dtype=np.float64).reshape(3)
    return (C.c_double * 9)(*R.flatten(order="F")), (C.c_double * 3)(*t)


def _trace(records, n) -> dict:
    recs = [records[k] for k in range(n)]
    return {"R": np.array([np.array(r.rotation[:]).reshape(3, 3, order="F") for r in recs]).reshape(n, 3, 3),
            "t": np.array([r.translation[:] for r in recs]).reshape(n, 3),
            "fitness": np.array([r.fitness for r in recs]),
            "inlier_rmse": np.array([r.inlier_rmse for r in recs]),
            "n_correspondences": np.array([r.n_correspondences for r in recs], dtype=np.int64)}


def _result(res: capi.IcpResult, records, corr) -> IcpResult:
    return IcpResult(R=np.array(res.rotation[:]).reshape(3, 3, order="F"), t=np.array(res.translation[:]),
                     fitness=res.fitness, inlier_rmse=res.inlier_rmse, n_correspondences=res.n_correspondences,
                     iterations=res.iterations, status=res.status, correspondences=corr,
                     trace=None if records is None else _trace(records, res.iterations + 1))


def icp(src, tgt, R0, t0, max_correspondence_distance: float, *, target_normals=None, point_to_plane: bool = False,
        max_iterations: int = 30, relative_fitness: float = 1e-6, relative_rmse: float = 1e-6,
        trace: bool = False) -> IcpResult:
    """psulvsb_icp_host: refine (R0, t0) so that tgt ~ R src + t.  src 3 x n_s, tgt 3 x n_t; target_normals 3 x n_t is
    required for point-to-plane (a target point with a non-finite normal is then no candidate)."""
    s, q = _cm(src, "src"), _cm(tgt, "tgt")
    nrm = None
    if target_normals is not None:
        nrm = _cm(target_normals, "target_normals")
        if nrm.shape != q.shape:
            raise ValueError("one normal per target point is needed")
    p = _params(max_correspondence_distance, point_to_plane, max_iterations, relative_fitness, relative_rmse)
    R, t = _transform(R0, t0)
    res = capi.IcpResult()
    records = (capi.IcpIteration * (max(int(max_iterations), 0) + 1))() if trace else None
    corr = np.empty(s.shape[1], dtype=np.int32)
    capi.check(capi.lib().psulvsb_icp_host(s.ctypes.data, s.shape[1], q.ctypes.data, q.shape[1],
                                           None if nrm is None else nrm.ctypes.data, C.byref(p), R, t, C.byref(res),
                                           records, corr.ctypes.data))
    return _result(res, records, corr)


def icp_device(d_src, d_tgt, R0, t0, max_correspondence_distance: float, *, d_target_normals=None,
               point_to_plane: bool = False, max_iterations: int = 30, relative_fitness: float = 1e-6,
               relative_rmse: float = 1e-6, trace: bool = False, work=None) -> IcpResult:
    """psulvsb_icp on CUDA tensors [n, 3] float64 and the current stream.  The small result (and the trace) are read
    back, which waits for the stream; the correspondences stay on the device.  `work`: an optional uint8 CUDA tensor
    of at least psulvsb_icp_workspace_bytes(n_s, n_t) bytes to reuse."""
    import torch

    from .stages import _dev, _stream

    ns, nt = d_src.shape[0], d_tgt.shape[0]
    dev = d_src.device
    if work is None:
        work = torch.empty(max(1, capi.lib().psulvsb_icp_workspace_bytes(ns, nt)), dtype=torch.uint8, device=dev)
    elif work.numel() < capi.lib().psulvsb_icp_workspace_bytes(ns, nt):
        raise ValueError("work is smaller than psulvsb_icp_workspace_bytes(n_s, n_t)")
    nrec = max(int(max_iterations), 0) + 1
    out = torch.empty(C.sizeof(capi.IcpResult), dtype=torch.uint8, device=dev)
    rec = torch.empty(nrec * C.sizeof(capi.IcpIteration) if trace else 1, dtype=torch.uint8, device=dev)
    corr = torch.empty(max(ns, 1), dtype=torch.int32, device=dev)
    p = _params(max_correspondence_distance, point_to_plane, max_iterations, relative_fitness, relative_rmse)
    R, t = _transform(R0, t0)
    capi.check(capi.lib().psulvsb_icp(_stream(), _dev(d_src) if ns else None, ns, _dev(d_tgt) if nt else None, nt,
                                      None if d_target_normals is None else _dev(d_target_normals), C.byref(p), R, t,
                                      _dev(work), _dev(out), _dev(rec) if trace else None, _dev(corr)))
    res = capi.IcpResult.from_buffer_copy(out.cpu().numpy().tobytes())
    records = None
    if trace:
        records = (capi.IcpIteration * nrec).from_buffer_copy(rec.cpu().numpy().tobytes())
    return _result(res, records, corr[:ns])


def _batch_transforms(R0s, t0s, B):
    R = np.asarray(R0s, dtype=np.float64).reshape(B, 3, 3)
    t = np.asarray(t0s, dtype=np.float64).reshape(B, 3)
    return R, t


def _batch_pairs(ptrs, sizes, R, t):
    """psulvsb_icp_pair_t[B] from (src, tgt, normals) pointers and (n_s, n_t) per pair."""
    pairs = (capi.IcpPair * max(len(sizes), 1))()
    for b, ((ps, pt, pn), (ns, nt)) in enumerate(zip(ptrs, sizes)):
        pairs[b].src, pairs[b].n_s, pairs[b].tgt, pairs[b].n_t, pairs[b].tgt_normals = ps, ns, pt, nt, pn
        pairs[b].R0[:] = R[b].flatten(order="F").tolist()
        pairs[b].t0[:] = t[b].tolist()
    return pairs


def _batch_results(res, records, nrec, corr, sizes):
    out, o = [], 0
    for b, (ns, _) in enumerate(sizes):
        recs = None if records is None else records[b * nrec:(b + 1) * nrec]
        out.append(_result(res[b], recs, corr[o:o + ns]))
        o += ns
    return out


def icp_batch(srcs, tgts, R0s, t0s, max_correspondence_distance: float, *, target_normals=None,
              point_to_plane: bool = False, max_iterations: int = 30, relative_fitness: float = 1e-6,
              relative_rmse: float = 1e-6, trace: bool = False) -> list:
    """psulvsb_icp_batch_host: refine B pairs in one call with shared parameters.  srcs, tgts (and target_normals, for
    point-to-plane): sequences of 3 x n arrays; R0s [B, 3, 3], t0s [B, 3].  Returns one IcpResult per pair, each equal bit
    for bit to `icp` on that pair alone."""
    s = [_cm(a, "src") for a in srcs]
    q = [_cm(a, "tgt") for a in tgts]
    B = len(s)
    if len(q) != B:
        raise ValueError(f"{B} sources and {len(q)} targets")
    nrm = [None] * B
    if target_normals is not None:                            # None for a pair without target points
        nrm = [None if a is None else _cm(a, "target_normals") for a in target_normals]
        if len(nrm) != B or any(n is not None and n.shape != t.shape for n, t in zip(nrm, q)):
            raise ValueError("one normal per target point is needed")
    R, t = _batch_transforms(R0s, t0s, B)
    sizes = [(a.shape[1], b.shape[1]) for a, b in zip(s, q)]
    pairs = _batch_pairs([(a.ctypes.data, b.ctypes.data, None if n is None else n.ctypes.data)
                          for a, b, n in zip(s, q, nrm)], sizes, R, t)
    p = _params(max_correspondence_distance, point_to_plane, max_iterations, relative_fitness, relative_rmse)
    nrec = max(int(max_iterations), 0) + 1
    res = (capi.IcpResult * max(B, 1))()
    records = (capi.IcpIteration * (B * nrec))() if trace and B else None
    corr = np.empty(sum(ns for ns, _ in sizes), dtype=np.int32)
    capi.check(capi.lib().psulvsb_icp_batch_host(pairs, B, C.byref(p), res, records, corr.ctypes.data))
    return _batch_results(res, records, nrec, corr, sizes)


def icp_batch_device(d_srcs, d_tgts, R0s, t0s, max_correspondence_distance: float, *, d_target_normals=None,
                     point_to_plane: bool = False, max_iterations: int = 30, relative_fitness: float = 1e-6,
                     relative_rmse: float = 1e-6, trace: bool = False, work=None) -> list:
    """psulvsb_icp_batch on sequences of CUDA tensors [n, 3] float64 and the current stream.  The small results (and the
    traces) are read back, which waits for the stream; the correspondences stay on the device as views into one tensor.
    `work`: an optional uint8 CUDA tensor of at least psulvsb_icp_batch_workspace_bytes bytes to reuse."""
    import torch

    from .stages import _dev, _stream

    B = len(d_srcs)
    if len(d_tgts) != B:
        raise ValueError(f"{B} sources and {len(d_tgts)} targets")
    nrm = [None] * B if d_target_normals is None else list(d_target_normals)
    if len(nrm) != B:
        raise ValueError(f"{B} targets and {len(nrm)} normal sets")
    R, t = _batch_transforms(R0s, t0s, B)
    sizes = [(a.shape[0], b.shape[0]) for a, b in zip(d_srcs, d_tgts)]
    pairs = _batch_pairs([(_dev(a) if a.shape[0] else None, _dev(b) if b.shape[0] else None,
                           None if n is None else _dev(n)) for a, b, n in zip(d_srcs, d_tgts, nrm)], sizes, R, t)
    L = capi.lib()
    nbytes = L.psulvsb_icp_batch_workspace_bytes(pairs, B)
    dev = d_srcs[0].device if B else torch.device("cuda")
    if work is None:
        work = torch.empty(max(1, nbytes), dtype=torch.uint8, device=dev)
    elif work.numel() < nbytes:
        raise ValueError("work is smaller than psulvsb_icp_batch_workspace_bytes(pairs, B)")
    nrec = max(int(max_iterations), 0) + 1
    out = torch.empty(max(B, 1) * C.sizeof(capi.IcpResult), dtype=torch.uint8, device=dev)
    rec = torch.empty(B * nrec * C.sizeof(capi.IcpIteration) if trace and B else 1, dtype=torch.uint8, device=dev)
    corr = torch.empty(max(sum(ns for ns, _ in sizes), 1), dtype=torch.int32, device=dev)
    p = _params(max_correspondence_distance, point_to_plane, max_iterations, relative_fitness, relative_rmse)
    capi.check(L.psulvsb_icp_batch(_stream(), pairs, B, C.byref(p), _dev(work), _dev(out),
                                   _dev(rec) if trace else None, _dev(corr)))
    res = (capi.IcpResult * max(B, 1)).from_buffer_copy(out.cpu().numpy().tobytes())
    records = None
    if trace and B:
        records = (capi.IcpIteration * (B * nrec)).from_buffer_copy(rec.cpu().numpy().tobytes())
    return _batch_results(res, records, nrec, corr, sizes)


def _normals(n, cloud, what) -> np.ndarray:
    n = _cm(n, what)
    if n.shape != cloud.shape:
        raise ValueError(f"{what}: one normal per point is needed, got {n.shape} for {cloud.shape}")
    return n


def gicp(src, tgt, src_normals, tgt_normals, R0, t0, max_correspondence_distance: float, *, epsilon: float = 1e-3,
         max_iterations: int = 30, relative_fitness: float = 1e-6, relative_rmse: float = 1e-6,
         trace: bool = False) -> IcpResult:
    """psulvsb_gicp_host: refine (R0, t0) so that tgt ~ R src + t with generalized ICP.  src, src_normals 3 x n_s; tgt,
    tgt_normals 3 x n_t.  Each point's covariance is I - (1 - epsilon) n n^T (a non-finite or zero normal gives I, and
    the point stays a candidate); 0 < epsilon <= 1, Open3D's default 1e-3."""
    s, q = _cm(src, "src"), _cm(tgt, "tgt")
    ns, nt = _normals(src_normals, s, "src_normals"), _normals(tgt_normals, q, "tgt_normals")
    p = _params(max_correspondence_distance, False, max_iterations, relative_fitness, relative_rmse)
    R, t = _transform(R0, t0)
    res = capi.IcpResult()
    records = (capi.IcpIteration * (max(int(max_iterations), 0) + 1))() if trace else None
    corr = np.empty(s.shape[1], dtype=np.int32)
    capi.check(capi.lib().psulvsb_gicp_host(s.ctypes.data, s.shape[1], ns.ctypes.data, q.ctypes.data, q.shape[1],
                                            nt.ctypes.data, C.byref(p), float(epsilon), R, t, C.byref(res), records,
                                            corr.ctypes.data))
    return _result(res, records, corr)


def gicp_device(d_src, d_tgt, d_src_normals, d_tgt_normals, R0, t0, max_correspondence_distance: float, *,
                epsilon: float = 1e-3, max_iterations: int = 30, relative_fitness: float = 1e-6,
                relative_rmse: float = 1e-6, trace: bool = False, work=None) -> IcpResult:
    """psulvsb_gicp on CUDA tensors [n, 3] float64 (normals the same shape as their clouds) and the current stream; the
    outputs as `icp_device`.  `work`: an optional uint8 CUDA tensor of at least psulvsb_icp_workspace_bytes(n_s, n_t)
    bytes to reuse."""
    import torch

    from .stages import _dev, _stream

    ns, nt = d_src.shape[0], d_tgt.shape[0]
    if tuple(d_src_normals.shape) != tuple(d_src.shape) or tuple(d_tgt_normals.shape) != tuple(d_tgt.shape):
        raise ValueError("one normal per point is needed")
    dev = d_src.device
    if work is None:
        work = torch.empty(max(1, capi.lib().psulvsb_icp_workspace_bytes(ns, nt)), dtype=torch.uint8, device=dev)
    elif work.numel() < capi.lib().psulvsb_icp_workspace_bytes(ns, nt):
        raise ValueError("work is smaller than psulvsb_icp_workspace_bytes(n_s, n_t)")
    nrec = max(int(max_iterations), 0) + 1
    out = torch.empty(C.sizeof(capi.IcpResult), dtype=torch.uint8, device=dev)
    rec = torch.empty(nrec * C.sizeof(capi.IcpIteration) if trace else 1, dtype=torch.uint8, device=dev)
    corr = torch.empty(max(ns, 1), dtype=torch.int32, device=dev)
    p = _params(max_correspondence_distance, False, max_iterations, relative_fitness, relative_rmse)
    R, t = _transform(R0, t0)
    capi.check(capi.lib().psulvsb_gicp(_stream(), _dev(d_src) if ns else None, ns,
                                       _dev(d_src_normals) if ns else None, _dev(d_tgt) if nt else None, nt,
                                       _dev(d_tgt_normals) if nt else None, C.byref(p), float(epsilon), R, t,
                                       _dev(work), _dev(out), _dev(rec) if trace else None, _dev(corr)))
    res = capi.IcpResult.from_buffer_copy(out.cpu().numpy().tobytes())
    records = None
    if trace:
        records = (capi.IcpIteration * nrec).from_buffer_copy(rec.cpu().numpy().tobytes())
    return _result(res, records, corr[:ns])


def _gicp_pairs(ptrs, sizes, R, t):
    """psulvsb_gicp_pair_t[B] from (src, tgt, src_normals, tgt_normals) pointers and (n_s, n_t) per pair."""
    pairs = (capi.GicpPair * max(len(sizes), 1))()
    for b, ((ps, pt, psn, ptn), (ns, nt)) in enumerate(zip(ptrs, sizes)):
        q = pairs[b]
        q.src, q.n_s, q.tgt, q.n_t, q.src_normals, q.tgt_normals = ps, ns, pt, nt, psn, ptn
        q.R0[:] = R[b].flatten(order="F").tolist()
        q.t0[:] = t[b].tolist()
    return pairs


def gicp_batch(srcs, tgts, src_normals, tgt_normals, R0s, t0s, max_correspondence_distance: float, *,
               epsilon: float = 1e-3, max_iterations: int = 30, relative_fitness: float = 1e-6,
               relative_rmse: float = 1e-6, trace: bool = False) -> list:
    """psulvsb_gicp_batch_host: refine B pairs with generalized ICP in one call with shared parameters.  srcs, tgts,
    src_normals, tgt_normals: sequences of 3 x n arrays; R0s [B, 3, 3], t0s [B, 3].  Returns one IcpResult per pair,
    each equal bit for bit to `gicp` on that pair alone."""
    s = [_cm(a, "src") for a in srcs]
    q = [_cm(a, "tgt") for a in tgts]
    B = len(s)
    if len(q) != B or len(src_normals) != B or len(tgt_normals) != B:
        raise ValueError(f"{B} sources, {len(q)} targets, {len(src_normals)} and {len(tgt_normals)} normal sets")
    sn = [_normals(n, c, "src_normals") for n, c in zip(src_normals, s)]
    tn = [_normals(n, c, "tgt_normals") for n, c in zip(tgt_normals, q)]
    R, t = _batch_transforms(R0s, t0s, B)
    sizes = [(a.shape[1], b.shape[1]) for a, b in zip(s, q)]
    pairs = _gicp_pairs([(a.ctypes.data, b.ctypes.data, c.ctypes.data, d.ctypes.data)
                         for a, b, c, d in zip(s, q, sn, tn)], sizes, R, t)
    p = _params(max_correspondence_distance, False, max_iterations, relative_fitness, relative_rmse)
    nrec = max(int(max_iterations), 0) + 1
    res = (capi.IcpResult * max(B, 1))()
    records = (capi.IcpIteration * (B * nrec))() if trace and B else None
    corr = np.empty(sum(ns for ns, _ in sizes), dtype=np.int32)
    capi.check(capi.lib().psulvsb_gicp_batch_host(pairs, B, C.byref(p), float(epsilon), res, records,
                                                  corr.ctypes.data))
    return _batch_results(res, records, nrec, corr, sizes)


def gicp_batch_device(d_srcs, d_tgts, d_src_normals, d_tgt_normals, R0s, t0s, max_correspondence_distance: float, *,
                      epsilon: float = 1e-3, max_iterations: int = 30, relative_fitness: float = 1e-6,
                      relative_rmse: float = 1e-6, trace: bool = False, work=None) -> list:
    """psulvsb_gicp_batch on sequences of CUDA tensors [n, 3] float64 and the current stream; the outputs as
    `icp_batch_device`.  `work`: an optional uint8 CUDA tensor of at least psulvsb_gicp_batch_workspace_bytes bytes."""
    import torch

    from .stages import _dev, _stream

    B = len(d_srcs)
    if len(d_tgts) != B or len(d_src_normals) != B or len(d_tgt_normals) != B:
        raise ValueError(f"{B} sources, {len(d_tgts)} targets, {len(d_src_normals)} and {len(d_tgt_normals)} normal "
                         "sets")
    for c, n in list(zip(d_srcs, d_src_normals)) + list(zip(d_tgts, d_tgt_normals)):
        if tuple(n.shape) != tuple(c.shape):
            raise ValueError("one normal per point is needed")
    R, t = _batch_transforms(R0s, t0s, B)
    sizes = [(a.shape[0], b.shape[0]) for a, b in zip(d_srcs, d_tgts)]
    ptr = lambda x: _dev(x) if x.shape[0] else None                  # noqa: E731
    pairs = _gicp_pairs([(ptr(a), ptr(b), ptr(c), ptr(d)) for a, b, c, d in
                         zip(d_srcs, d_tgts, d_src_normals, d_tgt_normals)], sizes, R, t)
    L = capi.lib()
    nbytes = L.psulvsb_gicp_batch_workspace_bytes(pairs, B)
    dev = d_srcs[0].device if B else torch.device("cuda")
    if work is None:
        work = torch.empty(max(1, nbytes), dtype=torch.uint8, device=dev)
    elif work.numel() < nbytes:
        raise ValueError("work is smaller than psulvsb_gicp_batch_workspace_bytes(pairs, B)")
    nrec = max(int(max_iterations), 0) + 1
    out = torch.empty(max(B, 1) * C.sizeof(capi.IcpResult), dtype=torch.uint8, device=dev)
    rec = torch.empty(B * nrec * C.sizeof(capi.IcpIteration) if trace and B else 1, dtype=torch.uint8, device=dev)
    corr = torch.empty(max(sum(ns for ns, _ in sizes), 1), dtype=torch.int32, device=dev)
    p = _params(max_correspondence_distance, False, max_iterations, relative_fitness, relative_rmse)
    capi.check(L.psulvsb_gicp_batch(_stream(), pairs, B, C.byref(p), float(epsilon), _dev(work), _dev(out),
                                    _dev(rec) if trace else None, _dev(corr)))
    res = (capi.IcpResult * max(B, 1)).from_buffer_copy(out.cpu().numpy().tobytes())
    records = None
    if trace and B:
        records = (capi.IcpIteration * (B * nrec)).from_buffer_copy(rec.cpu().numpy().tobytes())
    return _batch_results(res, records, nrec, corr, sizes)
