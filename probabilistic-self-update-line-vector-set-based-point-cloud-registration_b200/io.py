"""ctypes binding of include/psulvsb_io.h: the host-side helpers of the callers around the hot path
(normal-angle histogram pre-filter, reduced-set builder, PLY vertices, correspondence files)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi

IO_SYMBOLS = ["psulvsb_histogram_outlier_removal", "psulvsb_mask_filter", "psulvsb_prefilter_reduce",
              "psulvsb_prefilter_reduce_batch", "psulvsb_ply_vertex_count",
              "psulvsb_ply_read_xyz", "psulvsb_ply_read_xyz_rgb", "psulvsb_corr_count", "psulvsb_corr_read", "psulvsb_gtmat_read",
              "psulvsb_gtlog_read"]

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_fp = C.POINTER(C.c_float)
_llp = C.POINTER(C.c_longlong)
_declared = False


def _lib():
    global _declared
    L = capi.lib()
    if not _declared:
        L.psulvsb_histogram_outlier_removal.argtypes = [_dp, _dp, C.c_int, _ip, _ip]
        L.psulvsb_mask_filter.argtypes = [_dp, _dp, _ip, C.c_int, _dp, _dp, _ip, _ip]
        L.psulvsb_prefilter_reduce.argtypes = [_dp, _dp, _dp, _dp, C.c_int, _ip, _dp, _dp, _ip, _ip, _ip]
        pp = C.POINTER(C.c_void_p)
        L.psulvsb_prefilter_reduce_batch.argtypes = [C.c_int, pp, pp, pp, pp, _ip, pp, pp, pp, pp, _ip, _ip]
        L.psulvsb_ply_vertex_count.argtypes = [C.c_char_p, _llp]
        L.psulvsb_ply_read_xyz.argtypes = [C.c_char_p, _fp, C.c_longlong, _llp]
        L.psulvsb_ply_read_xyz_rgb.argtypes = [C.c_char_p, _fp, _dp, C.c_longlong, _llp]
        L.psulvsb_corr_count.argtypes = [C.c_char_p, _llp]
        L.psulvsb_corr_read.argtypes = [C.c_char_p, _dp, _dp, C.c_longlong, _llp]
        L.psulvsb_gtmat_read.argtypes = [C.c_char_p, _dp]
        L.psulvsb_gtlog_read.argtypes = [C.c_char_p, _ip, C.c_longlong, _llp]
        _declared = True
    return L


def _cm(a):
    a = np.asfortranarray(np.asarray(a, dtype=np.float64))
    assert a.ndim == 2 and a.shape[0] == 3
    return a


def histogram_outlier_removal(src_normals, tgt_normals):
    """PSULVSB.cc:87-172 -> (keep_mask[n] in {-1,0,1}, remain_count)."""
    a, b = _cm(src_normals), _cm(tgt_normals)
    n = a.shape[1]
    keep = np.zeros(n, dtype=np.int32)
    rem = C.c_int(0)
    capi.check(_lib().psulvsb_histogram_outlier_removal(a.ctypes.data_as(_dp), b.ctypes.data_as(_dp), n,
                                                        keep.ctypes.data_as(_ip), C.byref(rem)))
    return keep, rem.value


def mask_filter(src, tgt, keep_mask):
    """PSULVSB.cc:174-188 -> (src_reduce 3xC, tgt_reduce 3xC, dense reduce_map[n])."""
    a, b = _cm(src), _cm(tgt)
    n = a.shape[1]
    keep = np.ascontiguousarray(keep_mask, dtype=np.int32)
    sr = np.zeros((3, n), order="F")
    tr = np.zeros((3, n), order="F")
    rm = np.zeros(n, dtype=np.int32)
    c = C.c_int(0)
    capi.check(_lib().psulvsb_mask_filter(a.ctypes.data_as(_dp), b.ctypes.data_as(_dp), keep.ctypes.data_as(_ip), n,
                                          sr.ctypes.data_as(_dp), tr.ctypes.data_as(_dp), rm.ctypes.data_as(_ip),
                                          C.byref(c)))
    return np.asfortranarray(sr[:, :c.value]), np.asfortranarray(tr[:, :c.value]), rm


def prefilter_reduce(src_normals, tgt_normals, src, tgt):
    """The driver's whole timed pre-filter (PSULVSB.cc:310-317) in one device call:
    -> (keep_mask[n], src_reduce 3xC, tgt_reduce 3xC, dense reduce_map[n], remain_count)."""
    a, b, p, q = _cm(src_normals), _cm(tgt_normals), _cm(src), _cm(tgt)
    n = a.shape[1]
    keep = np.zeros(n, dtype=np.int32)
    sr = np.zeros((3, max(n, 1)), order="F")
    tr = np.zeros((3, max(n, 1)), order="F")
    rm = np.zeros(n, dtype=np.int32)
    c, rem = C.c_int(0), C.c_int(0)
    capi.check(_lib().psulvsb_prefilter_reduce(a.ctypes.data_as(_dp), b.ctypes.data_as(_dp), p.ctypes.data_as(_dp),
                                               q.ctypes.data_as(_dp), n, keep.ctypes.data_as(_ip),
                                               sr.ctypes.data_as(_dp), tr.ctypes.data_as(_dp), rm.ctypes.data_as(_ip),
                                               C.byref(c), C.byref(rem)))
    return keep, np.asfortranarray(sr[:, :c.value]), np.asfortranarray(tr[:, :c.value]), rm, rem.value


def prefilter_reduce_batch(src_normals, tgt_normals, srcs, tgts):
    """psulvsb_prefilter_reduce_batch: the pre-filter of B correspondence sets in ONE device launch (a CTA per set).
    Lists of 3xN arrays in; list of (keep_mask, src_reduce, tgt_reduce, reduce_map, remain_count) out."""
    B = len(srcs)
    a = [_cm(x) for x in src_normals]
    b = [_cm(x) for x in tgt_normals]
    p = [_cm(x) for x in srcs]
    q = [_cm(x) for x in tgts]
    n = np.array([x.shape[1] for x in p], dtype=np.int32)
    keep = [np.zeros(k, dtype=np.int32) for k in n]
    sr = [np.zeros((3, max(int(k), 1)), order="F") for k in n]
    tr = [np.zeros((3, max(int(k), 1)), order="F") for k in n]
    rm = [np.zeros(k, dtype=np.int32) for k in n]
    cc = np.zeros(B, dtype=np.int32)
    rem = np.zeros(B, dtype=np.int32)

    def ptrs(arrs):
        return (C.c_void_p * B)(*[x.ctypes.data for x in arrs])

    capi.check(_lib().psulvsb_prefilter_reduce_batch(B, ptrs(a), ptrs(b), ptrs(p), ptrs(q), n.ctypes.data_as(_ip),
                                                     ptrs(keep), ptrs(sr), ptrs(tr), ptrs(rm), cc.ctypes.data_as(_ip),
                                                     rem.ctypes.data_as(_ip)))
    return [(keep[i], np.asfortranarray(sr[i][:, :cc[i]]), np.asfortranarray(tr[i][:, :cc[i]]), rm[i], int(rem[i]))
            for i in range(B)]


def read_ply_xyz(path: str) -> np.ndarray:
    """Vertices of a PLY file as a 3xN float64 matrix (values are the file's x, y, z read as float32 like
    teaser::PointXYZ, teaser/src/ply_io.cc:26-79)."""
    n = C.c_longlong(0)
    capi.check(_lib().psulvsb_ply_vertex_count(path.encode(), C.byref(n)))
    xyz = np.zeros((max(n.value, 1), 3), dtype=np.float32)
    capi.check(_lib().psulvsb_ply_read_xyz(path.encode(), xyz.ctypes.data_as(_fp), n.value, C.byref(n)))
    return np.asfortranarray(xyz[:n.value].T.astype(np.float64))


def read_ply_xyz_rgb(path: str):
    """Vertices and colours of a PLY file: (3xN float64 positions, read as float32 like `read_ply_xyz`; 3xN float64
    [0, 1] RGB from the red, green and blue properties, uchar / uint8 over 255, float / double as stored)."""
    n = C.c_longlong(0)
    capi.check(_lib().psulvsb_ply_vertex_count(path.encode(), C.byref(n)))
    xyz = np.zeros((max(n.value, 1), 3), dtype=np.float32)
    rgb = np.zeros((max(n.value, 1), 3), dtype=np.float64)
    capi.check(_lib().psulvsb_ply_read_xyz_rgb(path.encode(), xyz.ctypes.data_as(_fp), rgb.ctypes.data_as(_dp),
                                               n.value, C.byref(n)))
    return np.asfortranarray(xyz[:n.value].T.astype(np.float64)), np.asfortranarray(rgb[:n.value].T)


def read_correspondences(path: str):
    """'x y z x y z' per line (optionally after a count header) -> (src 3xN, dst 3xN)."""
    n = C.c_longlong(0)
    capi.check(_lib().psulvsb_corr_count(path.encode(), C.byref(n)))
    src = np.zeros((3, max(n.value, 1)), order="F")
    dst = np.zeros((3, max(n.value, 1)), order="F")
    capi.check(_lib().psulvsb_corr_read(path.encode(), src.ctypes.data_as(_dp), dst.ctypes.data_as(_dp), n.value,
                                        C.byref(n)))
    return np.asfortranarray(src[:, :n.value]), np.asfortranarray(dst[:, :n.value])


def read_gtmat(path: str) -> np.ndarray:
    T = np.zeros(16)
    capi.check(_lib().psulvsb_gtmat_read(path.encode(), T.ctypes.data_as(_dp)))
    return T.reshape(4, 4, order="F")


def read_gtlog(path: str):
    n = C.c_longlong(0)
    capi.check(_lib().psulvsb_gtlog_read(path.encode(), None, 0, C.byref(n)))
    pairs = np.zeros((max(n.value, 1), 2), dtype=np.int32)
    capi.check(_lib().psulvsb_gtlog_read(path.encode(), pairs.ctypes.data_as(_ip), n.value, C.byref(n)))
    return [tuple(int(v) for v in p) for p in pairs[:n.value]]


def estimate_normals(points, k: int = 20, viewpoint=(0.0, 0.0, 0.0)) -> np.ndarray:
    """k-NN PCA normals on the GPU (psulvsb_estimate_normals_host): 3xN in, 3xN out."""
    p = _cm(points)
    out = np.zeros_like(p, order="F")
    vp = (C.c_double * 3)(*[float(v) for v in viewpoint])
    capi.check(capi.lib().psulvsb_estimate_normals_host(p.ctypes.data_as(_dp), p.shape[1], k, vp,
                                                        out.ctypes.data_as(_dp)))
    return out
