"""Correspondences from two raw clouds: FPFH descriptors, the two-way descriptor nearest neighbour and FGR's matcher.

What upstream TEASER++ gets from teaser::FPFHEstimation and teaser::Matcher (over PCL and FLANN), on the GPU through
the C ABI (include/psulvsb.h, csrc/k8_features.cu).  Host arrays in, host arrays out, except fpfh_device /
nearest_neighbours_device, which take and return CUDA tensors on the current stream.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi

DIM = 33
MAX_TUPLES = 1000


def _cm(points) -> np.ndarray:
    p = np.asarray(points, dtype=np.float64)
    if p.ndim != 2 or p.shape[0] != 3:
        raise ValueError(f"expected a 3xN matrix, got {p.shape}")
    return np.asfortranarray(p)


def _desc(f) -> np.ndarray:
    f = np.ascontiguousarray(f, dtype=np.float32)
    if f.ndim != 2 or f.shape[1] != DIM:
        raise ValueError(f"expected an n x {DIM} descriptor array, got {f.shape}")
    return f


def _vp(viewpoint):
    return (C.c_double * 3)(*[float(v) for v in viewpoint])


def fpfh(points, normal_radius: float, feature_radius: float, viewpoint=(0.0, 0.0, 0.0)):
    """psulvsb_fpfh_host: 3xN points -> (features N x 33 float32, normals 3xN float64)."""
    p = _cm(points)
    n = p.shape[1]
    feats = np.zeros((n, DIM), dtype=np.float32)
    normals = np.zeros((3, n), dtype=np.float64, order="F")
    capi.check(capi.lib().psulvsb_fpfh_host(p.ctypes.data, n, float(normal_radius), float(feature_radius),
                                            _vp(viewpoint), normals.ctypes.data, feats.ctypes.data))
    return feats, normals


def fpfh_device(d_pts, normal_radius: float, feature_radius: float, viewpoint=(0.0, 0.0, 0.0)):
    """psulvsb_fpfh on a CUDA tensor [N, 3] float64 (== column-major 3xN): (features [N, 33] float32, normals [N, 3])."""
    import torch

    from .stages import _dev, _stream

    n = d_pts.shape[0]
    work = torch.empty(max(1, capi.lib().psulvsb_fpfh_workspace_bytes(n)), dtype=torch.uint8, device=d_pts.device)
    feats = torch.empty((n, DIM), dtype=torch.float32, device=d_pts.device)
    normals = torch.empty((n, 3), dtype=torch.float64, device=d_pts.device)
    capi.check(capi.lib().psulvsb_fpfh(_stream(), _dev(d_pts), n, float(normal_radius), float(feature_radius),
                                       _vp(viewpoint), _dev(work), _dev(normals), _dev(feats)))
    return feats, normals


def nearest_neighbours_device(d_fs, d_ft):
    """psulvsb_feature_nn on CUDA tensors [n, 33] float32: (nn_src_to_tgt [n_src], nn_tgt_to_src [n_tgt]) int32."""
    import torch

    from .stages import _dev, _stream

    ns, nt = d_fs.shape[0], d_ft.shape[0]
    a = torch.empty(max(ns, 1), dtype=torch.int32, device=d_fs.device)
    b = torch.empty(max(nt, 1), dtype=torch.int32, device=d_fs.device)
    capi.check(capi.lib().psulvsb_feature_nn(_stream(), _dev(d_fs), ns, _dev(d_ft), nt, _dev(a), _dev(b)))
    return a[:ns], b[:nt]


def nearest_neighbours(fs, ft):
    """Two-way nearest neighbour of host descriptors (exact squared L2, ties to the lowest index):
    (nn_src_to_tgt [n_src], nn_tgt_to_src [n_tgt]) int32 numpy arrays."""
    import torch

    fs, ft = _desc(fs), _desc(ft)
    a, b = nearest_neighbours_device(torch.from_numpy(fs).cuda(), torch.from_numpy(ft).cuda())
    return a.cpu().numpy(), b.cpu().numpy()


def match(src, tgt, fs, ft, crosscheck: bool = True, tuple_test: bool = False, tuple_scale: float = 0.95,
          seed: int = 0) -> np.ndarray:
    """psulvsb_match_host (teaser::Matcher::calculateCorrespondences): (K, 2) int32 (source, target) index pairs."""
    s, t = _cm(src), _cm(tgt)
    fs, ft = _desc(fs), _desc(ft)
    if fs.shape[0] != s.shape[1] or ft.shape[0] != t.shape[1]:
        raise ValueError("one descriptor per point is needed on each side")
    cap = 3 * MAX_TUPLES if tuple_test else (fs.shape[0] + (0 if crosscheck else ft.shape[0]))
    out = np.zeros((max(cap, 1), 2), dtype=np.int32)
    n = C.c_longlong(0)
    capi.check(capi.lib().psulvsb_match_host(s.ctypes.data, s.shape[1], t.ctypes.data, t.shape[1], fs.ctypes.data,
                                             ft.ctypes.data, int(bool(crosscheck)), int(bool(tuple_test)),
                                             float(tuple_scale), int(seed), out.ctypes.data, cap, C.byref(n)))
    return out[:n.value].copy()
