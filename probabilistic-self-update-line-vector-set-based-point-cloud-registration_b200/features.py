"""Correspondences from two raw clouds: FPFH descriptors, the two-way descriptor nearest neighbour and FGR's matcher;
surface normals alone (radius or hybrid neighbourhood) on the same grid; the voxel-grid filter that comes first
(`colors=` carries a colour per point through it); and
the colour gradients of colored ICP (`color_gradients`, on the same grid; icp.colored_icp computes them itself).

What upstream TEASER++ gets from teaser::FPFHEstimation and teaser::Matcher (over PCL and FLANN), on the GPU through
the C ABI (include/psulvsb.h, csrc/k8_features.cu).  Host arrays in, host arrays out, except fpfh_device /
nearest_neighbours_device / fpfh_batch_device / match_batch_device / normals_device / normals_batch_device /
voxel_down_sample_device / voxel_down_sample_batch_device / color_gradients_batch_device, which take and return CUDA tensors on the current stream.
The _batch functions compute B clouds or B pairs in one call; each item's result is bit-identical to the single call
on it alone.
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


def _viewpoints(viewpoints, B):
    vps = [(0.0, 0.0, 0.0)] * B if viewpoints is None else [tuple(float(x) for x in v) for v in viewpoints]
    if len(vps) != B or any(len(v) != 3 for v in vps):
        raise ValueError(f"one 3-vector viewpoint per cloud is needed ({B} clouds)")
    return vps


def _clouds(ptrs, sizes, vps):
    arr = (capi.FpfhCloud * max(len(sizes), 1))()
    for c, (p, n, v) in enumerate(zip(ptrs, sizes, vps)):
        arr[c].pts, arr[c].n = p, n
        arr[c].viewpoint[:] = list(v)
    return arr


def fpfh_batch(clouds, normal_radius: float, feature_radius: float, viewpoints=None) -> list:
    """psulvsb_fpfh_batch_host: B clouds (3 x n_c each) with shared radii in one call.  Returns one (features n_c x 33
    float32, normals 3 x n_c float64) per cloud, each equal bit for bit to `fpfh` on that cloud alone."""
    ps = [_cm(p) for p in clouds]
    B = len(ps)
    sizes = [p.shape[1] for p in ps]
    arr = _clouds([p.ctypes.data if p.shape[1] else None for p in ps], sizes, _viewpoints(viewpoints, B))
    N = sum(sizes)
    feats = np.zeros((max(N, 1), DIM), dtype=np.float32)
    normals = np.zeros((max(N, 1), 3), dtype=np.float64)
    capi.check(capi.lib().psulvsb_fpfh_batch_host(arr, B, float(normal_radius), float(feature_radius),
                                                  normals.ctypes.data, feats.ctypes.data))
    out, o = [], 0
    for n in sizes:
        out.append((feats[o:o + n].copy(), np.asfortranarray(normals[o:o + n].T)))
        o += n
    return out


def fpfh_batch_device(d_clouds, normal_radius: float, feature_radius: float, viewpoints=None, work=None):
    """psulvsb_fpfh_batch on CUDA tensors [n_c, 3] float64 and the current stream.  Returns (features [sum n, 33],
    normals [sum n, 3], views): views[c] = (features, normals) of cloud c, views into the two tensors.  `work`: an
    optional uint8 CUDA tensor of at least psulvsb_fpfh_batch_workspace_bytes bytes to reuse."""
    import torch

    from .stages import _dev, _stream

    B = len(d_clouds)
    sizes = [int(p.shape[0]) for p in d_clouds]
    arr = _clouds([_dev(p) if n else None for p, n in zip(d_clouds, sizes)], sizes, _viewpoints(viewpoints, B))
    L = capi.lib()
    dev = d_clouds[0].device if B else torch.device("cuda")
    nbytes = L.psulvsb_fpfh_batch_workspace_bytes(arr, B)
    if work is None:
        work = torch.empty(max(1, nbytes), dtype=torch.uint8, device=dev)
    elif work.numel() < nbytes:
        raise ValueError("work is smaller than psulvsb_fpfh_batch_workspace_bytes(clouds, B)")
    N = sum(sizes)
    feats = torch.empty((max(N, 1), DIM), dtype=torch.float32, device=dev)
    normals = torch.empty((max(N, 1), 3), dtype=torch.float64, device=dev)
    capi.check(L.psulvsb_fpfh_batch(_stream(), arr, B, float(normal_radius), float(feature_radius), _dev(work),
                                    _dev(normals), _dev(feats)))
    views, o = [], 0
    for n in sizes:
        views.append((feats[o:o + n], normals[o:o + n]))
        o += n
    return feats[:N], normals[:N], views


def normals(points, radius: float, max_nn: int = 0, viewpoint=(0.0, 0.0, 0.0)) -> np.ndarray:
    """psulvsb_normals_host: 3xN points -> 3xN float64 normals (NaN below 3 neighbours), flipped towards `viewpoint`.
    max_nn = 0: every point within `radius` (the normals of `fpfh` with normal_radius = radius, bit for bit); 3 ... 32:
    the max_nn nearest of them (Open3D's KDTreeSearchParamHybrid(radius, max_nn)), ties to the lower index."""
    p = _cm(points)
    n = p.shape[1]
    out = np.zeros((3, n), dtype=np.float64, order="F")
    capi.check(capi.lib().psulvsb_normals_host(p.ctypes.data, n, float(radius), int(max_nn), _vp(viewpoint),
                                               out.ctypes.data))
    return out


def normals_device(d_pts, radius: float, max_nn: int = 0, viewpoint=(0.0, 0.0, 0.0), work=None):
    """psulvsb_normals on a CUDA tensor [N, 3] float64 (== column-major 3xN) and the current stream: normals [N, 3].
    `work`: an optional uint8 CUDA tensor of at least psulvsb_normals_workspace_bytes(N) bytes to reuse."""
    import torch

    from .stages import _dev, _stream

    n = d_pts.shape[0]
    nbytes = capi.lib().psulvsb_normals_workspace_bytes(n)
    if work is None:
        work = torch.empty(max(1, nbytes), dtype=torch.uint8, device=d_pts.device)
    elif work.numel() < nbytes:
        raise ValueError("work is smaller than psulvsb_normals_workspace_bytes(n)")
    out = torch.empty((max(n, 1), 3), dtype=torch.float64, device=d_pts.device)
    capi.check(capi.lib().psulvsb_normals(_stream(), _dev(d_pts) if n else None, n, float(radius), int(max_nn),
                                          _vp(viewpoint), _dev(work), _dev(out)))
    return out[:n]


def normals_batch(clouds, radius: float, max_nn: int = 0, viewpoints=None) -> list:
    """psulvsb_normals_batch_host: B clouds (3 x n_c each) with a shared radius and max_nn in one call.  Returns one
    3 x n_c float64 normal array per cloud, each equal bit for bit to `normals` on that cloud alone."""
    ps = [_cm(p) for p in clouds]
    B = len(ps)
    sizes = [p.shape[1] for p in ps]
    arr = _clouds([p.ctypes.data if p.shape[1] else None for p in ps], sizes, _viewpoints(viewpoints, B))
    out = np.zeros((max(sum(sizes), 1), 3), dtype=np.float64)
    capi.check(capi.lib().psulvsb_normals_batch_host(arr, B, float(radius), int(max_nn), out.ctypes.data))
    res, o = [], 0
    for n in sizes:
        res.append(np.asfortranarray(out[o:o + n].T))
        o += n
    return res


def normals_batch_device(d_clouds, radius: float, max_nn: int = 0, viewpoints=None, work=None):
    """psulvsb_normals_batch on CUDA tensors [n_c, 3] float64 and the current stream.  Returns (normals [sum n, 3],
    views): views[c] = cloud c's rows.  `work`: an optional uint8 CUDA tensor of at least
    psulvsb_normals_batch_workspace_bytes bytes to reuse."""
    import torch

    from .stages import _dev, _stream

    B = len(d_clouds)
    sizes = [int(p.shape[0]) for p in d_clouds]
    arr = _clouds([_dev(p) if n else None for p, n in zip(d_clouds, sizes)], sizes, _viewpoints(viewpoints, B))
    L = capi.lib()
    dev = d_clouds[0].device if B else torch.device("cuda")
    nbytes = L.psulvsb_normals_batch_workspace_bytes(arr, B)
    if work is None:
        work = torch.empty(max(1, nbytes), dtype=torch.uint8, device=dev)
    elif work.numel() < nbytes:
        raise ValueError("work is smaller than psulvsb_normals_batch_workspace_bytes(clouds, B)")
    N = sum(sizes)
    out = torch.empty((max(N, 1), 3), dtype=torch.float64, device=dev)
    capi.check(L.psulvsb_normals_batch(_stream(), arr, B, float(radius), int(max_nn), _dev(work), _dev(out)))
    views, o = [], 0
    for n in sizes:
        views.append(out[o:o + n])
        o += n
    return out[:N], views


def _color_clouds(ptrs, sizes):
    """psulvsb_color_cloud_t[B] from (points, colors, normals) pointers and n per cloud."""
    arr = (capi.ColorCloud * max(len(sizes), 1))()
    for c, ((pp, pc, pn), n) in enumerate(zip(ptrs, sizes)):
        arr[c].points, arr[c].n, arr[c].colors, arr[c].normals = pp, n, pc, pn
    return arr


def _same_shape(a, cloud, what) -> np.ndarray:
    a = _cm(a)
    if a.shape != cloud.shape:
        raise ValueError(f"{what}: one per point is needed, got {a.shape} for {cloud.shape}")
    return a


def color_gradients(points, colors, normals, radius: float, max_nn: int = 30) -> np.ndarray:
    """The colour gradient of every point (3 x n float64; Open3D's InitializePointCloudForColoredICP): points, colors
    ([0, 1] RGB) and normals 3 x n.  The hybrid neighbourhood (`radius`, 4 <= max_nn <= 32) of `normals`; 0 where
    fewer than 4 points are kept, the normal is not finite or the 3x3 solve fails.  A batch of one cloud."""
    return color_gradients_batch([points], [colors], [normals], radius, max_nn)[0]


def color_gradients_batch(clouds, colors, normals, radius: float, max_nn: int = 30) -> list:
    """psulvsb_color_gradients_batch_host: B clouds (3 x n_c each) with their colours and normals in one call.  Returns
    one 3 x n_c float64 gradient array per cloud, each equal bit for bit to a batch of that cloud alone."""
    ps = [_cm(p) for p in clouds]
    B = len(ps)
    if len(colors) != B or len(normals) != B:
        raise ValueError(f"{B} clouds, {len(colors)} colour and {len(normals)} normal sets")
    cs = [_same_shape(c, p, "colors") for c, p in zip(colors, ps)]
    ns = [_same_shape(n, p, "normals") for n, p in zip(normals, ps)]
    sizes = [p.shape[1] for p in ps]
    arr = _color_clouds([(p.ctypes.data, c.ctypes.data, n.ctypes.data) if p.shape[1] else (None, None, None)
                         for p, c, n in zip(ps, cs, ns)], sizes)
    out = np.zeros((max(sum(sizes), 1), 3), dtype=np.float64)
    capi.check(capi.lib().psulvsb_color_gradients_batch_host(arr, B, float(radius), int(max_nn), out.ctypes.data))
    res, o = [], 0
    for n in sizes:
        res.append(np.asfortranarray(out[o:o + n].T))
        o += n
    return res


def color_gradients_batch_device(d_clouds, d_colors, d_normals, radius: float, max_nn: int = 30, work=None):
    """psulvsb_color_gradients_batch on CUDA tensors [n_c, 3] float64 and the current stream.  Returns (gradients
    [sum n, 3], views): views[c] = cloud c's rows.  `work`: an optional uint8 CUDA tensor of at least
    psulvsb_color_gradients_batch_workspace_bytes bytes to reuse."""
    import torch

    from .stages import _dev, _stream

    B = len(d_clouds)
    if len(d_colors) != B or len(d_normals) != B:
        raise ValueError(f"{B} clouds, {len(d_colors)} colour and {len(d_normals)} normal sets")
    for p, c, n in zip(d_clouds, d_colors, d_normals):
        if tuple(c.shape) != tuple(p.shape) or tuple(n.shape) != tuple(p.shape):
            raise ValueError("one colour and one normal per point are needed")
    sizes = [int(p.shape[0]) for p in d_clouds]
    arr = _color_clouds([(_dev(p), _dev(c), _dev(n)) if k else (None, None, None)
                         for p, c, n, k in zip(d_clouds, d_colors, d_normals, sizes)], sizes)
    L = capi.lib()
    dev = d_clouds[0].device if B else torch.device("cuda")
    nbytes = L.psulvsb_color_gradients_batch_workspace_bytes(arr, B)
    if work is None:
        work = torch.empty(max(1, nbytes), dtype=torch.uint8, device=dev)
    elif work.numel() < nbytes:
        raise ValueError("work is smaller than psulvsb_color_gradients_batch_workspace_bytes(clouds, B)")
    N = sum(sizes)
    out = torch.empty((max(N, 1), 3), dtype=torch.float64, device=dev)
    capi.check(L.psulvsb_color_gradients_batch(_stream(), arr, B, float(radius), int(max_nn), _dev(work), _dev(out)))
    views, o = [], 0
    for n in sizes:
        views.append(out[o:o + n])
        o += n
    return out[:N], views


def voxel_down_sample(points, voxel_size: float, colors=None):
    """psulvsb_voxel_down_sample_host (Open3D's voxel_down_sample): 3xN points -> 3xM float64 voxel means, in ascending
    order of each voxel's lowest input index.  Points with a non-finite coordinate are dropped.  colors: 3xN [0, 1]
    RGB, one per point (psulvsb_voxel_down_sample_colors_host): returns (voxels, voxel colours 3xM), the voxels bit for
    bit those without colours, each colour the mean of its voxel's members' colours."""
    p = _cm(points)
    n = p.shape[1]
    out = np.zeros((3, max(n, 1)), dtype=np.float64, order="F")
    m = C.c_int(0)
    if colors is None:
        capi.check(capi.lib().psulvsb_voxel_down_sample_host(p.ctypes.data if n else None, n, float(voxel_size),
                                                             out.ctypes.data, C.byref(m)))
        return out[:, :m.value].copy(order="F")
    c = _same_shape(colors, p, "colors")
    oc = np.zeros((3, max(n, 1)), dtype=np.float64, order="F")
    capi.check(capi.lib().psulvsb_voxel_down_sample_colors_host(p.ctypes.data if n else None,
                                                                c.ctypes.data if n else None, n, float(voxel_size),
                                                                out.ctypes.data, oc.ctypes.data, C.byref(m)))
    return out[:, :m.value].copy(order="F"), oc[:, :m.value].copy(order="F")


def voxel_down_sample_device(d_pts, voxel_size: float, work=None, colors=None):
    """psulvsb_voxel_down_sample on a CUDA tensor [N, 3] float64 (== column-major 3xN) and the current stream, without
    a host round trip.  Returns (voxels [N, 3], count [1] int32): the first count[0] rows are the voxels, the rest is
    unspecified.  `work`: an optional uint8 CUDA tensor of at least psulvsb_voxel_down_sample_workspace_bytes(N) bytes
    to reuse.  colors: a CUDA tensor [N, 3] float64 of [0, 1] RGB (psulvsb_voxel_down_sample_colors): returns (voxels,
    voxel colours [N, 3], count), `work` then sized by psulvsb_voxel_down_sample_colors_workspace_bytes(N)."""
    import torch

    from .stages import _dev, _stream

    n = d_pts.shape[0]
    L = capi.lib()
    if colors is not None and tuple(colors.shape) != tuple(d_pts.shape):
        raise ValueError("colors: one colour per point is needed")
    name = "psulvsb_voxel_down_sample_workspace_bytes" if colors is None else \
        "psulvsb_voxel_down_sample_colors_workspace_bytes"
    nbytes = getattr(L, name)(n)
    if work is None:
        work = torch.empty(max(1, nbytes), dtype=torch.uint8, device=d_pts.device)
    elif work.numel() < nbytes:
        raise ValueError(f"work is smaller than {name}(n)")
    out = torch.empty((max(n, 1), 3), dtype=torch.float64, device=d_pts.device)
    count = torch.empty(1, dtype=torch.int32, device=d_pts.device)
    if colors is None:
        capi.check(L.psulvsb_voxel_down_sample(_stream(), _dev(d_pts) if n else None, n, float(voxel_size), _dev(work),
                                               _dev(out), _dev(count)))
        return out[:n], count
    oc = torch.empty((max(n, 1), 3), dtype=torch.float64, device=d_pts.device)
    capi.check(L.psulvsb_voxel_down_sample_colors(_stream(), _dev(d_pts) if n else None, _dev(colors) if n else None,
                                                  n, float(voxel_size), _dev(work), _dev(out), _dev(oc), _dev(count)))
    return out[:n], oc[:n], count


def voxel_down_sample_batch(clouds, voxel_size: float, colors=None) -> list:
    """psulvsb_voxel_down_sample_batch_host: B clouds (3 x n_c each) with a shared voxel size in one call.  Returns one
    3 x m_c float64 array per cloud, each equal bit for bit to `voxel_down_sample` on that cloud alone.  colors: one
    3 x n_c colour array per cloud (psulvsb_voxel_down_sample_colors_batch_host): returns (voxel list, colour list)."""
    ps = [_cm(p) for p in clouds]
    B = len(ps)
    sizes = [p.shape[1] for p in ps]
    out = np.zeros((max(sum(sizes), 1), 3), dtype=np.float64)
    counts = np.zeros(max(B, 1), dtype=np.int32)
    oc = None
    if colors is None:
        arr = _clouds([p.ctypes.data if p.shape[1] else None for p in ps], sizes, _viewpoints(None, B))
        capi.check(capi.lib().psulvsb_voxel_down_sample_batch_host(arr, B, float(voxel_size), out.ctypes.data,
                                                                   counts.ctypes.data))
    else:
        if len(colors) != B:
            raise ValueError(f"{B} clouds and {len(colors)} colour sets")
        cs = [_same_shape(c, p, "colors") for c, p in zip(colors, ps)]
        arr = _color_clouds([(p.ctypes.data, c.ctypes.data, None) if p.shape[1] else (None, None, None)
                             for p, c in zip(ps, cs)], sizes)
        oc = np.zeros_like(out)
        capi.check(capi.lib().psulvsb_voxel_down_sample_colors_batch_host(arr, B, float(voxel_size), out.ctypes.data,
                                                                          oc.ctypes.data, counts.ctypes.data))
    res, cres, o = [], [], 0
    for c, n in enumerate(sizes):
        res.append(np.asfortranarray(out[o:o + int(counts[c])].T))
        if oc is not None:
            cres.append(np.asfortranarray(oc[o:o + int(counts[c])].T))
        o += n
    return res if oc is None else (res, cres)


def voxel_down_sample_batch_device(d_clouds, voxel_size: float, work=None, colors=None):
    """psulvsb_voxel_down_sample_batch on CUDA tensors [n_c, 3] float64 and the current stream, without a host round
    trip.  Returns (voxels [sum n, 3] float64, counts [B] int32, offsets): cloud c's voxels are
    voxels[offsets[c]:offsets[c] + counts[c]], offsets[c] = sum of the sizes before it.  `work`: an optional uint8 CUDA
    tensor of at least psulvsb_voxel_down_sample_batch_workspace_bytes bytes to reuse.  colors: one CUDA tensor
    [n_c, 3] float64 per cloud (psulvsb_voxel_down_sample_colors_batch): returns (voxels, voxel colours [sum n, 3],
    counts, offsets), `work` then sized by psulvsb_voxel_down_sample_colors_batch_workspace_bytes."""
    import torch

    from .stages import _dev, _stream

    B = len(d_clouds)
    sizes = [int(p.shape[0]) for p in d_clouds]
    L = capi.lib()
    if colors is None:
        arr = _clouds([_dev(p) if n else None for p, n in zip(d_clouds, sizes)], sizes, _viewpoints(None, B))
        name = "psulvsb_voxel_down_sample_batch_workspace_bytes"
    else:
        if len(colors) != B or any(tuple(c.shape) != tuple(p.shape) for c, p in zip(colors, d_clouds)):
            raise ValueError("colors: one colour tensor per cloud, one colour per point, is needed")
        arr = _color_clouds([(_dev(p), _dev(c), None) if n else (None, None, None)
                             for p, c, n in zip(d_clouds, colors, sizes)], sizes)
        name = "psulvsb_voxel_down_sample_colors_batch_workspace_bytes"
    dev = d_clouds[0].device if B else torch.device("cuda")
    nbytes = getattr(L, name)(arr, B)
    if work is None:
        work = torch.empty(max(1, nbytes), dtype=torch.uint8, device=dev)
    elif work.numel() < nbytes:
        raise ValueError(f"work is smaller than {name}(clouds, B)")
    offsets = np.concatenate([[0], np.cumsum(sizes, dtype=np.int64)]).astype(np.int64)
    N = int(offsets[-1])
    out = torch.empty((max(N, 1), 3), dtype=torch.float64, device=dev)
    counts = torch.empty(max(B, 1), dtype=torch.int32, device=dev)
    if colors is None:
        capi.check(L.psulvsb_voxel_down_sample_batch(_stream(), arr, B, float(voxel_size), _dev(work), _dev(out),
                                                     _dev(counts)))
        return out[:N], counts[:B], offsets[:B]
    oc = torch.empty((max(N, 1), 3), dtype=torch.float64, device=dev)
    capi.check(L.psulvsb_voxel_down_sample_colors_batch(_stream(), arr, B, float(voxel_size), _dev(work), _dev(out),
                                                        _dev(oc), _dev(counts)))
    return out[:N], oc[:N], counts[:B], offsets[:B]


def match_caps(n_srcs, n_tgts, crosscheck: bool = True, tuple_test: bool = False) -> list:
    """The output capacity of every pair of a matcher batch (the header's formula): 0 when a side is empty, else
    3 * 1000 with the tuple test, else n_src with crosscheck and n_src + n_tgt without."""
    return [0 if ns == 0 or nt == 0 else (3 * MAX_TUPLES if tuple_test else (ns if crosscheck else ns + nt))
            for ns, nt in zip(n_srcs, n_tgts)]


def _seeds(seed, seeds, B):
    s = [int(seed) + b for b in range(B)] if seeds is None else [int(x) for x in seeds]
    if len(s) != B:
        raise ValueError(f"one seed per pair is needed ({B} pairs)")
    return s


def _match_pairs(ptrs, sizes, seeds):
    arr = (capi.MatchPair * max(len(sizes), 1))()
    for b, ((s, t, fs, ft), (ns, nt), seed) in enumerate(zip(ptrs, sizes, seeds)):
        arr[b].src, arr[b].n_src, arr[b].tgt, arr[b].n_tgt, arr[b].fs, arr[b].ft = s, ns, t, nt, fs, ft
        arr[b].seed = seed & (2 ** 64 - 1)
    return arr


def match_batch(srcs, tgts, fss, fts, crosscheck: bool = True, tuple_test: bool = False, tuple_scale: float = 0.95,
                seed: int = 0, seeds=None) -> list:
    """psulvsb_match_batch_host: B pairs with shared flags in one call.  Pair b's tuple test uses seeds[b], or seed + b
    without `seeds`.  Returns one (K, 2) int32 array per pair, each equal to `match` on that pair alone."""
    s = [_cm(a) for a in srcs]
    t = [_cm(a) for a in tgts]
    fs = [_desc(a) for a in fss]
    ft = [_desc(a) for a in fts]
    B = len(s)
    if not (len(t) == len(fs) == len(ft) == B):
        raise ValueError("srcs, tgts, fss and fts need one entry per pair")
    for a, b, fa, fb in zip(s, t, fs, ft):
        if fa.shape[0] != a.shape[1] or fb.shape[0] != b.shape[1]:
            raise ValueError("one descriptor per point is needed on each side")
    sizes = [(a.shape[1], b.shape[1]) for a, b in zip(s, t)]
    ptr = lambda a: a.ctypes.data if a.size else None  # noqa: E731
    arr = _match_pairs([(ptr(a), ptr(b), ptr(fa), ptr(fb)) for a, b, fa, fb in zip(s, t, fs, ft)], sizes,
                       _seeds(seed, seeds, B))
    caps = match_caps([a for a, _ in sizes], [b for _, b in sizes], crosscheck, tuple_test)
    out = np.zeros((max(sum(caps), 1), 2), dtype=np.int32)
    counts = np.zeros(max(B, 1), dtype=np.int64)
    capi.check(capi.lib().psulvsb_match_batch_host(arr, B, int(bool(crosscheck)), int(bool(tuple_test)),
                                                   float(tuple_scale), out.ctypes.data, counts.ctypes.data))
    res, o = [], 0
    for b, cap in enumerate(caps):
        res.append(out[o:o + int(counts[b])].copy())
        o += cap
    return res


def match_batch_device(d_srcs, d_tgts, d_fss, d_fts, crosscheck: bool = True, tuple_test: bool = False,
                       tuple_scale: float = 0.95, seed: int = 0, seeds=None, work=None):
    """psulvsb_match_batch on CUDA tensors (points [n, 3] float64, descriptors [n, 33] float32) and the current stream,
    without a host round trip inside.  Returns (pairs [sum cap, 2] int32, counts [B] int64, offsets): pair b's (source,
    target) pairs are pairs[offsets[b]:offsets[b] + counts[b]].  `work`: an optional uint8 CUDA tensor of at least
    psulvsb_match_batch_workspace_bytes bytes to reuse."""
    import torch

    from .stages import _dev, _stream

    B = len(d_srcs)
    if not (len(d_tgts) == len(d_fss) == len(d_fts) == B):
        raise ValueError("d_srcs, d_tgts, d_fss and d_fts need one entry per pair")
    sizes = [(int(a.shape[0]), int(b.shape[0])) for a, b in zip(d_srcs, d_tgts)]
    ptr = lambda a: _dev(a) if a.numel() else None  # noqa: E731
    arr = _match_pairs([(ptr(a), ptr(b), ptr(fa), ptr(fb)) for a, b, fa, fb in zip(d_srcs, d_tgts, d_fss, d_fts)],
                       sizes, _seeds(seed, seeds, B))
    L = capi.lib()
    cross, tup = int(bool(crosscheck)), int(bool(tuple_test))
    dev = d_srcs[0].device if B else torch.device("cuda")
    nbytes = L.psulvsb_match_batch_workspace_bytes(arr, B, cross, tup)
    if work is None:
        work = torch.empty(max(1, nbytes), dtype=torch.uint8, device=dev)
    elif work.numel() < nbytes:
        raise ValueError("work is smaller than psulvsb_match_batch_workspace_bytes(pairs, B, ...)")
    caps = match_caps([a for a, _ in sizes], [b for _, b in sizes], crosscheck, tuple_test)
    offsets = np.concatenate([[0], np.cumsum(caps)]).astype(np.int64)
    pairs = torch.empty((max(int(offsets[-1]), 1), 2), dtype=torch.int32, device=dev)
    counts = torch.empty(max(B, 1), dtype=torch.int64, device=dev)
    capi.check(L.psulvsb_match_batch(_stream(), arr, B, cross, tup, float(tuple_scale), _dev(work), _dev(pairs),
                                     _dev(counts)))
    return pairs[:int(offsets[-1])], counts[:B], offsets[:B]
