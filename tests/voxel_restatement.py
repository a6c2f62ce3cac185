"""numpy restatement of the voxel-grid filter (csrc/k8_voxel.cu; DESIGN.md section 10, "Voxel downsampling"): Open3D's
PointCloud::VoxelDownSample with the positions this project takes -- non-finite points dropped, cells saturated to
int64, voxels in ascending order of their lowest input index.  Every step is one float64 operation that the kernels
perform in the same order, so the GPU output must equal this bit for bit."""
import numpy as np

I64_MIN, I64_MAX = np.iinfo(np.int64).min, np.iinfo(np.int64).max


def origin(P, v):
    """origin = lo - v * 0.5, lo the per-coordinate minimum over the finite points (None without any)."""
    P = np.asarray(P, dtype=np.float64)
    fin = np.isfinite(P).all(axis=0)
    if not fin.any():
        return None
    return P[:, fin].min(axis=1) - v * 0.5


def cells(P, v):
    """(finite mask, int64 cells [3, n_finite]): floor((p - origin) / v), one subtraction and one division, saturated
    to the int64 range as the device's conversion does."""
    P = np.asarray(P, dtype=np.float64)
    fin = np.isfinite(P).all(axis=0)
    o = origin(P, v)
    if o is None:
        return fin, np.zeros((3, 0), dtype=np.int64)
    with np.errstate(over="ignore"):
        f = np.floor((P[:, fin] - o[:, None]) / v)
    c = np.where(f >= 2.0 ** 63, 0.0, np.where(f < -(2.0 ** 63), 0.0, f)).astype(np.int64)
    c[f >= 2.0 ** 63] = I64_MAX
    c[f < -(2.0 ** 63)] = I64_MIN
    return fin, c


def voxel_down_sample(P, v):
    """3 x m float64: the mean of each voxel's finite points (sequential float64 sums in ascending input index, then one
    division by the count), voxels in ascending order of their lowest input index."""
    P = np.asarray(P, dtype=np.float64)
    fin, c = cells(P, v)
    Q = P[:, fin]
    if Q.shape[1] == 0:
        return np.zeros((3, 0))
    _, first, inv = np.unique(c.T, axis=0, return_index=True, return_inverse=True)
    inv = inv.reshape(-1)
    m = first.size
    acc = np.zeros((m, 3))
    np.add.at(acc, inv, Q.T)                      # unbuffered: one add per point, in ascending input index
    cnt = np.bincount(inv, minlength=m).astype(np.float64)
    mean = acc / cnt[:, None]
    return np.asfortranarray(mean[np.argsort(first, kind="stable")].T)


def bucket_of(cx, cy, cz, mask):
    """grid.cuh's bucket hash on int64 cell arrays (uint64 arithmetic wraps as in the kernel)."""
    with np.errstate(over="ignore"):
        k = (cx.view(np.uint64) * np.uint64(0x9E3779B97F4A7C15)) ^ (cy.view(np.uint64) * np.uint64(0xC2B2AE3D27D4EB4F)) \
            ^ (cz.view(np.uint64) * np.uint64(0x165667B19E3779F9))
        k ^= k >> np.uint64(31)
        k *= np.uint64(0xBF58476D1CE4E5B9)
        k ^= k >> np.uint64(29)
    return (k & np.uint64(mask)).astype(np.int64)


def bucket_count(n):
    nb = 1
    while nb < n:
        nb <<= 1
    return nb


def voxels_per_bucket(P, v):
    """The largest number of distinct voxels that share one bucket of the cloud's grid (bucket_count(n) buckets)."""
    P = np.asarray(P, dtype=np.float64)
    _, c = cells(P, v)
    if c.shape[1] == 0:
        return 0
    u = np.unique(c.T, axis=0)
    c = np.ascontiguousarray(u.T)
    b = bucket_of(c[0].copy(), c[1].copy(), c[2].copy(), bucket_count(P.shape[1]) - 1)
    return int(np.bincount(b).max())
