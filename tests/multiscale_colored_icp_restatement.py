"""numpy restatement of multi-scale colored ICP (icp.multiscale_colored_icp_batch; DESIGN.md section 11, "Multi-scale
colored ICP"): per scale, tests/voxel_colors_restatement.py's filter on both clouds, tests/normals_restatement.py's
hybrid normals (radius 2 v, 30 points) on the target voxels, and tests/colored_icp_restatement.py's loop from the
previous scale's result.  Test infrastructure only; also the coloured, non-planar scene the tests pin."""
import numpy as np

from tests import colored_icp_restatement as CR
from tests import normals_restatement as NR
from tests import voxel_colors_restatement as VCR

# the scene: 20 000 points of a cubic patch over [-1, 1]^2 per cloud, the coarse voxel 0.2, so 0.05 at the finest
SCENE_V = 0.2
SCENE_SCALES = (SCENE_V, SCENE_V / 2, SCENE_V / 4)
# the start is 2.5 fine voxels off the truth along z: farther than d = v / 4 from every target point
SCENE_OFFSET = 2.5 * SCENE_V / 4
MAX_DEG, MAX_FINE = 0.01, 0.01   # bounds on the pyramid's final error: degrees and fine voxel spacings


def patch(x, y):
    return 0.15 * x * x + 0.08 * x * y - 0.12 * y * y + 0.04 * x ** 3


def colors_of(P):
    I = 0.5 + 0.2 * np.sin(3.0 * P[0]) * np.cos(2.0 * P[1]) + 0.1 * P[2]
    return np.vstack([I, 0.8 * I, 1.1 * I - 0.05])


def scene(seed=0, n=20_000):
    """(P, Q, Cs, Ct, R_true, t_true, R0, t0): two independent samples of the coloured patch, Q ~ R_true P + t_true,
    and the start (identity, t_true moved SCENE_OFFSET along z)."""
    rng = np.random.default_rng(seed)

    def sample():
        xy = rng.uniform(-1.0, 1.0, (2, n))
        S = np.vstack([xy, patch(xy[0], xy[1])])
        return S, colors_of(S)

    Q, Ct = sample()
    S, Cs = sample()
    ax = np.array([0.3, -0.5, 0.8]) / np.linalg.norm([0.3, -0.5, 0.8])
    a = np.deg2rad(2.0)
    K = np.array([[0.0, -ax[2], ax[1]], [ax[2], 0.0, -ax[0]], [-ax[1], ax[0], 0.0]])
    R = np.eye(3) + np.sin(a) * K + (1.0 - np.cos(a)) * K @ K
    t = np.array([0.05, -0.03, 0.02])
    P = R.T @ (S - t[:, None])
    return P, Q, Cs, Ct, R, t, np.eye(3), t + np.array([0.0, 0.0, SCENE_OFFSET])


def pose_errors(R, t, R_true, t_true):
    """(rotation error in degrees, translation error)."""
    c = np.clip((np.trace(R @ R_true.T) - 1.0) / 2.0, -1.0, 1.0)
    return float(np.degrees(np.arccos(c))), float(np.linalg.norm(t - t_true))


def multiscale_colored_icp(P, Q, Cs, Ct, R0, t0, voxel_sizes, distances=None, max_iterations=30, lam=0.968):
    """One restatement result (colored_icp_restatement's dict) per scale."""
    distances = voxel_sizes if distances is None else distances
    its = [max_iterations] * len(voxel_sizes) if np.ndim(max_iterations) == 0 else list(max_iterations)
    R, t, out = np.asarray(R0, dtype=np.float64), np.asarray(t0, dtype=np.float64), []
    for v, d, k in zip(voxel_sizes, distances, its):
        Ps, Css = VCR.voxel_down_sample_colors(P, Cs, v)
        Qs, Cts = VCR.voxel_down_sample_colors(Q, Ct, v)
        N = NR.hybrid_normals(Qs, 2.0 * v, CR.MAX_NN)[0]
        r = CR.colored_icp(Ps, Qs, Css, Cts, N, R, t, d, lam, max_iterations=k)
        out.append(r)
        R, t = r["R"], r["t"]
    return out
