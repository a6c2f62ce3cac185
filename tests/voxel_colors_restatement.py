"""numpy restatement of the voxel filter that carries colours (csrc/k8_voxel_colors.cu; DESIGN.md section 10, "Voxel
downsampling with colours"), on tests/voxel_restatement.py's cells: the voxels are the plain filter's, and a voxel's
colour is the sum of its members' colours per channel, one float64 add per member in ascending input index from 0.0,
divided once by the count.  The GPU output must equal this bit for bit."""
import numpy as np

from tests import voxel_restatement as VR


def voxel_down_sample_colors(P, C, v):
    """(3 x m voxels, 3 x m colours): VR.voxel_down_sample's voxels and the mean colour of each voxel's members.  A
    point dropped for a non-finite coordinate drops its colour; a non-finite colour stays in its own voxel."""
    P = np.asarray(P, dtype=np.float64)
    C = np.asarray(C, dtype=np.float64)
    fin, c = VR.cells(P, v)
    Q, K = P[:, fin], C[:, fin]
    if Q.shape[1] == 0:
        return np.zeros((3, 0)), np.zeros((3, 0))
    _, first, inv = np.unique(c.T, axis=0, return_index=True, return_inverse=True)
    inv = inv.reshape(-1)
    m = first.size
    acc = np.zeros((m, 3))
    cacc = np.zeros((m, 3))
    with np.errstate(invalid="ignore"):
        np.add.at(acc, inv, Q.T)                  # unbuffered: one add per point, in ascending input index
        np.add.at(cacc, inv, K.T)
    cnt = np.bincount(inv, minlength=m).astype(np.float64)
    order = np.argsort(first, kind="stable")
    with np.errstate(invalid="ignore"):
        mean, cmean = acc / cnt[:, None], cacc / cnt[:, None]
    return np.asfortranarray(mean[order].T), np.asfortranarray(cmean[order].T)
