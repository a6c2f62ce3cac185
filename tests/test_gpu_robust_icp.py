"""Robust kernels of point-to-plane ICP and generalized ICP on the GPU against the numpy restatement
(tests/robust_icp_restatement.py): step-locked on every trace record for each loss and both objectives, the L2 loss
against the plain calls, batches against single calls, determinism, an outlier scene and an all-zero weight."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

import psulvsb_b200  # noqa: F401
from oracle import icp as OI
from psulvsb_b200 import capi, icp, synth
from psulvsb_b200 import io as pio
from tests import robust_icp_restatement as RR
from tests.test_gpu_gicp import bunny, mixed_batch, radius_normals, same  # noqa: F401  (bunny: a fixture)
from tests.test_gpu_icp import extent, scene, spacing
from tests.test_robust_icp import OUTLIER_D, OUTLIER_START, outlier_scene, pose_errors

pytestmark = pytest.mark.gpu


def losses(sigma):
    """One kernel of each type at a scale of a few noise sigmas (GM's k is a squared residual)."""
    return {"l2": icp.L2Loss(), "huber": icp.HuberLoss(3 * sigma), "cauchy": icp.CauchyLoss(3 * sigma),
            "gm": icp.GMLoss((3 * sigma) ** 2), "tukey": icp.TukeyLoss(5 * sigma)}


def objective_kw(objective, Ns, Nt):
    """The restatement's keywords of an objective."""
    return dict(normals=Nt) if objective == "p2l" else dict(src_normals=Ns, tgt_normals=Nt, epsilon=1e-3)


def run(objective, src, tgt, Ns, Nt, R0, t0, d, loss, **kw):
    if objective == "p2l":
        return icp.icp(src, tgt, R0, t0, d, target_normals=Nt, point_to_plane=True, loss=loss, **kw)
    return icp.gicp(src, tgt, Ns, Nt, R0, t0, d, loss=loss, **kw)


def check_step_locked(objective, src, tgt, Ns, Nt, d, loss, out, *, max_iterations=30, relative_fitness=1e-6,
                      relative_rmse=1e-6):
    """Every trace record k against the restatement evaluated at the GPU's T_k: correspondences, counts, fitness and
    rmse exact (rmse to the last bits of its sum's order), T_{k+1} within the GICP tests' tolerances; the stop rule
    applied to the trace."""
    tr = out.trace
    K = len(tr["fitness"])
    assert K == out.iterations + 1
    scale = max(extent(tgt), np.abs(tgt).max(initial=0.0), 1e-300)
    okw = objective_kw(objective, Ns, Nt)
    keep = OI.candidate_mask(tgt, Nt if objective == "p2l" else None)
    tree = cKDTree(tgt[:, keep].T) if keep.any() else None
    prev = None
    for k in range(K):
        chk = RR.step_check(src, tgt, d, tr["R"][k], tr["t"][k], loss, tree=tree, **okw)
        assert tr["n_correspondences"][k] == chk["n_corr"], k
        assert tr["fitness"][k] == chk["fitness"], k
        assert abs(tr["inlier_rmse"][k] - chk["inlier_rmse"]) <= 1e-12 * chk["inlier_rmse"], k
        cur = (tr["fitness"][k], tr["inlier_rmse"][k])
        status = OI.stop(k, prev, cur, max_iterations, relative_fitness, relative_rmse)
        if k < K - 1:
            assert status is None and chk["next"] is not None, k
            Rn, tn = chk["next"]
            assert np.abs(tr["R"][k + 1] - Rn).max() <= 1e-10, (k, np.abs(tr["R"][k + 1] - Rn).max())
            assert np.abs(tr["t"][k + 1] - tn).max() <= 1e-10 * scale, (k, np.abs(tr["t"][k + 1] - tn).max())
        else:
            if status is None:
                assert chk["next"] is None
                status = OI.NO_UPDATE
            assert out.status == status
            assert np.array_equal(out.correspondences, chk["corr"])
            assert np.array_equal(out.R, tr["R"][k]) and np.array_equal(out.t, tr["t"][k])
            assert out.fitness == cur[0] and out.inlier_rmse == cur[1] and out.n_correspondences == chk["n_corr"]
        prev = cur


@pytest.mark.parametrize("objective", ["p2l", "gicp"])
@pytest.mark.parametrize("name", ["l2", "huber", "cauchy", "gm", "tukey"])
def test_step_locked_vs_restatement(bunny, objective, name):
    src, tgt, R, t, R0, t0, d = scene(bunny, 71)
    Ns, Nt = pio.estimate_normals(src, 20), pio.estimate_normals(tgt, 20)
    loss = losses(0.002 * extent(bunny))[name]
    out = run(objective, src, tgt, Ns, Nt, R0, t0, d, loss, trace=True)
    check_step_locked(objective, src, tgt, Ns, Nt, d, loss, out)
    assert out.iterations >= 2 and out.fitness > 0.4


@pytest.mark.parametrize("objective", ["p2l", "gicp"])
def test_step_locked_on_a_surface_with_radius_normals(objective):
    """NaN radius normals: point-to-plane drops those targets, GICP gives them covariance I (W = I / sqrt2)."""
    S = synth.make_surface(50_000, 4)
    src, tgt, R, t, R0, t0, d = scene(S, 72)
    rn = 4 * spacing(S)
    Ns, Nt = radius_normals(src, rn), radius_normals(tgt, rn)
    Nt[:, ::11] = np.nan
    Ns[:, 5::13] = 0.0
    loss = icp.TukeyLoss(0.01 * extent(S))
    out = run(objective, src, tgt, Ns, Nt, R0, t0, d, loss, trace=True)
    check_step_locked(objective, src, tgt, Ns, Nt, d, loss, out)
    assert out.iterations >= 2


def test_l2_point_to_plane_is_psulvsb_icp_bit_for_bit(bunny):
    src, tgt, R, t, R0, t0, d = scene(bunny, 73)
    Nt = radius_normals(tgt, 4 * spacing(bunny))
    Nt[:, ::9] = np.nan                                              # targets left out of the grid
    kw = dict(target_normals=Nt, point_to_plane=True, trace=True)
    assert same(icp.icp(src, tgt, R0, t0, d, loss=icp.L2Loss(), **kw), icp.icp(src, tgt, R0, t0, d, **kw))
    items, db = mixed_batch(bunny)
    srcs, tgts, nts = [it[0] for it in items], [it[1] for it in items], [it[3] for it in items]
    R0s, t0s = np.array([it[4] for it in items]), np.array([it[5] for it in items])
    kw = dict(target_normals=nts, point_to_plane=True, trace=True, max_iterations=15)
    a = icp.icp_batch(srcs, tgts, R0s, t0s, db, loss=icp.L2Loss(), **kw)
    b = icp.icp_batch(srcs, tgts, R0s, t0s, db, **kw)
    assert all(same(x, y) for x, y in zip(a, b))
    assert a[4].iterations >= 2


def test_l2_gicp_is_close_to_psulvsb_gicp(bunny):
    """W^T W = M, so the two systems are equal but for rounding: per correspondence ~1e-15 relative (W's closed form
    and products against M's adjugate), summed in another order.  On the bunny (extent ~2, near the origin, condition
    of the 6x6 system ~1e4) that moves each update by ~1e-12; over 10 rounds with the same correspondences, T agrees to
    1e-9."""
    src, tgt, R, t, R0, t0, d = scene(bunny, 74)
    Ns, Nt = pio.estimate_normals(src, 20), pio.estimate_normals(tgt, 20)
    kw = dict(trace=True, max_iterations=10, relative_fitness=0, relative_rmse=0)
    a = icp.gicp(src, tgt, Ns, Nt, R0, t0, d, loss=icp.L2Loss(), **kw)
    b = icp.gicp(src, tgt, Ns, Nt, R0, t0, d, **kw)
    assert np.array_equal(a.trace["n_correspondences"], b.trace["n_correspondences"])
    assert np.array_equal(a.correspondences, b.correspondences)
    assert np.abs(a.trace["R"] - b.trace["R"]).max() <= 1e-9
    assert np.abs(a.trace["t"] - b.trace["t"]).max() <= 1e-9 * extent(tgt)


@pytest.mark.parametrize("objective", ["p2l", "gicp"])
def test_batch_items_are_single_calls_whatever_the_permutation(bunny, objective):
    import torch

    from psulvsb_b200 import stages

    items, d = mixed_batch(bunny)
    loss = icp.HuberLoss(0.5 * d)
    kw = dict(trace=True, max_iterations=15)
    want = [run(objective, s, q, ns, nt, R0, t0, d, loss, **kw) for s, q, ns, nt, R0, t0 in items]

    def batch(order, device=False):
        its = [items[k] for k in order]
        R0s, t0s = np.array([it[4] for it in its]), np.array([it[5] for it in its])
        if not device:
            if objective == "p2l":
                return icp.icp_batch([it[0] for it in its], [it[1] for it in its], R0s, t0s, d,
                                     target_normals=[it[3] for it in its], point_to_plane=True, loss=loss, **kw)
            return icp.gicp_batch(*zip(*[it[:4] for it in its]), R0s, t0s, d, loss=loss, **kw)
        dev = lambda a: stages.to_device_points(a) if a.shape[1] else torch.empty(  # noqa: E731
            (0, 3), dtype=torch.float64, device="cuda")
        cols = [[dev(it[j]) for it in its] for j in range(4)]
        work = torch.full((int(2e8),), 0xFF, dtype=torch.uint8, device="cuda")
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            if objective == "p2l":
                res = icp.icp_batch_device(cols[0], cols[1], R0s, t0s, d, d_target_normals=cols[3],
                                           point_to_plane=True, work=work, loss=loss, **kw)
            else:
                res = icp.gicp_batch_device(*cols, R0s, t0s, d, work=work, loss=loss, **kw)
        side.synchronize()
        for r in res:
            r.correspondences = r.correspondences.cpu().numpy()
        return res

    ident = list(range(len(items)))
    assert all(same(g, w) for g, w in zip(batch(ident), want))
    perm = list(np.random.default_rng(3).permutation(len(items)))
    assert all(same(g, want[k]) for k, g in zip(perm, batch(perm)))
    assert all(same(g, want[k]) for k, g in zip(perm[::-1], batch(perm[::-1], device=True)))
    assert want[0].status == want[1].status == OI.NO_UPDATE and want[0].iterations == 0
    assert want[4].iterations >= 2


@pytest.mark.parametrize("objective", ["p2l", "gicp"])
def test_determinism_dirty_workspace_and_side_stream(bunny, objective):
    import torch

    from psulvsb_b200 import stages

    src, tgt, R, t, R0, t0, d = scene(bunny, 75)
    Ns, Nt = pio.estimate_normals(src, 20), pio.estimate_normals(tgt, 20)
    loss = icp.CauchyLoss(0.006 * extent(bunny))
    kw = dict(trace=True, relative_fitness=0, relative_rmse=0, max_iterations=12)
    a = run(objective, src, tgt, Ns, Nt, R0, t0, d, loss, **kw)
    assert same(a, run(objective, src, tgt, Ns, Nt, R0, t0, d, loss, **kw))
    ds, dt = stages.to_device_points(src), stages.to_device_points(tgt)
    dns, dnt = stages.to_device_points(Ns), stages.to_device_points(Nt)
    side = torch.cuda.Stream()
    nbytes = capi.lib().psulvsb_icp_workspace_bytes(src.shape[1], tgt.shape[1])
    work = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    for _ in range(2):                              # the second call finds the first one's leftovers
        with torch.cuda.stream(side):
            if objective == "p2l":
                c = icp.icp_device(ds, dt, R0, t0, d, d_target_normals=dnt, point_to_plane=True, work=work,
                                   loss=loss, **kw)
            else:
                c = icp.gicp_device(ds, dt, dns, dnt, R0, t0, d, work=work, loss=loss, **kw)
        side.synchronize()
        c.correspondences = c.correspondences.cpu().numpy()
        assert same(c, a)
    assert a.status == OI.MAX_ITERATIONS and a.iterations == 12


@pytest.mark.parametrize("objective", ["p2l", "gicp"])
def test_robust_kernels_beat_l2_on_structured_outliers(objective):
    """The clutter sheet of test_robust_icp.outlier_scene: L2's translation lands about 0.015 off; Tukey and Cauchy
    with k = 5 sigma land at least 5 times closer, step-locked with the restatement."""
    for seed in (0, 1, 2):
        S, Sn, Q, Nt, R_true, t_true = outlier_scene(seed)
        R0, t0 = OUTLIER_START[0] @ R_true, t_true + OUTLIER_START[1]
        err = {}
        for name, loss in (("l2", icp.L2Loss()), ("tukey", icp.TukeyLoss(0.01)), ("cauchy", icp.CauchyLoss(0.01))):
            out = run(objective, S, Q, Sn, Nt, R0, t0, OUTLIER_D, loss, trace=True)
            check_step_locked(objective, S, Q, Sn, Nt, OUTLIER_D, loss, out)
            err[name] = pose_errors(out.R, out.t, R_true, t_true)
        assert err["l2"][1] > 0.01, err
        for name in ("tukey", "cauchy"):
            assert err[name][1] < err["l2"][1] / 5, (seed, name, err)


@pytest.mark.parametrize("objective", ["p2l", "gicp"])
def test_tukey_with_every_weight_zero_stops_at_t0(bunny, objective):
    """k far below every residual: J^T J = 0, the Cholesky's first pivot is 0, so no update and T = T0."""
    src, tgt, R, t, R0, t0, d = scene(bunny, 76)
    Ns, Nt = pio.estimate_normals(src, 20), pio.estimate_normals(tgt, 20)
    out = run(objective, src, tgt, Ns, Nt, R0, t0, d, icp.TukeyLoss(1e-30), trace=True)
    assert out.status == OI.NO_UPDATE and out.iterations == 0 and out.n_correspondences > 100
    assert np.array_equal(out.R, R0) and np.array_equal(out.t, t0)
    check_step_locked(objective, src, tgt, Ns, Nt, d, icp.TukeyLoss(1e-30), out)
