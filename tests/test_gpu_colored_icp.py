"""Colored ICP and its colour-gradient stage on the GPU against the numpy restatement
(tests/colored_icp_restatement.py): the gradients, every trace record step-locked for several lambdas and each loss,
lambda = 1 against point-to-plane ICP bit for bit, batches against single calls, determinism, the textured plane on
which point-to-plane stalls, a 592-pair batch and the normals -> colored ICP chain after the batch solver."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

import psulvsb_b200  # noqa: F401
from oracle import icp as OI
from psulvsb_b200 import capi, features, icp, synth
from tests import colored_icp_restatement as CR
from tests.test_colored_icp import PLANE_D, PLANE_MAX_DEG, PLANE_MAX_T, pose_errors, textured_plane
from tests.test_gpu_gicp import radius_normals, same
from tests.test_gpu_icp import bunny, extent, scene, spacing  # noqa: F401  (bunny: a fixture)
from tests.test_gpu_robust_icp import losses

pytestmark = pytest.mark.gpu


def colour_field(X, scale):
    """Smooth [0, 1] RGB over world coordinates, varying on the scale `scale`."""
    x, y, z = X / scale
    return np.clip(np.vstack([0.5 + 0.3 * np.sin(x) * np.cos(y), 0.5 + 0.3 * np.sin(y + 0.5 * z),
                              0.5 + 0.3 * np.cos(z - x)]), 0.0, 1.0)


def coloured_scene(P, seed):
    """tests/test_gpu_icp.scene with colours: the source's from the field at its true world position (its outliers'
    too), the target's at its own; target radius normals (NaN where too few neighbours)."""
    src, tgt, R, t, R0, t0, d = scene(P, seed)
    sc = 0.1 * extent(P)
    Cs = colour_field(R @ src + t[:, None], sc)
    Ct = colour_field(tgt, sc)
    Nt = radius_normals(tgt, 4 * spacing(P))
    return src, tgt, Cs, Ct, Nt, R, t, R0, t0, d


def gpu_gradients(Q, Ct, Nt, d):
    """The target gradients colored ICP computes inside its call: radius 2 d, max_nn 30, the same kernel."""
    return features.color_gradients(Q, Ct, Nt, 2.0 * d, CR.MAX_NN)


def bits_equal(a, b):
    return np.ascontiguousarray(a).tobytes() == np.ascontiguousarray(b).tobytes()


def same_bits(a, b):
    """`same`, with the transforms and traces compared bit for bit (signed zeros included)."""
    return same(a, b) and bits_equal(a.R, b.R) and bits_equal(a.t, b.t) and \
        (a.trace is None or all(bits_equal(a.trace[k], b.trace[k]) for k in a.trace))


def check_step_locked(src, tgt, Cs, Ct, Nt, Gt, d, lam, loss, out, *, max_iterations=30, relative_fitness=1e-6,
                      relative_rmse=1e-6):
    """Every trace record k against the restatement at the GPU's T_k with the GPU's gradients: correspondences, counts,
    fitness and rmse exact (rmse to the last bits of its sum's order), T_{k+1} within the robust tests' tolerances; the
    stop rule applied to the trace."""
    tr = out.trace
    K = len(tr["fitness"])
    assert K == out.iterations + 1
    scale = max(extent(tgt), np.abs(tgt).max(initial=0.0), 1e-300)
    keep = OI.candidate_mask(tgt, Nt)
    tree = cKDTree(tgt[:, keep].T) if keep.any() else None
    prev = None
    for k in range(K):
        chk = CR.step_check(src, tgt, Nt, Gt, Cs, Ct, d, tr["R"][k], tr["t"][k], lam, loss, tree)
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
        prev = cur


def test_gradients_against_the_restatement_and_batches(bunny):
    src, tgt, Cs, Ct, Nt, R, t, R0, t0, d = coloured_scene(bunny, 81)
    S = synth.make_surface(50_000, 4)
    Cq = colour_field(S, 0.1 * extent(S))
    Nq = radius_normals(S, 4 * spacing(S))
    Nq[:, ::13] = np.nan
    for P, Cc, N, r in ((tgt, Ct, Nt, 2 * d), (S, Cq, Nq, 6 * spacing(S))):
        G = features.color_gradients(P, Cc, N, r)
        Gr, frag = CR.gradients(P, Cc, N, r)
        ok = ~frag
        assert ok.mean() > 0.95
        gmax = np.abs(Gr).max()
        err = np.abs(G - Gr)[:, ok].max()
        assert err <= 1e-9 * gmax, err
        assert np.array_equal(G[:, ~np.isfinite(N).all(axis=0)], np.zeros((3, int((~np.isfinite(N).all(axis=0)).sum()))))
    clouds = [tgt, S[:, :0], S, tgt[:, :3]]
    cols = [Ct, Cq[:, :0], Cq, Ct[:, :3]]
    nrms = [Nt, Nq[:, :0], Nq, Nt[:, :3]]
    got = features.color_gradients_batch(clouds, cols, nrms, 2 * d, 24)
    for c, g in enumerate(got):
        assert bits_equal(g, features.color_gradients_batch([clouds[c]], [cols[c]], [nrms[c]], 2 * d, 24)[0]), c
    assert np.array_equal(got[3], np.zeros((3, 3)))
    import torch

    from psulvsb_b200 import stages
    dev = lambda a: stages.to_device_points(a) if a.shape[1] else torch.empty(  # noqa: E731
        (0, 3), dtype=torch.float64, device="cuda")
    work = torch.full((int(1e8),), 0xFF, dtype=torch.uint8, device="cuda")
    _, views = features.color_gradients_batch_device([dev(a) for a in clouds], [dev(a) for a in cols],
                                                     [dev(a) for a in nrms], 2 * d, 24, work=work)
    for v, g in zip(views, got):
        assert bits_equal(np.asfortranarray(v.cpu().numpy().T), g)


@pytest.mark.parametrize("lam", [0.968, 0.5, 0.0])
@pytest.mark.parametrize("name", ["l2", "huber", "cauchy", "gm", "tukey"])
def test_step_locked_vs_restatement(bunny, lam, name):
    src, tgt, Cs, Ct, Nt, R, t, R0, t0, d = coloured_scene(bunny, 82)
    loss = None if name == "l2" else losses(0.002 * extent(bunny))[name]
    out = icp.colored_icp(src, tgt, Cs, Ct, Nt, R0, t0, d, lambda_geometric=lam, loss=loss, trace=True)
    check_step_locked(src, tgt, Cs, Ct, Nt, gpu_gradients(tgt, Ct, Nt, d), d, lam, loss, out)
    if lam > 0.0 and name == "l2":
        assert out.iterations >= 2 and out.fitness > 0.4


def test_lambda_one_is_point_to_plane_bit_for_bit(bunny):
    src, tgt, Cs, Ct, Nt, R, t, R0, t0, d = coloured_scene(bunny, 83)
    Nt[:, ::9] = np.nan
    kw = dict(trace=True)
    want = icp.icp(src, tgt, R0, t0, d, target_normals=Nt, point_to_plane=True, **kw)
    got = icp.colored_icp(src, tgt, Cs, Ct, Nt, R0, t0, d, lambda_geometric=1.0, **kw)
    assert same_bits(got, want) and want.iterations >= 2
    assert same_bits(icp.colored_icp(src, tgt, Cs, Ct, Nt, R0, t0, d, lambda_geometric=1.0, loss=icp.L2Loss(), **kw),
                     want)
    # a plane: p' x n has exact zeros of both signs there
    P, Q, Cps, Cpt, Npt, _, _ = textured_plane(3, n=5000)
    R1, t1 = np.eye(3), np.array([0.0, 0.0, 0.05])
    a = icp.colored_icp(P, Q, Cps, Cpt, Npt, R1, t1, PLANE_D, lambda_geometric=1.0, **kw)
    b = icp.icp(P, Q, R1, t1, PLANE_D, target_normals=Npt, point_to_plane=True, **kw)
    assert same_bits(a, b)


def test_no_loss_is_the_l2_loss(bunny):
    src, tgt, Cs, Ct, Nt, R, t, R0, t0, d = coloured_scene(bunny, 84)
    kw = dict(trace=True, lambda_geometric=0.8)
    assert same_bits(icp.colored_icp(src, tgt, Cs, Ct, Nt, R0, t0, d, **kw),
                     icp.colored_icp(src, tgt, Cs, Ct, Nt, R0, t0, d, loss=icp.L2Loss(), **kw))


def mixed_colored_batch(bunny):
    """(src, tgt, Cs, Ct, Nt, R0, t0) of an empty-source, empty-target, tiny, far-away and 50k pair, and d."""
    rng = np.random.default_rng(6)
    P = bunny[:, :40]
    Cc = rng.uniform(size=P.shape)
    N = rng.normal(size=P.shape)
    items = [(P[:, :0], P, Cc[:, :0], Cc, N, np.eye(3), np.zeros(3)),
             (P, P[:, :0], Cc, Cc[:, :0], N[:, :0], np.eye(3), np.zeros(3)),
             (P[:, :2], P, Cc[:, :2], Cc, N, np.eye(3), np.zeros(3))]
    src, tgt, Cs, Ct, Nt, R, t, R0, t0, d = coloured_scene(bunny[:, ::2], 85)
    off = 1e6 * d * np.array([1.0, -0.7, 0.4])
    items.append((src + off[:, None], tgt + off[:, None], Cs, Ct, Nt, R0, t0 + off - R0 @ off))
    S = synth.make_surface(50_000, 4)
    src, tgt, Cs, Ct, Nt, R, t, R0, t0, _ = coloured_scene(S, 86)
    items.append((src, tgt, Cs, Ct, Nt, R0, t0))
    return items, d


def test_batches_are_single_calls_whatever_the_permutation(bunny):
    import torch

    from psulvsb_b200 import stages

    items, d = mixed_colored_batch(bunny)
    loss = icp.HuberLoss(0.5 * d)
    kw = dict(trace=True, max_iterations=15, loss=loss, lambda_geometric=0.9)
    want = [icp.colored_icp(*it, d, **kw) for it in items]

    def batch(order, device=False):
        its = [items[k] for k in order]
        R0s, t0s = np.array([it[5] for it in its]), np.array([it[6] for it in its])
        if not device:
            return icp.colored_icp_batch(*zip(*[it[:5] for it in its]), R0s, t0s, d, **kw)
        dev = lambda a: stages.to_device_points(a) if a.shape[1] else torch.empty(  # noqa: E731
            (0, 3), dtype=torch.float64, device="cuda")
        cols = [[dev(it[j]) for it in its] for j in range(5)]
        work = torch.full((int(2e8),), 0xFF, dtype=torch.uint8, device="cuda")
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            res = icp.colored_icp_batch_device(*cols, R0s, t0s, d, work=work, **kw)
        side.synchronize()
        for r in res:
            r.correspondences = r.correspondences.cpu().numpy()
        return res

    ident = list(range(len(items)))
    assert all(same_bits(g, w) for g, w in zip(batch(ident), want))
    perm = list(np.random.default_rng(3).permutation(len(items)))
    assert all(same_bits(g, want[k]) for k, g in zip(perm, batch(perm)))
    assert all(same_bits(g, want[k]) for k, g in zip(perm[::-1], batch(perm[::-1], device=True)))
    assert want[0].status == want[1].status == want[2].status == OI.NO_UPDATE and want[0].iterations == 0
    assert want[4].iterations >= 2


def test_determinism_dirty_workspace_and_side_stream(bunny):
    import torch

    from psulvsb_b200 import stages

    src, tgt, Cs, Ct, Nt, R, t, R0, t0, d = coloured_scene(bunny, 87)
    kw = dict(trace=True, relative_fitness=0, relative_rmse=0, max_iterations=12, loss=icp.CauchyLoss(0.01))
    a = icp.colored_icp(src, tgt, Cs, Ct, Nt, R0, t0, d, **kw)
    assert same_bits(a, icp.colored_icp(src, tgt, Cs, Ct, Nt, R0, t0, d, **kw))
    dv = [stages.to_device_points(x) for x in (src, tgt, Cs, Ct, Nt)]
    side = torch.cuda.Stream()
    nbytes = capi.lib().psulvsb_colored_icp_workspace_bytes(src.shape[1], tgt.shape[1])
    work = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    for _ in range(2):                              # the second call finds the first one's leftovers
        with torch.cuda.stream(side):
            c = icp.colored_icp_device(*dv, R0, t0, d, work=work, **kw)
        side.synchronize()
        c.correspondences = c.correspondences.cpu().numpy()
        assert same_bits(c, a)
    assert a.status == OI.MAX_ITERATIONS and a.iterations == 12


def test_textured_plane_point_to_plane_stalls_and_colored_icp_recovers_the_motion():
    for seed in (0, 1):
        P, Q, Cs, Ct, Nt, R_true, t_true = textured_plane(seed)
        p2l = icp.icp(P, Q, np.eye(3), np.zeros(3), PLANE_D, target_normals=Nt, point_to_plane=True)
        assert p2l.status == OI.NO_UPDATE and p2l.iterations == 0
        Gt = gpu_gradients(Q, Ct, Nt, PLANE_D)
        for lam in (0.968, 0.5):
            out = icp.colored_icp(P, Q, Cs, Ct, Nt, np.eye(3), np.zeros(3), PLANE_D, lambda_geometric=lam, trace=True)
            err = pose_errors(out.R, out.t, R_true, t_true)
            print("plane", seed, lam, out.status, out.iterations, err)
            assert out.status == OI.CONVERGED and out.iterations >= 2
            assert err[0] < PLANE_MAX_DEG and err[1] < PLANE_MAX_T, (seed, lam, err)
            check_step_locked(P, Q, Cs, Ct, Nt, Gt, PLANE_D, lam, None, out)


def test_592_pairs_of_5000_points():
    rng = np.random.default_rng(0)
    srcs, tgts, css, cts, nts, R0s, t0s = [], [], [], [], [], [], []
    sp = 2.0 / np.sqrt(5000)
    normals = {}
    for b in range(592):
        S = synth.make_surface(5000, b % 37)
        if b % 37 not in normals:
            normals[b % 37] = radius_normals(S, 4 * sp)
        R, _ = synth.random_rigid(rng)
        t = rng.normal(size=3)
        C = colour_field(S, 0.2)
        srcs.append(S + rng.normal(0, 0.1 * sp, S.shape))
        tgts.append(R @ S + t[:, None])
        css.append(C)
        cts.append(C)
        nts.append(R @ normals[b % 37])
        a = np.deg2rad(2.0)
        R0s.append(R @ (np.cos(a) * np.eye(3) + np.sin(a) * np.array([[0, -1, 0], [1, 0, 0], [0, 0, 0]]) +
                        (1 - np.cos(a)) * np.diag([0, 0, 1.0])))
        t0s.append(t + 0.01 * rng.normal(size=3))
    d = 3 * sp
    got = icp.colored_icp_batch(srcs, tgts, css, cts, nts, np.array(R0s), np.array(t0s), d)
    for b in (0, 1, 295, 591):
        want = icp.colored_icp(srcs[b], tgts[b], css[b], cts[b], nts[b], R0s[b], t0s[b], d)
        assert same_bits(got[b], want), b
    assert np.mean([g.fitness for g in got]) > 0.95


def test_normals_batch_then_colored_icp_batch_after_the_solver(bunny):
    """The chain of INTEGRATION.md section 5: the batch solver on known correspondences, the targets' hybrid normals,
    then colored ICP on a coloured scene."""
    ext = extent(bunny)
    rng = np.random.default_rng(21)
    tgts, cts, truth, problems = [], [], [], []
    Cb = colour_field(bunny, 0.1 * ext)
    for seed in (31, 32):
        R, _ = synth.random_rigid(np.random.default_rng(seed))
        t = np.array([0.4, -0.3, 0.2])
        tgt = R @ bunny + t[:, None] + rng.normal(0, 0.001 * ext, bunny.shape)
        tgts.append(tgt)
        cts.append(Cb)
        truth.append((R, t))
        idx = rng.choice(bunny.shape[1], 300, replace=False)
        dst = tgt[:, idx].copy()
        dst[:, :60] = rng.uniform(tgt.min(axis=1)[:, None], tgt.max(axis=1)[:, None], (3, 60))
        problems.append(capi.HostProblem(bunny[:, idx], dst))
    kw = dict(noise_bound=0.01 * ext, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005,
              wallclock_cap_s=0.0, seed=1)
    sols = capi.Handle(0).solve_batch(capi.default_params(**kw), problems)
    assert all(s.valid for s in sols)
    d = 3.0 * spacing(bunny)
    nts = features.normals_batch(tgts, 4 * spacing(bunny), 30)
    res = icp.colored_icp_batch([bunny] * 2, tgts, [Cb] * 2, cts, nts, np.array([s.R for s in sols]),
                                np.array([s.t for s in sols]), d)
    for o, s, (R, t) in zip(res, sols, truth):
        print("solve", synth.rotation_error(s.R, R), "colored", synth.rotation_error(o.R, R), o.fitness, o.iterations)
        assert o.status in (OI.CONVERGED, OI.MAX_ITERATIONS) and o.fitness > 0.95
        assert synth.rotation_error(o.R, R) <= max(synth.rotation_error(s.R, R), 1e-3)
        assert np.linalg.norm(o.t - t) <= max(np.linalg.norm(s.t - t), 1e-3 * ext)
