"""The colour-carrying voxel filter (psulvsb_voxel_down_sample_colors*, csrc/k8_voxel_colors.cu) and multi-scale
colored ICP (icp.multiscale_colored_icp*) on the GPU.  Filter: points and counts bit-identical to the plain call,
colours bit-identical to tests/voxel_colors_restatement.py, on the bunny, a seeded surface, a far-shifted cloud,
boundary / duplicate / non-finite points, tiny and empty clouds and buckets holding several voxels; determinism with a
dirty workspace on a side stream, batches against single calls in any order, host against device, 592 x 5 000 in one
device call.  Pyramid: every scale bit-identical to the three calls composed by hand, batches against batches of one,
host against device, the pinned scene of tests/multiscale_colored_icp_restatement.py, and the raw-scan chain with
colours."""
import os

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from psulvsb_b200 import capi, features, icp, stages, synth
from tests import multiscale_colored_icp_restatement as MR
from tests import voxel_colors_restatement as VCR

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bunny():
    return np.load(os.path.join(ROOT, "tests", "golden", "bunny_res3.npz"))["vertices"].astype(np.float64) * 10


@pytest.fixture(scope="module")
def surface():
    return synth.make_surface(50000, 9)


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


def colours(P, seed):
    return np.random.default_rng(seed).uniform(0.0, 1.0, P.shape)


def check(P, Cl, v):
    gv, gc = features.voxel_down_sample(P, v, colors=Cl)
    wv, wc = VCR.voxel_down_sample_colors(P, Cl, v)
    assert same(gv, features.voxel_down_sample(P, v)), (P.shape, v)
    assert same(gv, wv) and same(gc, wc), (P.shape, v, gv.shape, wv.shape)
    return gv, gc


def lattice(seed=0):
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(np.arange(6), np.arange(5), np.arange(4)), 0).reshape(3, -1).astype(np.float64)
    return g[:, rng.permutation(g.shape[1])] - 3.0


def dirty(seed=1):
    """A surface with duplicated points, NaN / Inf coordinates and a few non-finite colours."""
    rng = np.random.default_rng(seed)
    S = synth.make_surface(3000, 5)
    P = np.concatenate([S, S[:, rng.choice(3000, 400)]], axis=1)[:, rng.permutation(3400)]
    for k, bad in zip(rng.choice(3400, 60, replace=False), [np.nan, np.inf, -np.inf] * 20):
        P[rng.integers(3), k] = bad
    Cl = colours(P, seed)
    for k, bad in zip(rng.choice(3400, 12, replace=False), [np.nan, np.inf, -np.inf] * 4):
        Cl[rng.integers(3), k] = bad
    return P, Cl


# ---- against the plain filter and the restatement -------------------------------------------------------------------

def test_bunny_surface_and_far_shifted_cloud(bunny, surface):
    for P, sizes in ((bunny, (1e-4, 0.03, 0.3, 5.0)), (surface, (1e-4, 0.02, 0.2, 3.0))):
        Cl = colours(P, 3)
        counts = [check(P, Cl, v)[0].shape[1] for v in sizes]
        assert counts == sorted(counts, reverse=True) and counts[-1] <= 8, counts
    gv, gc = check(bunny, colours(bunny, 4), 1e-4)
    assert same(gv, bunny) and same(gc, colours(bunny, 4))              # one point per voxel: the input, in order
    ext = float(np.linalg.norm(np.ptp(bunny, axis=1)))
    far = bunny - bunny.mean(axis=1, keepdims=True) + 1e4 * ext * np.array([[1.0], [-0.5], [0.25]])
    for v in (0.01, 0.3):
        check(far, colours(far, 5), v)


def test_boundaries_duplicates_non_finite_tiny_and_empty():
    L = lattice()
    for v in (1.0, 2.0, 0.5):
        check(L, colours(L, 6), v)
    LL = np.concatenate([L, L, L[:, ::-1]], axis=1)
    check(LL, colours(LL, 7), 1.0)
    P, Cl = dirty()
    for v in (0.02, 0.1, 1.0):
        gv, gc = check(P, Cl, v)
        assert (~np.isfinite(gc)).any(axis=0).sum() <= 12                # a bad colour reaches its own voxel only
    v, c = features.voxel_down_sample(np.zeros((3, 0)), 0.1, colors=np.zeros((3, 0)))
    assert v.shape == (3, 0) and c.shape == (3, 0)
    one = np.array([[1.5], [-2.0], [3.25]])
    assert same(check(one, np.array([[0.1], [0.2], [0.3]]), 0.1)[1], [[0.1], [0.2], [0.3]])
    for n in (2, 127, 128, 129, 257):
        S = synth.make_surface(n, n)
        check(S, colours(S, n), 0.3)


def test_buckets_holding_several_voxels():
    P = np.random.default_rng(4).uniform(0.0, 1.0, (3, 8192))
    check(P, colours(P, 8), 1.0 / 12.0)
    Q = np.floor(np.random.default_rng(5).uniform(0.0, 1.0, (3, 300)) * 1e3) * 7.0
    check(Q, colours(Q, 9), 1.0)


# ---- determinism, host and device, batches --------------------------------------------------------------------------

def test_device_entry_dirty_workspace_side_stream(bunny, surface):
    import torch

    L = capi.lib()
    big = surface[:, :20000]
    work = torch.full((int(L.psulvsb_voxel_down_sample_colors_workspace_bytes(big.shape[1])),), 0xFF,
                      dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    for (P, Cl), v in (((big, colours(big, 1)), 0.02), ((bunny, colours(bunny, 2)), 0.05), (dirty(), 0.05),
                       ((lattice(), colours(lattice(), 3)), 1.0)):
        n = P.shape[1]
        d_pts, d_col = stages.to_device_points(P), stages.to_device_points(Cl)
        wv, wc = VCR.voxel_down_sample_colors(P, Cl, v)
        outs = []
        for _ in range(2):
            out = torch.full((n, 3), 7.0, dtype=torch.float64, device="cuda")
            oc = torch.full((n, 3), 7.0, dtype=torch.float64, device="cuda")
            cnt = torch.full((1,), -5, dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()
            capi.check(L.psulvsb_voxel_down_sample_colors(side.cuda_stream, d_pts.data_ptr(), d_col.data_ptr(), n, v,
                                                          work.data_ptr(), out.data_ptr(), oc.data_ptr(),
                                                          cnt.data_ptr()))
            side.synchronize()
            m = int(cnt.item())
            outs.append((out[:m].cpu().numpy().T, oc[:m].cpu().numpy().T))
            work.fill_(0xFF)
        assert same(outs[0][0], outs[1][0]) and same(outs[0][1], outs[1][1])
        assert same(outs[0][0], wv) and same(outs[0][1], wc)
        with torch.cuda.stream(side):
            dv, dcol, dc = features.voxel_down_sample_device(d_pts, v, work=work, colors=d_col)
        side.synchronize()
        m = int(dc.item())
        assert same(dv[:m].cpu().numpy().T, wv) and same(dcol[:m].cpu().numpy().T, wc)


def mixed(bunny):
    clouds = [bunny, lattice(2), np.zeros((3, 0)), np.full((3, 200), np.nan), synth.make_surface(5000, 3), dirty(6)[0],
              np.array([[0.5], [0.5], [0.5]]), np.zeros((3, 0)), synth.make_surface(129, 4)]
    return clouds, [colours(P, 10 + k) for k, P in enumerate(clouds)]


def test_batch_items_equal_single_calls_host_and_device(bunny):
    import torch

    clouds, cols = mixed(bunny)
    for v in (0.05, 1.0):
        want = [features.voxel_down_sample(P, v, colors=Cl) for P, Cl in zip(clouds, cols)]
        for order in (list(range(len(clouds))), list(reversed(range(len(clouds))))):
            gv, gc = features.voxel_down_sample_batch([clouds[c] for c in order], v, colors=[cols[c] for c in order])
            for k, c in enumerate(order):
                assert same(gv[k], want[c][0]) and same(gc[k], want[c][1]), (v, order, c)
            d = [stages.to_device_points(clouds[c]) for c in order]
            dcs = [stages.to_device_points(cols[c]) for c in order]
            allv, allc, counts, offsets = features.voxel_down_sample_batch_device(d, v, colors=dcs)
            torch.cuda.synchronize()
            counts = counts.cpu().numpy()
            for k, c in enumerate(order):
                sl = slice(offsets[k], offsets[k] + counts[k])
                assert same(allv[sl].cpu().numpy().T, want[c][0]) and same(allc[sl].cpu().numpy().T, want[c][1])
        for (P, Cl), w in zip(zip(clouds, cols), want):                  # B = 1
            gv, gc = features.voxel_down_sample_batch([P], v, colors=[Cl])
            assert same(gv[0], w[0]) and same(gc[0], w[1])


def test_batch_592_clouds_of_5000_on_the_device():
    import torch

    clouds = [synth.make_surface(5000, b) for b in range(592)]
    cols = [colours(P, b) for b, P in enumerate(clouds)]
    d = [stages.to_device_points(P) for P in clouds]
    dc = [stages.to_device_points(Cl) for Cl in cols]
    v = 0.04
    allv, allc, counts, offsets = features.voxel_down_sample_batch_device(d, v, colors=dc)
    plain, pcounts, _ = features.voxel_down_sample_batch_device(d, v)
    torch.cuda.synchronize()
    counts = counts.cpu().numpy()
    assert same(counts, pcounts.cpu().numpy())
    allv, allc, plain = allv.cpu().numpy(), allc.cpu().numpy(), plain.cpu().numpy()
    for b in range(592):
        sl = slice(offsets[b], offsets[b] + counts[b])
        assert same(allv[sl], plain[sl]), b
        if b % 74 == 0:
            wv, wc = VCR.voxel_down_sample_colors(clouds[b], cols[b], v)
            assert same(allv[sl].T, wv) and same(allc[sl].T, wc), b


# ---- the pyramid ----------------------------------------------------------------------------------------------------

def pyramid_pairs(B=3, n=20_000):
    out = []
    for b in range(B):
        P, Q, Cs, Ct, Rt, tt, R0, t0 = MR.scene(seed=b, n=n)
        out.append((P, Q, Cs, Ct, R0, t0))
    return out


def same_result(a, b):
    return (same(a.R, b.R) and same(a.t, b.t) and a.fitness == b.fitness and a.inlier_rmse == b.inlier_rmse
            and a.iterations == b.iterations and a.status == b.status and a.n_correspondences == b.n_correspondences
            and same(np.asarray(a.correspondences), np.asarray(b.correspondences)))


def test_pyramid_scales_equal_the_hand_composed_calls():
    pairs = pyramid_pairs()
    B = len(pairs)
    srcs, tgts, scs, tcs = ([p[k] for p in pairs] for k in range(4))
    R0s, t0s = np.array([p[4] for p in pairs]), np.array([p[5] for p in pairs])
    scales, its = MR.SCENE_SCALES, (12, 9, 7)
    got = icp.multiscale_colored_icp_batch(srcs, tgts, scs, tcs, R0s, t0s, scales, max_iterations=its)
    R, t = R0s, t0s
    for s, v in enumerate(scales):
        vox, col = features.voxel_down_sample_batch(srcs + tgts, v, colors=scs + tcs)
        nrm = features.normals_batch(vox[B:], 2.0 * v, 30)
        want = icp.colored_icp_batch(vox[:B], vox[B:], col[:B], col[B:], nrm, R, t, v, max_iterations=its[s])
        assert all(same_result(a, b) for a, b in zip(got[s], want)), s
        R, t = np.array([r.R for r in want]), np.array([r.t for r in want])
    for b in range(B):                                                   # batches of one
        one = icp.multiscale_colored_icp(srcs[b], tgts[b], scs[b], tcs[b], R0s[b], t0s[b], scales, max_iterations=its)
        assert all(same_result(one[s], got[s][b]) for s in range(len(scales))), b
    # host against device
    d = [[stages.to_device_points(a) for a in arrs] for arrs in (srcs, tgts, scs, tcs)]
    dev = icp.multiscale_colored_icp_batch_device(*d, R0s, t0s, scales, max_iterations=its)
    for s in range(len(scales)):
        for a, b in zip(dev[s], got[s]):
            a.correspondences = a.correspondences.cpu().numpy()
            assert same_result(a, b), s


def test_pinned_scene_converges_on_the_gpu_and_the_finest_scale_alone_does_not():
    P, Q, Cs, Ct, Rt, tt, R0, t0 = MR.scene()
    fine = MR.SCENE_SCALES[-1]
    res = icp.multiscale_colored_icp(P, Q, Cs, Ct, R0, t0, MR.SCENE_SCALES)
    deg, dt = MR.pose_errors(res[-1].R, res[-1].t, Rt, tt)
    print(f"pyramid: {deg:.2e} deg, {dt / fine:.2e} fine spacings, iterations {[r.iterations for r in res]}")
    assert deg < MR.MAX_DEG and dt / fine < MR.MAX_FINE
    alone = icp.multiscale_colored_icp(P, Q, Cs, Ct, R0, t0, (fine,))[0]
    assert alone.n_correspondences == 0 and alone.status == icp.NO_UPDATE
    deg1, dt1 = MR.pose_errors(alone.R, alone.t, Rt, tt)
    assert dt1 / fine > 2.0 and deg1 > 1.0


def test_colour_chain_voxel_fpfh_match_solve_then_pyramid():
    """Two coloured 200 000-point surfaces related by known rigid transforms: the colour filter, FPFH, the matcher and
    the solver find the transforms on the coarse voxels, and the pyramid refines them from there."""
    src = synth.make_surface(200000, 31)
    src_col = MR.colors_of(src)
    truth, tgts, tgt_cols = [], [], []
    for seed in (41, 42):
        R, _ = synth.random_rigid(np.random.default_rng(seed))
        t = np.array([0.4, -0.3, 0.2])
        perm = np.random.default_rng(seed + 1).permutation(src.shape[1])
        tgts.append((R @ src + t[:, None])[:, perm])
        tgt_cols.append(src_col[:, perm])
        truth.append((R, t))
    v = 0.04
    down, down_col = features.voxel_down_sample_batch([src] + tgts, v, colors=[src_col] + tgt_cols)
    out = features.fpfh_batch(down, 2.0 * v, 5.0 * v)
    matches = features.match_batch([down[0]] * 2, down[1:], [out[0][0]] * 2, [f for f, _ in out[1:]], crosscheck=True)
    problems = [capi.HostProblem(down[0][:, m[:, 0]], dn[:, m[:, 1]]) for m, dn in zip(matches, down[1:])]
    kw = dict(noise_bound=1.5 * v, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005, wallclock_cap_s=0.0,
              seed=1)
    sols = capi.Handle(0).solve_batch(capi.default_params(**kw), problems)
    assert all(s.valid for s in sols)
    res = icp.multiscale_colored_icp_batch([src] * 2, tgts, [src_col] * 2, tgt_cols, np.array([s.R for s in sols]),
                                           np.array([s.t for s in sols]), (v, v / 2, v / 4), max_iterations=(50, 30, 14))
    for s, o, (R, t) in zip(sols, res[-1], truth):
        print(f"solve: {synth.rotation_error(s.R, R):.2e} rad {np.linalg.norm(s.t - t):.2e}; "
              f"pyramid: {synth.rotation_error(o.R, R):.2e} rad {np.linalg.norm(o.t - t):.2e} fitness {o.fitness:.4f}")
        assert synth.rotation_error(s.R, R) < 0.05 and np.linalg.norm(s.t - t) < 0.1
        assert synth.rotation_error(o.R, R) < 5e-3 and np.linalg.norm(o.t - t) < 1e-2
        assert o.fitness > 0.9
