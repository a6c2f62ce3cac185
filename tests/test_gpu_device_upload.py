"""psulvsb_batch_upload_device (Handle.upload_device / solve_batch_device): solutions bit-identical, field by field, to
psulvsb_solve_batch on the same arrays from the host -- mixed aliased and pre-filtered batches split over several
engines, the cfg-B shape, inputs produced behind a long kernel on a side stream, signed zeros, and the raw-scan chain on
device buffers; every refusal and what it leaves behind."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PKW = dict(noise_bound=0.05, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005, wallclock_cap_s=0.0)


@pytest.fixture(scope="module")
def env():
    import torch

    import psulvsb_b200  # noqa: F401
    from psulvsb_b200 import capi, features, icp, synth

    if capi.lib().psulvsb_device_count() < 1:
        pytest.fail("no CUDA device: the product has no CPU fallback")
    h = capi.Handle(0)
    yield {"capi": capi, "synth": synth, "features": features, "icp": icp, "torch": torch, "h": h}
    h.close()


def same(a, b):
    """Two lists of psulvsb_solution_t, equal bit for bit in every field."""
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        for name, ty in x._fields_:
            u, v = getattr(x, name), getattr(y, name)
            if ty in (C.c_double,) or hasattr(u, "__len__"):
                u, v = np.array(u, dtype=np.float64).tobytes(), np.array(v, dtype=np.float64).tobytes()
            assert u == v, (i, name, getattr(x, name), getattr(y, name))


def is_aliased(hp):
    return (hp.ori_src.ctypes.data == hp.src.ctypes.data and hp.ori_dst.ctypes.data == hp.dst.ctypes.data
            and hp.ori_src.shape == hp.src.shape)


def to_device(env, hp):
    """The DeviceProblem of a HostProblem: the same arrays on the device (ori_* alias src / dst where they do on the
    host)."""
    capi, torch = env["capi"], env["torch"]
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a.T)).cuda()  # noqa: E731  3xN column-major == [N, 3]
    src, dst = d(hp.src), d(hp.dst)
    if is_aliased(hp):
        return capi.DeviceProblem(src, dst)
    return capi.DeviceProblem(src, dst, d(hp.ori_src), d(hp.ori_dst), torch.from_numpy(hp.keep_mask).cuda(),
                              torch.from_numpy(hp.reduce_map).cuda())


def prefiltered(env, n, seed, outliers=0.9):
    capi, synth = env["capi"], env["synth"]
    pair = synth.make_pair(n, outliers, seed)
    pre = synth.prefilter(pair, seed)
    return capi.HostProblem(pre["src_reduce"], pre["dst_reduce"], pair["src"], pair["dst"], pre["keep_mask"],
                            pre["reduce_map"])


def aliased(env, n, seed, outliers=0.9):
    p = env["synth"].make_pair(n, outliers, seed)
    return env["capi"].HostProblem(p["src"], p["dst"])


SIZES = [64, 300, 1200, 5000, 500, 2000, 800, 150, 3000, 700, 64]


@pytest.fixture(scope="module")
def mixed(env):
    host = [(aliased if i % 2 == 0 else prefiltered)(env, n, 900 + i) for i, n in enumerate(SIZES)]
    masks = np.concatenate([p.keep_mask for p in host[1::2]])
    assert set(np.unique(masks)) == {-1, 0, 1}
    return host, [to_device(env, p) for p in host]


def test_mixed_batches_equal_the_host_path(env, mixed):
    capi, h = env["capi"], env["h"]
    host, dev = mixed
    assert all(d.aliased for d in dev[0::2]) and not any(d.aliased for d in dev[1::2])
    params = capi.default_params(seed=17, **PKW)
    seeds = list(range(300, 300 + len(host)))
    h.set_batching(0, 0)
    ref = h.solve_batch(params, host)
    ref_seeded = h.solve_batch(params, host, seeds)
    assert all(s.status == 0 for s in ref)
    for chunk, lanes in ((0, 0), (3, 2), (4, 3), (2, 4)):
        h.set_batching(chunk, lanes)
        same(ref, h.solve_batch_device(params, dev))
        assert h.resident_size == len(dev)
        same(ref_seeded, h.solve_resident(params, seeds))
        same(ref, h.solve_resident(params))
        # and the host upload on the same split
        h.upload(host)
        same(ref_seeded, h.solve_resident(params, seeds))
    h.set_batching(0, 0)


def test_cfg_b_shape(env):
    """One 100 000-correspondence registration at 99 % outliers (the cfg-B workload)."""
    capi, synth, h = env["capi"], env["synth"], env["h"]
    pair = synth.make_pair(100_000, 0.99, 4242, side=30.0)
    hp = capi.HostProblem(pair["src"], pair["dst"])
    params = capi.default_params(seed=11, **PKW)
    ref = h.solve_batch(params, [hp])
    same(ref, h.solve_batch_device(params, [to_device(env, hp)]))


def test_inputs_from_a_side_stream_and_reuse_after_the_call(env, mixed):
    """The inputs are produced on a non-default stream behind a long kernel; the upload waits for them.  Once the call
    has returned the tensors are overwritten, and the resident batch still solves to the reference, twice."""
    capi, torch, h = env["capi"], env["torch"], env["h"]
    host, dev = mixed
    params = capi.default_params(seed=5, **PKW)
    ref = h.solve_batch(params, host)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)  # about 0.1 s of one SM spinning ahead of the producers
        made = []
        for d in dev:  # fresh tensors, written on the side stream only
            if d.aliased:
                made.append(capi.DeviceProblem(d.src * 1.0, d.dst * 1.0))
            else:
                made.append(capi.DeviceProblem(d.src * 1.0, d.dst * 1.0, d.ori_src * 1.0, d.ori_dst * 1.0,
                                               d.keep_mask.clone(), d.reduce_map.clone()))
        h.upload_device(made)
        for m in made:
            for t in (m.src, m.dst, m.ori_src, m.ori_dst):
                t.fill_(float("nan"))
            m.keep_mask.fill_(7)
            m.reduce_map.fill_(-5)
    side.synchronize()
    same(ref, h.solve_resident(params))
    same(ref, h.solve_resident(params))


def host_message(env, problems):
    capi, h = env["capi"], env["h"]
    with pytest.raises(capi.PsulvsbError) as e:
        h.upload(problems)
    assert e.value.code == capi.ERR_INVALID
    return str(e.value)


def test_refusals_match_the_host_path_and_leave_nothing_resident(env, mixed):
    capi, torch, h = env["capi"], env["torch"], env["h"]
    host, dev = mixed
    good_h, good_d = host[:3], dev[:3]
    params = capi.default_params(seed=3, **PKW)
    ref = h.solve_batch(params, good_h)

    def refused(bad_host, bad_dev, match):
        msg = host_message(env, bad_host)
        assert match in msg
        h.solve_batch_device(params, good_d)  # something resident, then the refusal drops it
        with pytest.raises(capi.PsulvsbError) as e:
            h.upload_device(bad_dev)
        assert e.value.code == capi.ERR_INVALID and str(e.value) == msg
        assert h.resident_size == 0
        same(ref, h.solve_batch_device(params, good_d))

    def copy_host(p):
        if is_aliased(p):
            return capi.HostProblem(p.src.copy(), p.dst.copy())
        return capi.HostProblem(p.src.copy(), p.dst.copy(), p.ori_src.copy(), p.ori_dst.copy(), p.keep_mask.copy(),
                                p.reduce_map.copy())

    # non-finite coordinates: src and dst of an aliased problem, ori_src of a pre-filtered one
    for field, b in (("src", 2), ("dst", 2), ("ori_src", 1)):
        bad = [copy_host(p) for p in good_h]
        getattr(bad[b], field)[1, 5] = np.nan
        refused(bad, [to_device(env, p) for p in bad], "problem %d has non-finite coordinates" % b)
    # a kept correspondence naming no column: -1 and C
    kept = int(np.flatnonzero(good_h[1].keep_mask == 1)[3])
    for v in (-1, good_h[1].src.shape[1]):
        bad = [copy_host(p) for p in good_h]
        bad[1].reduce_map[kept] = v
        refused(bad, [to_device(env, p) for p in bad], "problem 1 has keep_mask[j] == 1 with reduce_map[j] outside")
    # host memory through the C ABI is refused before anything is launched: pageable (numpy) and pinned
    h.solve_batch_device(params, good_d)
    pinned = torch.empty(good_d[0].src.shape, dtype=torch.float64, pin_memory=True)
    for name, addr in (("src", good_h[0].src.ctypes.data), ("dst", good_h[0].src.ctypes.data),
                       ("reduce_map", good_h[0].reduce_map.ctypes.data), ("src", pinned.data_ptr())):
        arr = (capi.Problem * 3)(*[p.c_struct() for p in good_d])
        cast = C.POINTER(C.c_int) if name == "reduce_map" else C.POINTER(C.c_double)
        setattr(arr[0], name, C.cast(C.c_void_p(addr), cast))
        launches = h.launch_count
        rc = capi.lib().psulvsb_batch_upload_device(h._h, None, arr, 3)
        assert rc == capi.ERR_INVALID
        assert ("problem 0: %s is not device memory" % name).encode() in capi.lib().psulvsb_last_error()
        assert h.launch_count == launches
        assert h.resident_size == 0
        same(ref, h.solve_batch_device(params, good_d))
    # the argument refusals of the host path
    arr = (capi.Problem * 1)(good_d[0].c_struct())
    arr[0].C = 1
    assert capi.lib().psulvsb_batch_upload_device(h._h, None, arr, 1) == capi.ERR_INVALID
    assert b"problem 0 has a null array, C < 2 or M < 1" in capi.lib().psulvsb_last_error()
    assert capi.lib().psulvsb_batch_upload_device(h._h, None, arr, 0) == capi.ERR_INVALID
    same(ref, h.solve_batch_device(params, good_d))


def host_centre_is_minus_zero(P, aligned):
    """Per coordinate r whose values are all +-0: whether the host path's centre is -0.0.  Its staging scan
    (engine.cu stage_points) keeps, per SSE lane, the LAST zero it meets (MINPD / MAXPD return the source operand on
    equal zeros); both extrema of coordinate r then come from lane r + 3, i.e. from flat index 6 j + r + 3 of the last
    whole group of six doubles.  Without a 16-byte aligned destination the scalar loop keeps the first point's value.
    The src side is staged aligned, the dst side at 3 C doubles after it (aligned iff C is even)."""
    flat = np.asfortranarray(P).ravel(order="F")
    out = []
    for r in range(3):
        if np.any(P[r] != 0):
            out.append(False)
            continue
        v = flat[(flat.size // 6 - 1) * 6 + r + 3] if aligned else flat[r]
        out.append(bool(np.signbit(v)))
    return out


def test_signed_zeros(env):
    """Every point has z = +0 or -0, both signs present on both sides: the device path's extrema order -0 before +0,
    so its centre of such a coordinate is +0.0, while the host's SIMD scan keeps whichever zero it meets last.  The
    cases where the host's centre is -0.0 do occur (problems 0, 2 and 4 by construction: an even C puts the last
    point's z in lane 5 on both sides, and it is -0), and the solutions do not depend on it."""
    capi, synth, h = env["capi"], env["synth"], env["h"]
    host = []
    for seed in range(6):
        rng = np.random.default_rng(700 + seed)
        n = [64, 257, 1000, 3001, 500, 2048][seed]
        src = np.zeros((3, n))
        src[:2] = rng.uniform(-1.5, 1.5, (2, n))
        a = rng.uniform(0, np.pi)
        R = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
        dst = R @ src + np.array([0.3, -0.2, 0.0])[:, None]
        dst[:2] += rng.uniform(-0.01, 0.01, (2, n))
        out = rng.permutation(n)[: int(0.8 * n)]
        dst[:2, out] = rng.uniform(-2, 2, (2, out.size))
        for P in (src, dst):
            P[2] = np.where(rng.uniform(0, 1, n) < 0.5, 0.0, -0.0)
            P[2, 0], P[2, -1] = (-0.0, 0.0) if seed % 2 else (0.0, -0.0)
            assert np.signbit(P[2]).any() and not np.signbit(P[2]).all()
        host.append(capi.HostProblem(np.asfortranarray(src), np.asfortranarray(dst)))
    host.append(prefiltered(env, 900, 31))
    for p in host[-1:]:
        for P in (p.src, p.dst, p.ori_src, p.ori_dst):
            P[1] = np.where(np.arange(P.shape[1]) % 3 == 0, -0.0, 0.0)
    flips = [(b, side) for b, p in enumerate(host) for side, P in (("src", p.src), ("dst", p.dst))
             if any(host_centre_is_minus_zero(P, side == "src" or P.shape[1] % 2 == 0))]
    assert {(0, "src"), (0, "dst"), (2, "src"), (2, "dst"), (4, "src"), (4, "dst")} <= set(flips), flips
    params = capi.default_params(seed=9, **PKW)
    ref = h.solve_batch(params, host)
    same(ref, h.solve_batch_device(params, [to_device(env, p) for p in host]))


def test_raw_scan_chain_on_device_buffers(env):
    """voxel_down_sample_batch_device -> fpfh_batch_device -> match_batch_device -> DeviceProblem.from_matches ->
    solve_batch_device, 16 pairs of the seeded surface, against match_batch -> HostProblem -> solve_batch on the same
    voxels; then icp_batch_device on the dense clouds."""
    capi, synth, features, icp, torch, h = (env[k] for k in ("capi", "synth", "features", "icp", "torch", "h"))
    B, n, v = 16, 50_000, 0.04
    srcs, tgts, truth = [], [], []
    for b in range(B):
        src = synth.make_surface(n, 60 + b)
        R, _ = synth.random_rigid(np.random.default_rng(80 + b))
        t = np.array([0.4, -0.3, 0.2])
        tgts.append(np.asfortranarray((R @ src + t[:, None])[:, np.random.default_rng(90 + b).permutation(n)]))
        srcs.append(src)
        truth.append((R, t))
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a.T)).cuda()  # noqa: E731
    d_srcs, d_tgts = [d(a) for a in srcs], [d(a) for a in tgts]
    vox, counts, offsets = features.voxel_down_sample_batch_device(d_srcs + d_tgts, v)
    counts = counts.cpu().numpy()  # the voxel counts size the next launches
    down = [vox[int(o):int(o) + int(c)] for o, c in zip(offsets, counts)]
    _, _, views = features.fpfh_batch_device(down, 2.0 * v, 5.0 * v)
    pairs, mcounts, moff = features.match_batch_device(down[:B], down[B:], [f for f, _ in views[:B]],
                                                       [f for f, _ in views[B:]], crosscheck=True)
    mcounts = mcounts.cpu().numpy()  # the one host read of the solve: the B match counts slice the pairs
    dev = [capi.DeviceProblem.from_matches(down[b], down[B + b], pairs[int(moff[b]):int(moff[b]) + int(mcounts[b])])
           for b in range(B)]
    kw = dict(noise_bound=1.5 * v, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005, wallclock_cap_s=0.0,
              seed=1)
    params = capi.default_params(**kw)
    sols = h.solve_batch_device(params, dev)
    # the host hop on the same voxels and matches
    hv = [a.cpu().numpy().T for a in down]
    matches = [pairs[int(moff[b]):int(moff[b]) + int(mcounts[b])].cpu().numpy() for b in range(B)]
    assert all(np.array_equal(m, mh) for m, mh in zip(matches, features.match_batch(
        hv[:B], hv[B:], [f.cpu().numpy() for f, _ in views[:B]], [f.cpu().numpy() for f, _ in views[B:]],
        crosscheck=True)))
    host = [capi.HostProblem(hv[b][:, m[:, 0]], hv[B + b][:, m[:, 1]]) for b, m in enumerate(matches)]
    same(h.solve_batch(params, host), sols)
    res = icp.icp_batch_device(d_srcs, d_tgts, np.array([s.R for s in sols]), np.array([s.t for s in sols]), v,
                               max_iterations=60)
    for s, o, (R, t) in zip(sols, res, truth):
        assert s.valid and synth.rotation_error(s.R, R) < 0.05 and np.linalg.norm(s.t - t) < 0.1
        assert synth.rotation_error(o.R, R) < 2e-3 and np.linalg.norm(o.t - t) < 5e-3
