"""GNC-TLS micro-benchmark in the shape of one engine tick of the bench workload: B registrations, one basic subset of
K line vectors each (cfg-A with FPFH-style outliers: K ~ 22 000), all solved by one launch.
    python profiles/tools/gnc_batch.py [B] [K] [line-vector scratch 0|1] [parking 0|1]
Prints, per cluster size, the launch time and thread 0's cycle split (line-vector passes / SVD / rest) per iteration."""
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
import psulvsb_b200  # noqa: E402,F401
from psulvsb_b200 import capi, stages, synth  # noqa: E402


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
    K = int(sys.argv[2]) if len(sys.argv) > 2 else 22000
    use_lv = (sys.argv[3] != "0") if len(sys.argv) > 3 else True
    use_perm = (sys.argv[4] != "0") if len(sys.argv) > 4 else True
    pair = synth.make_pair(5000, 0.95, 3, outliers="fpfh")
    r = stages.consistency_mask(pair["src"], pair["dst"], 0.1)  # the reduced set from the product's own stage 1
    e_all, _ = stages.compact_edges(r["mask"], r["row_counts"], r["n"], r["stride"])
    e_all = e_all.cpu().numpy()
    pi, pj = e_all[:, 0], e_all[:, 1]
    rng = np.random.default_rng(0)
    d_src, d_dst = stages.to_device_points(pair["src"]), stages.to_device_points(pair["dst"])
    edges = np.empty((B, K, 2), dtype=np.int32)
    for b in range(B):
        sel = rng.permutation(len(pi))[:K]
        edges[b, :, 0], edges[b, :, 1] = pi[sel], pj[sel]
    e = torch.from_numpy(edges).cuda()
    w = torch.zeros(B * K, dtype=torch.float64, device="cuda")
    lv_cap = K
    lv = torch.zeros(B * 6 * lv_cap, dtype=torch.float64, device="cuda") if use_lv else None
    perm = torch.zeros(B * 2 * lv_cap, dtype=torch.int32, device="cuda") if (use_lv and use_perm) else None
    R = torch.zeros(B * 9, dtype=torch.float64, device="cuda")
    info = torch.zeros(B * 4, dtype=torch.int32, device="cuda")
    prof = torch.zeros(B * 8, dtype=torch.int64, device="cuda")
    L = capi.lib()
    print(f"B={B} K={K} reduced set {len(pi)} lv scratch {'on' if use_lv else 'off'} parking {'on' if perm is not None else 'off'}")
    Rs = {}
    for cluster in (0, 1, 2, 4, 8):
        if cluster * B > 148 * 2 and cluster > 1:
            continue

        def run():
            capi.check(L.psulvsb_gnc_tls_rotation_batch(torch.cuda.current_stream().cuda_stream, d_src.data_ptr(),
                                                        d_dst.data_ptr(), 5000, e.data_ptr(), K, B, 0.1, 100, 1.4, 0.005,
                                                        cluster, w.data_ptr(), lv.data_ptr() if use_lv else None, lv_cap,
                                                        perm.data_ptr() if perm is not None else None, R.data_ptr(),
                                                        None, info.data_ptr(), prof.data_ptr()))
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(10):
            run()
        t1.record()
        torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / 10
        i = info.cpu().numpy().reshape(B, 4)
        p = prof.cpu().numpy().reshape(B, 8)
        its = i[:, 0].mean()
        Rs[cluster] = (R.cpu().numpy().copy(), i[:, :2].copy())
        print(f"cluster={cluster}: {ms * 1000:8.1f} us/launch  its {its:.1f}  per iteration: loop {p[:, 1].mean() / its:8.0f} "
              f"cycles = line-vector pass {p[:, 0].mean() / its:8.0f} + svd {p[:, 2].mean() / its:6.0f} + rest "
              f"{(p[:, 1] - p[:, 0] - p[:, 2]).mean() / its:6.0f};  cached {int(p[0, 3])} per CTA; whole kernel: prologue "
              f"{p[:, 4].mean():8.0f} + loop {p[:, 1].mean():8.0f} + epilogue {p[:, 5].mean():8.0f} cycles; parking: "
              f"{(p[:, 7] % 100).mean():.1f} compactions (first after iteration {((p[:, 7] // 100) % 100).mean() - 1:.1f}, "
              f"{(p[:, 7] // 10000).mean():.3f} repeated without sleeping), mean active positions per pass {p[:, 6].mean() / its:.0f}")
    # every configuration must end at the same rotations, iteration counts and inlier counts
    ref = Rs[1]
    for c, (r, ii) in Rs.items():
        print(f"cluster={c}: max |R - R(cluster=1)| = {np.abs(r - ref[0]).max():.2e}, iterations/inliers equal: "
              f"{np.array_equal(ii, ref[1])}")


if __name__ == "__main__":
    main()
