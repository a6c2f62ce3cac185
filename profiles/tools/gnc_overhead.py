import sys, numpy as np, torch
sys.path.insert(0, '.')
import psulvsb_b200
from psulvsb_b200 import capi, stages, synth
pair = synth.make_pair(5000, 0.95, 3)
r = stages.consistency_mask(pair['src'], pair['dst'], 0.1)  # the reduced set from the product's own stage 1
e_all, _ = stages.compact_edges(r['mask'], r['row_counts'], r['n'], r['stride'])
e_all = e_all.cpu().numpy()
pi, pj = e_all[:, 0], e_all[:, 1]
rng = np.random.default_rng(0)
d_src, d_dst = stages.to_device_points(pair['src']), stages.to_device_points(pair['dst'])
L = capi.lib()
for K in [512, 2048, 8192, 20000]:
    sel = rng.permutation(len(pi))[:K]
    e = torch.from_numpy(np.stack([pi[sel], pj[sel]], axis=1).astype(np.int32)).cuda()
    w = torch.zeros(K, dtype=torch.float64, device='cuda'); Rr = torch.zeros(9, dtype=torch.float64, device='cuda')
    info = torch.zeros(4, dtype=torch.int32, device='cuda'); c = torch.zeros(1, dtype=torch.float64, device='cuda')
    def run():
        capi.check(L.psulvsb_gnc_tls_rotation(torch.cuda.current_stream().cuda_stream, d_src.data_ptr(), d_dst.data_ptr(), e.data_ptr(), K, 1.0, 0.1, 100, 1.4, 0.005, None, w.data_ptr(), Rr.data_ptr(), None, info.data_ptr(), c.data_ptr()))
    for _ in range(5): run()
    torch.cuda.synchronize()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(20): run()
    t1.record(); torch.cuda.synchronize()
    ms = t0.elapsed_time(t1)/20
    i = info.cpu().numpy()
    its = int(i[0])
    print(f"K={K:6d} its={its:3d} call_ms={ms:.4f} us/iter={1000*ms/its:.2f}  svd_cycles/iter={16*i[2]/max(its-1,1):.0f} loop_cycles/iter={16*i[3]/its:.0f}")
