"""Small end-to-end + stage run for compute-sanitizer (memcheck): every kernel family once."""
import sys
import numpy as np
sys.path.insert(0, '.')
import psulvsb_b200
from psulvsb_b200 import capi, stages, synth, io
import torch

h = capi.Handle(0)
kw = dict(noise_bound=0.05, cbar2=1.0, estimate_scaling=0, rotation_cost_threshold=0.005, wallclock_cap_s=0.0)
# known scale with self-update
pair = synth.make_pair(700, 0.85, 3)
pre = synth.prefilter(pair, 3)
prob = capi.HostProblem(pre["src_reduce"], pre["dst_reduce"], pair["src"], pair["dst"], pre["keep_mask"], pre["reduce_map"])
sol, _ = h.solve(capi.default_params(seed=3, **kw), prob, trace_cap=64)
print("self-update solve", sol.status, sol.valid, sol.final_inlier_count, sol.final_C)
# batch of 3 of different sizes
probs = [capi.HostProblem(*(lambda p: (p["src"], p["dst"]))(synth.make_pair(n, 0.9, 10 + n)) ) for n in (130, 517, 300)]
sols = h.solve_batch(capi.default_params(**kw), probs, [1, 2, 3])
print("batch", [(s.status, s.final_inlier_count) for s in sols])
# unknown scale
p2 = synth.make_pair(300, 0.6, 9, outliers="gross")
kw2 = dict(kw); kw2["estimate_scaling"] = 1
sol, _ = h.solve(capi.default_params(seed=9, **kw2), capi.HostProblem(p2["src"], p2["dst"]))
print("unknown scale", sol.status, sol.valid, sol.scale)
# clique escalation
p3 = synth.make_pair(100, 0.9, 4, outliers="fpfh")
sol, _ = h.solve(capi.default_params(seed=4, **kw), capi.HostProblem(p3["src"], p3["dst"]))
print("clique", sol.status, sol.valid, sol.escalations)
# stages
r = stages.consistency_mask(pair["src"], pair["dst"], 0.1, symmetrize=True)
e, off = stages.compact_edges(r["mask"], r["row_counts"], r["n"], r["stride"])
print("k1", int(r["row_counts"].sum()), r["border"])
print("sample", stages.sample(5, 1, 0, 5000, 700)[1])
hyp = np.zeros((300, 12)); hyp[:, 0] = hyp[:, 4] = hyp[:, 8] = 1.0
c, b, bd = stages.score_batch(r["f_src"], r["f_dst"], r["d_src"], r["d_dst"], torch.from_numpy(hyp).cuda(), 1.0, 0.04, r["bound"], r["centres"])
torch.cuda.synchronize()
print("k4", int(c.max()))
print("normals", float(np.linalg.norm(io.estimate_normals(pair["src"][:, :300]), axis=0).mean()))
print("DONE")
