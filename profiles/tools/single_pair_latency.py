import sys, json, numpy as np, time
sys.path.insert(0, '.')
import psulvsb_b200
from psulvsb_b200 import capi, synth
kw = dict(noise_bound=0.05, cbar2=1.0, estimate_scaling=0, rotation_max_iterations=100, rotation_gnc_factor=1.4, rotation_cost_threshold=0.005, wallclock_cap_s=0.0)
pair = synth.make_pair(5000, 0.95, 1000001)
prob = capi.HostProblem(pair["src"], pair["dst"])
params = capi.default_params(seed=5, **kw)
h = capi.Handle(0)
base = None
for lv in (0, 2048, 1024, 512, 256):
    capi.debug_set("reset", 0)
    if lv: capi.debug_set("gnc_grid_lv", lv)
    ms = []
    for i in range(8):
        sol, _ = h.solve(params, prob)
        ms.append(h.last_device_ms)
    key = (sol.final_inlier_count, sol.local_iters, sol.n_reduced, tuple(np.round(sol.t, 12)))
    base = base or key
    print(json.dumps({"gnc_grid_lv": lv, "device_ms_median": float(np.median(ms[2:])), "gnc_ms": h.last_stage_ms(3) if hasattr(h, "last_stage_ms") else None, "same_result": key == base}))
