import sys, time, numpy as np
sys.path.insert(0, '.')
import psulvsb_b200
from psulvsb_b200 import capi, synth
import bench
B=int(sys.argv[1]) if len(sys.argv) > 1 else 64
pairs = bench.make_pairs(0, B)
probs = [capi.HostProblem(p["src"], p["dst"]) for p in pairs]
seeds = list(range(B))
params = capi.default_params(**bench.PARAM_KW)
h = capi.Handle(0)
for _ in range(3): h.solve_batch(params, probs, seeds)
def t(f, n=10):
    t0=time.perf_counter()
    for _ in range(n): f()
    return (time.perf_counter()-t0)/n*1000
print("upload ms", t(lambda: h.upload(probs)))
print("solve_resident ms", t(lambda: h.solve_resident(params, seeds)), "device ms", h.last_device_ms)
print("solve_batch ms", t(lambda: h.solve_batch(params, probs, seeds)))
arr = capi.Handle._problem_array(probs)
print("problem array build ms", t(lambda: capi.Handle._problem_array(probs)))
