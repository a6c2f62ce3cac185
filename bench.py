#!/usr/bin/env python
"""bench.py -- the PSULVSB hot path on B200 (BASELINE.json metric: registrations/s at N = 5000, 95 % outliers).

    python bench.py --gpus N --steps K --warmup W [--config cfgA|cfgB|cfgC|cfgD|bunny] [--impl reference]
                    [--dump-outputs DIR]

Workloads (BASELINE.json configs; SURVEY.md section 8d).  One STEP = one pass of the hot path
(RobustRegistrationSolver::solve, registration.cc:622-1535) over one batch of synthetic input, fixed seeds.

  cfgA (default, configs[1]) : B independent fragment pairs per GPU per step, each N = 5000 FPFH-style correspondences
          with 95 % outliers.  Pairs shard across GPUs with no data-path collective (weak scaling).  The default line
          also carries: `parity` (the GPU solutions of the CPU sample against the oracle's -- a mismatch exits non-zero),
          `stages` (the consistency kernel at N = 100 000 and the scoring sweep 2^20 x 50 000, sharded over the same
          N GPUs through the library's own NCCL communicator), `variants` (pre-filter + self-update inputs, gross
          outliers) and `latency_ms_single` (one pair alone).
  cfgC (configs[3]) : 4096 independent cfg-A pairs, strong-scaled: 4096 / N pairs per GPU.
  cfgB (configs[2]) : ONE registration with N = 100 000 correspondences, 99 % outliers; the consistency rows are
          sharded across the N GPUs (psulvsb_solve_sharded: edge lists all-gathered over NCCL).
  cfgD (configs[4]) : hypothesis-scoring sweep, 2^20 hypotheses x N = 50 000 correspondences, hypotheses sharded across
          GPUs, global best through ONE 8-byte ncclAllReduce(max) inside psulvsb_score_batch_sharded.
  bunny (configs[0]) : the reference driver's own case (examples/teaser_cpp_ply/PSULVSB.cc): Stanford bunny vertices,
          random rigid transform, +-0.05 noise, 90 % gross outliers; the timed region is the reference's
          (PSULVSB.cc:309-329): normal-angle histogram pre-filter + mask_filter + solve.

  value : the metric with inputs resident in HBM, device time from CUDA events, max over ranks.
  e2e   : the same through the C ABI with HOST buffers: staging + H2D + solve + D2H inside the timed region.
  roofline     : the consistency-mask kernel (stage 1), FP32-pipe bound (SURVEY.md 8d): 16 issue slots per unordered
                 pair; peak = SMs x 128 lanes x SM clock under load; timed live by CUDA events around its launches.
  cpu_baseline : the CPU oracle (a port of the reference's algorithm; the reference itself cannot be built in this
                 image) on a bounded sample of the same problems, 1 core.
  --impl reference : the oracle on all host cores (process pool), same metric / config.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_CORR = 5000
OUTLIER_RATIO = 0.95
CFGC_PAIRS = 4096
PARAM_KW = dict(noise_bound=0.05, cbar2=1.0, estimate_scaling=0, rotation_max_iterations=100,
                rotation_gnc_factor=1.4, rotation_cost_threshold=0.005, wallclock_cap_s=0.0)
K1_SLOTS_PER_PAIR = 16  # SURVEY.md section 8(d)
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch from an `ncu --set full` capture (it cannot be measured
# in-process); refreshed every round by profiles/tools/traffic_from_ncu.py -> profiles/ncu_traffic.json.  Stored per
# registration of a cfg-A batch, so other batch sizes scale.
NCU_TRAFFIC = {
    "k1_mask_kernel": {"bytes_per_registration": (472_137_000 + 899_623_000) / 296,
                       "source": "ncu capture profiles/r1_ncu_step_b296_final.txt (B = 296)"},
    "gnc_tls_kernel": {"bytes_per_registration": (2_886_296_000 + 692_751_000) / 296,
                       "source": "ncu capture profiles/r1_ncu_step_b296_final.txt (B = 296)"},
}
try:
    with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as _f:
        NCU_TRAFFIC.update(json.load(_f))
except Exception:
    pass
# What the FP32 pipe sustains on this part, measured by profiles/tools/fp32_pipe_probe.cu (committed output:
# profiles/r2_fp32_pipe_probe.jsonl): the nominal 128 lanes x clock of the roofline is reached by neither FFMA nor FFMA2
# streams, and every ALU-pipe instruction beside them costs 1.6-2.3 issue cycles.  Reported next to the roofline, not
# used as its peak.
PIPE_PROBE = None
try:
    _rows = [json.loads(l) for l in open(os.path.join(ROOT, "profiles", "r2_fp32_pipe_probe.jsonl")) if l.startswith("{")]

    def _best(sub, key):
        v = [r[key] for r in _rows if sub in r.get("case", "") and key in r]
        return max(v) if v else None
    PIPE_PROBE = {"ffma_stream_frac_of_128_lanes": _best("scalar FFMA", "frac_of_128"),
                  "ffma2_stream_64bit_operand_shared": _best("matrix operand shared (6 x 4)", "frac_of_128"),
                  "ffma2_stream_32bit_operand_shared": _best("scalar operand shared (6 x 4)", "frac_of_128"),
                  "k1_word_loop_alone_frac_of_16_slot_roofline": _best("(the kernel's loop)", "frac_of_16_slot_roofline"),
                  "source": "profiles/r2_fp32_pipe_probe.jsonl (profiles/tools/fp32_pipe_probe.cu on one B200)"}
except Exception:
    pass


# ----------------------------------------------------------------------------------------------------------------
# workloads
# ----------------------------------------------------------------------------------------------------------------
def make_pairs(rank: int, batch: int, first: int = 0, outliers: str = "fpfh"):
    import psulvsb_b200  # noqa: F401
    from psulvsb_b200 import synth

    return [synth.make_pair(N_CORR, OUTLIER_RATIO, 1_000_000 + rank * 100_000 + first + i, outliers=outliers)
            for i in range(batch)]


def pair_seed(rank: int, i: int) -> int:
    return 1000 + rank * 100_000 + i


def host_problem(capi, synth, pair, mode: int, seed: int):
    """mode 1: keep_mask all ones (C = M, self-update idle); mode 2: emulated pre-filter (exercises self-update)."""
    if mode == 1:
        return capi.HostProblem(pair["src"], pair["dst"]), None
    f = synth.prefilter(pair, seed)
    return capi.HostProblem(f["src_reduce"], f["dst_reduce"], pair["src"], pair["dst"], f["keep_mask"], f["reduce_map"]), f


def bunny_case(seed: int):
    """configs[0]: PSULVSB.cc:256-286 on the bunny vertices the reference ships (bun_zipper_res3, 1889 points)."""
    import psulvsb_b200  # noqa: F401
    from psulvsb_b200 import synth

    z = np.load(os.path.join(ROOT, "tests", "golden", "bunny_res3.npz"))
    pts = np.asarray(z[z.files[0]], dtype=np.float64)
    if pts.shape[0] != 3:
        pts = pts.T
    return synth.make_pair(pts.shape[1], 0.90, seed, sigma=0.05, outliers="gross", src_points=pts)


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons while the timed region runs (NVML every 5 ms; nvidia-smi, which
    needs ~100 ms per query, only as a fallback)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.sm, self.mx, self.reasons = [], [], set()
        self._stop_evt = threading.Event()
        self._nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
        self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(self._h, n.NVML_CLOCK_SM)))
        r = n.nvmlDeviceGetCurrentClocksEventReasons(self._h) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
            else n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for name, bit in (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40),
                          ("sw_power_cap", 0x4)):
            if r & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        f = [x.strip() for x in out.strip().split(",")]
        if len(f) >= 6:
            self.sm.append(float(f[0]))
            self.mx.append(float(f[1]))
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[2:6]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def run(self):
        while not self._stop_evt.is_set():
            try:
                if self._nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop_evt.wait(0.005 if self._nvml is not None else 0.05)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None,
                "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "source": "nvml" if self._nvml is not None else "nvidia-smi"}


# ----------------------------------------------------------------------------------------------------------------
# the CPU oracle: the checker and the CPU baseline (never on the product path)
# ----------------------------------------------------------------------------------------------------------------
def _oracle_solve_one(job):
    """job = (src, dst, seed[, dict(ori_src, ori_dst, keep_mask, reduce_map)]) -> result summary."""
    from oracle import oracle as O

    src, dst, seed = job[0], job[1], job[2]
    extra = job[3] if len(job) > 3 and job[3] is not None else {}
    p = O.default_params(seed=seed, **PARAM_KW)
    sol, tr = O.solve(p, src, dst, trace_cap=1, **extra)
    return {"valid": sol.valid, "final_inlier_count": sol.final_inlier_count, "n_reduced": sol.n_reduced,
            "local_iters": sol.local_iters, "host_rounds": sol.host_rounds, "final_C": sol.final_C,
            "R": O.solution_R(sol), "t": O.solution_t(sol), "scale": sol.scale,
            "final_inliers": np.packbits(tr["final_inliers"] != 0)}


def cpu_run(jobs, workers: int):
    """(wall seconds, results) of the oracle over `jobs` with `workers` processes (1 = in-process, scalar port)."""
    from oracle import oracle as O

    O.lib()
    if workers <= 1:
        t0 = time.perf_counter()
        res = [_oracle_solve_one(j) for j in jobs]
        return time.perf_counter() - t0, res
    import multiprocessing as mp

    with mp.get_context("fork").Pool(workers) as pool:
        pool.map(_oracle_solve_one, jobs[:workers])  # warm the workers
        t0 = time.perf_counter()
        res = pool.map(_oracle_solve_one, jobs, chunksize=1)
        return time.perf_counter() - t0, res


def compare_with_oracle(sols, refs, final_inlier_sets=None):
    """GPU solutions vs the oracle's on the same problems and sample streams (north_star: inlier sets bit-exact,
    R within 1e-5 rad, t within 1e-5 units).  Returns the `parity` object of the JSON line."""
    import psulvsb_b200  # noqa: F401
    from psulvsb_b200 import synth

    mism, worst_R, worst_t = [], 0.0, 0.0
    for i, (s, r) in enumerate(zip(sols, refs)):
        bad = []
        if s.status != 0:
            bad.append(f"status {s.status}")
        for f in ("valid", "final_inlier_count", "n_reduced", "local_iters", "host_rounds", "final_C"):
            if int(getattr(s, f)) != int(r[f]):
                bad.append(f"{f} {getattr(s, f)} != {r[f]}")
        if r["valid"]:
            eR = synth.rotation_error(s.R, r["R"])
            et = float(np.abs(s.t - r["t"]).max())
            worst_R, worst_t = max(worst_R, eR), max(worst_t, et)
            if not (eR < 1e-5):
                bad.append(f"R off by {eR:.3g} rad")
            if not (et < 1e-5):
                bad.append(f"t off by {et:.3g}")
        if final_inlier_sets is not None and i < len(final_inlier_sets) and final_inlier_sets[i] is not None:
            if not np.array_equal(np.packbits(np.asarray(final_inlier_sets[i]) != 0), r["final_inliers"]):
                bad.append("final_inliers set differs")
        if bad:
            mism.append({"problem": i, "what": bad})
    out = {"checked": len(refs), "mismatch": len(mism), "max_R_err_rad": worst_R, "max_t_err": worst_t,
           "final_inlier_sets_compared": 0 if final_inlier_sets is None else sum(x is not None for x in final_inlier_sets),
           "fields": "valid, final_inlier_count, n_reduced, local_iters, host_rounds, final_C exact; R < 1e-5 rad; "
                     "t < 1e-5; final_inliers[M] bit-exact where compared"}
    if mism:
        out["first_mismatches"] = mism[:4]
    return out


DUMP_LIMIT_BYTES = 64 << 20


def solution_arrays(sols):
    """What a caller of the solve entry points receives, one row per registration, as float64 arrays."""
    out = {"rotation": np.stack([s.R for s in sols]), "translation": np.stack([s.t for s in sols])}
    for f in ("valid", "scale", "final_inlier_count", "host_rounds", "local_iters", "n_line_vectors", "n_reduced",
              "final_C", "refined", "escalations", "borderline_pairs", "status"):
        out[f] = np.array([getattr(s, f) for s in sols], dtype=np.float64)
    return out


def dump_outputs(directory: str, arrays: dict, rank: int):
    """Writes arrays as DIR/<name>.npy (float64; DIR/<name>.rank<r>.npy for ranks > 0).  Should they exceed 64 MB in
    all, a fixed, seeded sample of their rows is written instead, with the row indices as DIR/sampled_rows.npy."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        n = max(a.shape[0] for a in arrays.values())
        rows = np.sort(np.random.default_rng(0).choice(n, int(n * DUMP_LIMIT_BYTES / total), replace=False))
        arrays = {k: (a[rows] if a.shape[0] == n else a) for k, a in arrays.items()}
        arrays["sampled_rows"] = rows.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(directory, k + (f".rank{rank}" if rank else "") + ".npy"), a)


def cpu_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ----------------------------------------------------------------------------------------------------------------
# reference arm: the oracle on all host cores
# ----------------------------------------------------------------------------------------------------------------
def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    cores = cpu_cores()
    cfg = args.config
    if cfg not in ("cfgA", "cfgC"):
        print(json.dumps({"impl": "reference", "unavailable":
                          f"{cfg}: no all-cores CPU arm (cfgB / cfgD are beyond what the reference can represent -- int "
                          f"pair indices, registration.cc:682-686 -- and the bunny driver needs PCL normals); the CPU "
                          f"sample of this config is the cpu_baseline object of `bench.py --config {cfg}`"}))
        return
    per_step = max(cores * 2, 8)
    pairs = make_pairs(0, per_step)
    jobs = [(p["src"], p["dst"], pair_seed(0, i)) for i, p in enumerate(pairs)]
    for _ in range(args.warmup):
        cpu_run(jobs[:cores], cores)
    t = 0.0
    for _ in range(args.steps):
        t += cpu_run(jobs, cores)[0]
    value = per_step * args.steps / t
    line = {
        "impl": "reference", "metric": "registrations/s", "value": value, "unit": "registrations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * t / args.steps,
        "higher_is_better": True, "scaling": "weak" if cfg == "cfgA" else "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": f"{cfg}: N={N_CORR} correspondences, {int(OUTLIER_RATIO * 100)}% FPFH-style outliers, "
                               f"independent fragment pairs", "pairs_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": "registrations/s", "cores": cores, "kind": "port",
                         "sample": f"{per_step} cfg-A pairs per step on {cores} host processes (CPU oracle: a port; the "
                                   f"reference needs Eigen3/Boost/PCL/PMC and cannot be built in this image)"},
        "e2e": {"value": value, "unit": "registrations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# GPU arms
# ----------------------------------------------------------------------------------------------------------------
class Ctx:
    pass


def setup(args):
    import torch
    import torch.distributed as dist

    import psulvsb_b200  # noqa: F401
    from psulvsb_b200 import capi, synth

    c = Ctx()
    c.torch, c.dist, c.capi, c.synth = torch, dist, capi, synth
    c.rank = int(os.environ.get("RANK", "0"))
    c.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available() or capi.lib().psulvsb_device_count() < 1:
        raise SystemExit("bench.py: no CUDA device (the product has no CPU fallback)")
    torch.cuda.set_device(c.local_rank)
    if c.world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", c.local_rank))
    c.h = capi.Handle(c.local_rank)
    c.h.set_batching(args.chunk, args.lanes)
    if c.world > 1:  # every rank of the node gets its share of the host cores for staging
        c.h.set_host_threads(max(1, cpu_cores() // c.world))
    for kv in filter(None, args.debug.split(",")):
        capi.debug_set(kv.split("=")[0], float(kv.split("=")[1]))
    if c.world > 1:
        # the library's own communicator (NCCL): rank 0 makes the id, torch.distributed only carries its 128 bytes
        uid = torch.zeros(capi.UNIQUE_ID_BYTES, dtype=torch.uint8)
        if c.rank == 0:
            uid = torch.from_numpy(np.frombuffer(capi.comm_unique_id(), dtype=np.uint8).copy())
        uid = uid.cuda()
        dist.broadcast(uid, 0)
        c.h.comm_create(c.rank, c.world, uid.cpu().numpy().tobytes())
    c.peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            c.peaks = json.load(f)
    except Exception:
        pass
    c.sms = torch.cuda.get_device_properties(c.local_rank).multi_processor_count
    return c


def barrier(c):
    if c.world > 1:
        c.dist.barrier()
    c.torch.cuda.synchronize()


def max_over_ranks(c, *vals):
    t = c.torch.tensor(list(vals), dtype=c.torch.float64, device="cuda")
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()]


def gather_ints(c, vals):
    """Every rank's list (same length) -> list of lists on every rank."""
    t = c.torch.tensor(list(vals), dtype=c.torch.int64, device="cuda")
    if c.world == 1:
        return [t.tolist()]
    parts = [c.torch.zeros_like(t) for _ in range(c.world)]
    c.dist.all_gather(parts, t)
    return [p.tolist() for p in parts]


def timed_resident(c, params, probs, seeds, steps, warmup):
    """`steps` resident solves; per-rank sums (device ms, k1 ms, gnc ms), ticks, launches and the last solutions."""
    h = c.h
    h.upload(probs)
    for _ in range(warmup):
        sols = h.solve_resident(params, seeds)
    bad = [s.status for s in sols if s.status != 0]
    if bad:
        raise SystemExit(f"bench.py: solve failed with status {bad[:4]}")
    barrier(c)
    l0 = h.launch_count
    dev_ms = k1_ms = gnc_ms = 0.0
    ticks = []
    t0 = time.perf_counter()
    for _ in range(steps):
        sols = h.solve_resident(params, seeds)
        dev_ms += h.last_device_ms
        k1_ms += h.last_stage_ms(2)
        gnc_ms += h.last_stage_ms(3)
        ticks.append(h.last_ticks)
    barrier(c)
    wall_ms = (time.perf_counter() - t0) * 1000.0
    return {"dev_ms": dev_ms, "k1_ms": k1_ms, "gnc_ms": gnc_ms, "ticks": ticks, "wall_ms": wall_ms,
            "launches": h.launch_count - l0, "sols": sols, "chunk_ticks": h.last_chunk_ticks}


def timed_e2e(c, params, probs, seeds, steps, warmup=2, depth=3):
    """`steps` batches with HOST buffers through the C ABI; every step's staging + H2D copy and its D2H of the solutions
    lie inside the timed region.  depth 1: psulvsb_solve_batch, one call after the other (each drains the device);
    depth 3: psulvsb_batch_submit / psulvsb_batch_wait with three batches in flight -- a stream of batches: two are being
    solved (the handle's two lanes) while the third is staged and copied, so the uploads run under the solves."""
    h = c.h
    for _ in range(warmup):
        h.solve_batch(params, probs, seeds)
    if depth > 1:  # (every lane's engine has its arenas before the clock starts)
        for t in [h.submit(params, probs, seeds) for _ in range(depth + 1)]:
            h.wait(t)
    barrier(c)
    t0 = time.perf_counter()
    if depth <= 1:
        for _ in range(steps):
            sols = h.solve_batch(params, probs, seeds)
    else:
        tickets = []
        for _ in range(steps):
            tickets.append(h.submit(params, probs, seeds))
            if len(tickets) >= depth:
                sols = h.wait(tickets.pop(0))
        while tickets:
            sols = h.wait(tickets.pop(0))
    barrier(c)
    return (time.perf_counter() - t0) * 1000.0, sols


def final_inlier_sets(c, params, probs, seeds, n):
    """final_inliers[M] of the first n problems (single solves with a trace: the batch calls return solutions only)."""
    out = []
    keep = params.seed
    for i in range(n):
        params.seed = seeds[i]
        _, tr = c.h.solve(params, probs[i], trace_cap=8)
        out.append(tr["final_inliers"].copy())
    params.seed = keep
    return out


def k1_roofline(c, clocks, B, k1_ms_per_step, dev_ms_per_step):
    f_mhz = clocks["sm_mhz"] or c.peaks.get("clocks_under_load", {}).get("sm_mhz_median") or 1965.0
    pairs = B * (N_CORR * (N_CORR - 1) // 2)
    k1_s = k1_ms_per_step / 1000.0
    achieved = pairs * K1_SLOTS_PER_PAIR / k1_s / 1e9 if k1_s > 0 else None
    peak = c.sms * 128 * f_mhz * 1e6 / 1e9
    stride = ((N_CORR + 31) // 32 + 7) // 8 * 8
    mask_bytes = B * N_CORR * stride * 4
    hbm_peak = c.peaks.get("hbm_gbs", 6650.0)
    tr = NCU_TRAFFIC["k1_mask_kernel"]
    return {"bound": "fp32-pipe", "kernel": "k1_mask_kernel (line-vector length-consistency bit mask)",
            "achieved": achieved, "peak": peak, "unit": "Gslot/s (FP32-pipe issue slots, 16 per pair)",
            "frac": (achieved / peak) if achieved else None,
            "traffic": int(tr["bytes_per_registration"] * B), "traffic_source": tr["source"],
            "algorithmic_bytes": mask_bytes // 2 + 2 * B * N_CORR * 16,
            "pairs_per_s": pairs / k1_s if k1_s > 0 else None,
            "kernel_ms": k1_ms_per_step,
            "share_of_step": k1_ms_per_step / dev_ms_per_step if dev_ms_per_step > 0 else None,
            "peak_source": f"{c.sms} SMs x 128 lanes x {f_mhz:.0f} MHz (SM clock sampled during the run)",
            "pipe_probe": PIPE_PROBE,
            "hbm_mask_write": {"achieved": mask_bytes / k1_s / 1e9 if k1_s > 0 else None, "peak": hbm_peak,
                               "unit": "GB/s", "frac": (mask_bytes / k1_s / 1e9 / hbm_peak) if k1_s > 0 else None,
                               "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if "hbm_gbs" in c.peaks
                               else "fallback 6650 GB/s"}}


def gnc_report(c, B, sols, gnc_ms_per_step, dev_ms_per_step, ticks_per_step):
    # mean basic-subset size of the step (line vectors handed to one GNC-TLS solve): the algorithmic input of that kernel
    k_mean = float(np.mean([s.n_reduced for s in sols])) * 0.1 * 0.3
    hbm_peak = c.peaks.get("hbm_gbs", 6650.0)
    per_launch_ms = gnc_ms_per_step / ticks_per_step if ticks_per_step else None
    alg = B * k_mean * 48
    tr = NCU_TRAFFIC["gnc_tls_kernel"]
    return {"kernel": "gnc_tls_kernel (GNC-TLS rotation, FP64; one launch per tick and chunk)",
            "share_of_step": gnc_ms_per_step / dev_ms_per_step if dev_ms_per_step > 0 else None,
            "ms_per_launch": per_launch_ms, "bound": "hbm", "algorithmic_bytes": int(alg),
            "achieved": alg / (per_launch_ms / 1e3) / 1e9 if per_launch_ms else None, "peak": hbm_peak, "unit": "GB/s",
            "frac": (alg / (per_launch_ms / 1e3) / 1e9 / hbm_peak) if per_launch_ms else None,
            "traffic": int(tr["bytes_per_registration"] * B), "traffic_source": tr["source"],
            "note": "algorithmic bytes = every line vector of a solve read once (48 B); the kernel re-reads the part of a "
                    "registration's line vectors that does not fit in shared memory every GNC iteration until parked"}


def run_variant(c, params, name, mode, outliers, B, steps, n_check):
    """A short resident measurement of a cfg-A-sized variant workload + parity of its first problems."""
    capi, synth = c.capi, c.synth
    pairs = make_pairs(c.rank, B, first=50_000 if outliers == "gross" else 0, outliers=outliers)
    seeds = [pair_seed(c.rank, i) for i in range(B)]
    built = [host_problem(capi, synth, p, mode, s) for p, s in zip(pairs, seeds)]
    probs = [b[0] for b in built]
    r = timed_resident(c, params, probs, seeds, steps, 2)
    (dev_max,) = max_over_ranks(c, r["dev_ms"])
    out = None
    if c.rank == 0:
        sols = r["sols"]
        out = {"workload": name, "value": B * steps * c.world / (dev_max / 1e3), "unit": "registrations/s",
               "pairs_per_gpu_per_step": B, "ms_per_step": dev_max / steps, "ticks_per_step": float(np.mean(r["ticks"])),
               "mean_final_inliers": float(np.mean([s.final_inlier_count for s in sols])),
               "mean_final_C": float(np.mean([s.final_C for s in sols])),
               "mean_host_rounds": float(np.mean([s.host_rounds for s in sols]))}
        if n_check > 0:
            jobs = []
            for i in range(n_check):
                f = built[i][1]
                extra = None if f is None else dict(ori_src=pairs[i]["src"], ori_dst=pairs[i]["dst"],
                                                    keep_mask=f["keep_mask"], reduce_map=f["reduce_map"])
                jobs.append((probs[i].src, probs[i].dst, seeds[i], extra))
            tcpu, refs = cpu_run(jobs, 1)
            sets = final_inlier_sets(c, params, probs, seeds, min(n_check, 4))
            out["parity"] = compare_with_oracle(sols[:n_check], refs, sets)
            out["cpu_baseline"] = {"value": n_check / tcpu, "unit": "registrations/s", "cores": 1, "kind": "port",
                                   "sample": f"first {n_check} problems"}
    barrier(c)
    return out


def shard(n, rank, world):
    base, rem = divmod(n, world)
    b = rank * base + min(rank, rem)
    return b, b + base + (1 if rank < rem else 0)


def run_cfgA(args, c, strong_total: int = 0):
    capi = c.capi
    world, rank = c.world, c.rank
    if strong_total:
        b0, b1 = shard(strong_total, rank, world)
        B, first = b1 - b0, b0
        pairs = make_pairs(0, B, first=first)  # one global problem list, sliced
        seeds = [pair_seed(0, first + i) for i in range(B)]
    else:
        B = args.batch
        pairs = make_pairs(rank, B)
        seeds = [pair_seed(rank, i) for i in range(B)]
    probs = [capi.HostProblem(p["src"], p["dst"]) for p in pairs]
    params = capi.default_params(**PARAM_KW)
    W = max(args.warmup, 3)

    sampler = ClockSampler(c.local_rank)
    sampler.start()
    r = timed_resident(c, params, probs, seeds, args.steps, W)
    clocks = sampler.stop()
    e2e_ms, _ = timed_e2e(c, params, probs, seeds, args.steps, depth=3)
    e2e_sync_ms, _ = timed_e2e(c, params, probs, seeds, args.steps, depth=1)
    dev_max, e2e_max, wall_max, e2e_sync_max = max_over_ranks(c, r["dev_ms"], e2e_ms, r["wall_ms"], e2e_sync_ms)
    total_regs = (strong_total if strong_total else B * world) * args.steps
    rank_ticks = gather_ints(c, [max(r["ticks"]), min(r["ticks"])])
    tot = gather_ints(c, [sum(p.nbytes for p in probs), B * ctypes.sizeof(capi.Solution)])

    # single-pair latency (configs[1] is ONE pair on one B200): host buffers in, solution out
    lat = []
    one_params = capi.default_params(**PARAM_KW)
    one_params.seed = seeds[0]
    for _ in range(8):
        t0 = time.perf_counter()
        c.h.solve(one_params, probs[0])
        lat.append(((time.perf_counter() - t0) * 1e3, c.h.last_device_ms))
    lat = lat[3:]

    line = None
    if rank == 0:
        sols = r["sols"]
        name = "cfgC" if strong_total else "cfgA"
        line = {
            "metric": "registrations/s", "value": total_regs / (dev_max / 1000.0), "unit": "registrations/s",
            "n_gpus": world, "steps": args.steps, "warmup": W, "ms_per_step": dev_max / args.steps,
            "higher_is_better": True, "scaling": "strong" if strong_total else "weak", "vs_baseline": None,
            "dtype": "f64+f32", "data": "synthetic",
            "config": {"workload": f"{name}: N={N_CORR} correspondences, {int(OUTLIER_RATIO * 100)}% FPFH-style "
                                   f"outliers, independent fragment pairs"
                                   + (f", {strong_total} pairs in total split over the GPUs" if strong_total else ""),
                       "pairs_per_gpu_per_step": B,
                       "l2": "no flush: per-step working set (edge arena + masks) exceeds the 126 MB L2",
                       "params": "noise_bound 0.05, cbar2 1, known scale, GNC-TLS 1.4/100/0.005, replay mode, "
                                 "keep_mask all ones (mode 1)",
                       "ticks_per_step": float(np.mean(r["ticks"])), "ticks_per_rank_max_min": rank_ticks,
                       "chunk_ticks_last_step": r["chunk_ticks"],
                       "mean_inliers": float(np.mean([s.final_inlier_count for s in sols])),
                       "wall_ms_per_step": wall_max / args.steps},
            "e2e": {"value": total_regs / (e2e_max / 1000.0), "unit": "registrations/s",
                    "h2d_bytes_per_step": int(sum(t[0] for t in tot)), "d2h_bytes_per_step": int(sum(t[1] for t in tot)),
                    "how": "psulvsb_batch_submit / psulvsb_batch_wait, host buffers, three batches in flight (a stream of "
                           "batches: two being solved on the handle's two lanes while the next is staged and copied; "
                           "every step's H2D and D2H copies are inside the timed region)",
                    "one_call_at_a_time": total_regs / (e2e_sync_max / 1000.0)},
            "gpu_launches": int(r["launches"]),
            "clocks": clocks,
            "latency_ms_single": {"wall_ms": float(np.median([x[0] for x in lat])),
                                  "device_ms": float(np.median([x[1] for x in lat])),
                                  "what": "psulvsb_solve of ONE cfg-A pair, host buffers in, solution out (median of 5)"},
        }
        line["roofline"] = k1_roofline(c, clocks, B, r["k1_ms"] / args.steps, r["dev_ms"] / args.steps)
        line["roofline"]["largest_kernel"] = gnc_report(c, B, sols, r["gnc_ms"] / args.steps, r["dev_ms"] / args.steps,
                                                        float(np.mean(r["ticks"])))
        if not args.no_cpu_baseline:
            n_cpu = min(B, 64)
            reps = max(1, int(round(120 / n_cpu)))  # ~120 registrations ~ 11 s of single-core work
            jobs = [(p["src"], p["dst"], s) for p, s in zip(pairs[:n_cpu], seeds[:n_cpu])]
            tcpu, refs = 0.0, None
            for _ in range(reps):
                t, res = cpu_run(jobs, 1)
                tcpu += t
                refs = refs or res
            line["cpu_baseline"] = {"value": reps * n_cpu / tcpu, "unit": "registrations/s", "cores": 1, "kind": "port",
                                    "sample": f"first {n_cpu} pairs of rank 0's batch x {reps}, CPU oracle (scalar port "
                                              f"of registration.cc:622-1535; the reference cannot be built here), "
                                              f"{tcpu:.1f} s"}
            # result agreement on the sample (the oracle as the checker, never as the thing measured)
            sets = final_inlier_sets(c, params, probs, seeds, min(n_cpu, 8))
            line["parity"] = compare_with_oracle(sols[:n_cpu], refs, sets)
    barrier(c)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, solution_arrays(r["sols"]), rank)
    return line, params


def sm_clock_now(c):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(c.local_rank), "--query-gpu=clocks.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        return float(out.strip().split(",")[0])
    except Exception:
        return None


def timed_stream(c, fn, steps, warmup):
    """CUDA events on torch's current stream (the stage entry points are launched on it); mean ms, max over ranks."""
    torch = c.torch
    for _ in range(max(warmup, 3)):
        fn()
    barrier(c)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
    return max_over_ranks(c, float(np.mean(ms)))[0]


def stage_k1(c, n=100_000, steps=3, warmup=2):
    """The consistency kernel at cfg-B's size, inside the library's own sharded registration (psulvsb_solve_sharded:
    rows split over the ranks with triangular balancing, edge counts and edge lists exchanged over NCCL).  Timed by the
    engine's CUDA events around the kernel launch alone (psulvsb_last_stage_ms(2)); max over ranks."""
    capi = c.capi
    pair = c.synth.make_pair(n, 0.99, 4242, side=30.0)
    prob = capi.HostProblem(pair["src"], pair["dst"])
    params = capi.default_params(seed=11, **PARAM_KW)
    solve = (lambda: c.h.solve_sharded(params, prob)) if c.world > 1 else (lambda: c.h.solve(params, prob)[0])
    for _ in range(warmup):
        sol = solve()
    barrier(c)
    k1 = dev = 0.0
    for _ in range(steps):
        sol = solve()
        k1 += c.h.last_stage_ms(2)
        dev += c.h.last_device_ms
    barrier(c)
    f = sm_clock_now(c) or 1965.0
    k1_max, dev_max = max_over_ranks(c, k1 / steps, dev / steps)
    pairs_total = n * (n - 1) // 2
    peak = c.world * c.sms * 128 * f * 1e6 / 1e9
    ach = pairs_total * 16 / (k1_max / 1e3) / 1e9
    return {"case": "consistency kernel of ONE registration, N = 100000 correspondences, 99% outliers (cfg-B)", "n": n,
            "n_gpus": c.world, "pairs": pairs_total, "n_reduced": int(sol.n_reduced), "ms": k1_max,
            "pairs_per_s": pairs_total / (k1_max / 1e3), "registration_ms": dev_max,
            "final_inliers": int(sol.final_inlier_count),
            "roofline": {"bound": "fp32-pipe", "achieved": ach, "peak": peak, "frac": ach / peak,
                         "unit": "Gslot/s (16 FP32-pipe issue slots per unordered pair)",
                         "peak_source": f"{c.world} x {c.sms} SMs x 128 lanes x {f:.0f} MHz (nvidia-smi after the run)"},
            "sharding": "triangular row blocks inside psulvsb_solve_sharded; edge counts all-gathered, edge lists "
                        "all-gathered in place (grouped ncclBroadcast), RANSAC replicated"}


def stage_k4(c, n=50_000, H=1 << 20, steps=5, warmup=3, with_e2e=False):
    """cfg-D: hypotheses sharded over the ranks; psulvsb_score_batch_sharded ends with the 8-byte ncclAllReduce(max).
    -> (summary, outputs of the last step: this rank's inlier counts and the global best)."""
    torch, capi = c.torch, c.capi
    from psulvsb_b200 import sharding, stages

    L = capi.lib()
    pair = c.synth.make_pair(n, 0.95, 777)
    (cs, cd), bound = stages.centre_and_bound(pair["src"], pair["dst"])
    d_src, d_dst = stages.to_device_points(pair["src"]), stages.to_device_points(pair["dst"])
    f_src, f_dst = stages.pack_points(d_src, cs), stages.pack_points(d_dst, cd)
    hb, he = sharding.shard_range(H, c.rank, c.world)
    g = torch.Generator(device="cuda").manual_seed(99)  # same stream of hypotheses on every rank, sliced
    q = torch.randn((H, 4), generator=g, device="cuda", dtype=torch.float64)
    q = q / q.norm(dim=1, keepdim=True)
    w, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y + z * w), 2 * (x * z - y * w),
                     2 * (x * y - z * w), 1 - 2 * (x * x + z * z), 2 * (y * z + x * w),
                     2 * (x * z + y * w), 2 * (y * z - x * w), 1 - 2 * (x * x + y * y)], dim=1)  # column-major
    t = torch.randn((H, 3), generator=g, device="cuda", dtype=torch.float64)
    hyp = torch.cat([R, t], dim=1)
    truth = torch.from_numpy(np.concatenate([pair["R"].ravel(order="F"), pair["t"]])).cuda()
    hyp[H // 3] = truth  # one hypothesis is the ground truth: the argmax must find it
    hyp_local = hyp[hb:he].contiguous()
    del hyp, R, t, q
    tau = 0.04
    counts = torch.zeros(he - hb, dtype=torch.int32, device="cuda")
    best = torch.zeros(1, dtype=torch.int64, device="cuda")
    border = torch.zeros(1, dtype=torch.int64, device="cuda")
    csa = (ctypes.c_double * 3)(*[float(v) for v in cs])
    cda = (ctypes.c_double * 3)(*[float(v) for v in cd])

    def run():
        best.zero_()
        capi.check(L.psulvsb_score_batch_sharded(c.h._h, torch.cuda.current_stream().cuda_stream, f_src.data_ptr(),
                                                 f_dst.data_ptr(), d_src.data_ptr(), d_dst.data_ptr(), n,
                                                 hyp_local.data_ptr(), he - hb, hb, 1.0, tau, bound, csa, cda,
                                                 counts.data_ptr(), best.data_ptr(), border.data_ptr()))

    # inside the default line this stage follows seconds of host-only work (CPU baseline, parity check): the SM clock
    # has dropped to idle by then and three 26 ms warm-up launches do not bring it back (measured: 29.9 ms against
    # 26.5 ms with the clocks up) -- warm up for half a second, then time with the clock sampled DURING the steps
    # (a FIXED number of launches -- every rank must make the same number of calls: run() ends with a collective --
    # of about half a second in total: 20 launches of 26 ms on one GPU, 160 of 3.4 ms on eight)
    for _ in range(min(20 * c.world, 200)):
        run()
    torch.cuda.synchronize()
    stage_sampler = ClockSampler(c.local_rank)
    stage_sampler.start()
    ms = timed_stream(c, run, steps, warmup)
    stage_clocks = stage_sampler.stop()
    f = stage_clocks.get("sm_mhz") or sm_clock_now(c) or 1965.0
    cnt, hid = sharding.unpack_best(int(best.item()))
    if hid != H // 3:
        raise SystemExit(f"bench.py: scoring sweep found hypothesis {hid} (count {cnt}), expected {H // 3}")
    # end to end: this rank's hypotheses start in pinned host memory, the packed best key ends on the host
    e2e = None
    if with_e2e:
        hyp_host = hyp_local.cpu().pin_memory()
        best_host = torch.zeros(1, dtype=torch.int64).pin_memory()

        def run_e2e():
            hyp_local.copy_(hyp_host, non_blocking=True)
            run()
            best_host.copy_(best, non_blocking=True)

        ms_e2e = timed_stream(c, run_e2e, steps, 1)
        e2e = {"value": H * n / (ms_e2e / 1e3), "unit": "scores/s", "ms_per_step": ms_e2e,
               "h2d_bytes_per_step": int(hyp_host.numel() * 8) * c.world, "d2h_bytes_per_step": 8 * c.world,
               "how": "every step copies the rank's hypotheses (96 B each) from pinned host memory, scores, and reads the "
                      "packed best key back; the correspondences stay resident"}
    units = H * n
    peak = c.world * c.sms * 128 * f * 1e6 / 1e9
    ach = units * 16 / (ms / 1e3) / 1e9
    outputs = {"inlier_counts": counts.cpu().numpy(), "best_count": [cnt], "best_hypothesis": [hid]}
    return {"case": "hypothesis scoring sweep (cfg-D)", "n": n, "hypotheses": H, "n_gpus": c.world, "units": units,
            "ms": ms, "scores_per_s": units / (ms / 1e3),
            "best": {"count": cnt, "hypothesis": hid, "expected_hypothesis": H // 3},
            "roofline": {"bound": "fp32-pipe", "achieved": ach, "peak": peak, "frac": ach / peak,
                         "unit": "Gslot/s (16 FP32-pipe issue slots per (hypothesis, point))",
                         "peak_source": f"{c.world} x {c.sms} SMs x 128 lanes x {f:.0f} MHz (SM clock sampled during the steps)"},
            "clocks": stage_clocks, "e2e": e2e,
            "hbm_hypothesis_stream_gbs": H * 96 / c.world / (ms / 1e3) / 1e9,
            "sharding": "hypotheses sliced across ranks; one 8-byte ncclAllReduce(max) of (count<<32 | ~id) on the same "
                        "stream, inside psulvsb_score_batch_sharded"}, outputs


def run_cfgD(args, c):
    steps, W = args.steps, max(args.warmup, 3)
    sampler = ClockSampler(c.local_rank)
    sampler.start()
    s, outputs = stage_k4(c, steps=steps, warmup=W, with_e2e=True)
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs, c.rank)
    if c.rank != 0:
        return None
    return {"metric": "hypothesis-point scores/s", "value": s["scores_per_s"], "unit": "scores/s", "n_gpus": c.world,
            "steps": steps, "warmup": W, "ms_per_step": s["ms"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32 (+f64 recheck of borderline points)",
            "data": "synthetic",
            "config": {"workload": "cfgD: 2^20 hypotheses x N=50000 correspondences, hypotheses sharded across GPUs",
                       "l2": "hypothesis stream (100 MB per GPU at N=1) read once per step; points from L2"},
            "e2e": s["e2e"], "gpu_launches": 3 * steps, "clocks": clocks,  # two re-layout launches + the scoring kernel
            "roofline": dict(s["roofline"], kernel="score_batch_kernel"), "best": s["best"], "sharding": s["sharding"]}


def run_cfgB(args, c):
    """ONE registration at N = 100 000, 99 % outliers, rows of the consistency stage sharded over the ranks."""
    capi, synth = c.capi, c.synth
    n = 100_000
    pair = synth.make_pair(n, 0.99, 4242, side=30.0)
    prob = capi.HostProblem(pair["src"], pair["dst"])
    params = capi.default_params(seed=11, **PARAM_KW)
    steps, W = args.steps, 2
    solve = (lambda: c.h.solve_sharded(params, prob)) if c.world > 1 else (lambda: c.h.solve(params, prob)[0])
    sampler = ClockSampler(c.local_rank)
    sampler.start()
    for _ in range(W):
        sol = solve()
    barrier(c)
    dev = k1 = 0.0
    t0 = time.perf_counter()
    for _ in range(steps):
        sol = solve()
        dev += c.h.last_device_ms
        k1 += c.h.last_stage_ms(2)
    barrier(c)
    wall = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop()
    dev_max, wall_max, k1_max = max_over_ranks(c, dev, wall, k1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, solution_arrays([sol]), c.rank)
    if c.rank != 0:
        return None
    f_mhz = clocks["sm_mhz"] or 1965.0
    pairs_total = n * (n - 1) // 2
    ach = pairs_total * 16 / (k1_max / steps / 1e3) / 1e9
    peak = c.world * c.sms * 128 * f_mhz * 1e6 / 1e9
    return {"metric": "registrations/s", "value": steps / (dev_max / 1e3), "unit": "registrations/s", "n_gpus": c.world,
            "steps": steps, "warmup": W, "ms_per_step": dev_max / steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64+f32", "data": "synthetic",
            "config": {"workload": "cfgB: ONE registration, N=100000 correspondences, 99% outliers, cube side 30, "
                                   "consistency rows sharded across the GPUs",
                       "n_reduced": int(sol.n_reduced), "final_inliers": int(sol.final_inlier_count),
                       "rotation_error_vs_truth_rad": synth.rotation_error(sol.R, pair["R"]),
                       "translation_error_vs_truth": float(np.linalg.norm(sol.t - pair["t"])),
                       "l2": "the 1.25 GB mask exceeds the L2"},
            "e2e": {"value": steps / (wall_max / 1e3), "unit": "registrations/s",
                    "h2d_bytes_per_step": prob.nbytes * c.world, "d2h_bytes_per_step": ctypes.sizeof(capi.Solution) * c.world},
            "gpu_launches": None, "clocks": clocks,
            "roofline": {"bound": "fp32-pipe", "kernel": "k1_mask_kernel", "achieved": ach, "peak": peak,
                         "frac": ach / peak, "unit": "Gslot/s (16 per pair)", "kernel_ms": k1_max / steps,
                         "share_of_step": k1_max / dev_max,
                         "peak_source": f"{c.world} x {c.sms} SMs x 128 lanes x {f_mhz:.0f} MHz"}}


def run_bunny(args, c):
    """configs[0] with the reference's timed region (PSULVSB.cc:309-329): pre-filter + mask_filter + solve.  The
    reference's driver runs its trials one after the other; here the trials of a step advance together as one batch
    (`value`, `e2e`), and one trial alone is reported as `latency_ms_single`."""
    capi = c.capi
    from psulvsb_b200 import io as pio

    trials = 592  # one batch of lock-step chunks, like cfgA
    cases = [bunny_case(500 + c.rank * 1000 + i) for i in range(trials)]
    seeds = [500 + c.rank * 1000 + i for i in range(trials)]
    normals = [(pio.estimate_normals(p["src"]), pio.estimate_normals(p["dst"])) for p in cases]  # untimed (PSULVSB.cc:307)
    params = capi.default_params(**PARAM_KW)

    def prefilter(i):
        # PSULVSB.cc:310-317 in one device call: normal-angle histogram, keep_mask, reduced clouds, reduce_map
        p = cases[i]
        keep, src_r, dst_r, rmap, _ = pio.prefilter_reduce(normals[i][0], normals[i][1], p["src"], p["dst"])
        return capi.HostProblem(src_r, dst_r, p["src"], p["dst"], keep, rmap)

    def prefilter_all():
        # ... and for the whole batch in one launch (a CTA per trial): psulvsb_prefilter_reduce_batch
        res = pio.prefilter_reduce_batch([x[0] for x in normals], [x[1] for x in normals], [p["src"] for p in cases],
                                         [p["dst"] for p in cases])
        return [capi.HostProblem(sr, tr, p["src"], p["dst"], keep, rmap) for (keep, sr, tr, rmap, _), p in zip(res, cases)]

    steps, W = args.steps, 3
    probs = prefilter_all()
    r = timed_resident(c, params, probs, seeds, steps, W)
    barrier(c)
    t0 = time.perf_counter()
    pre_ms = 0.0
    for _ in range(steps):
        t1 = time.perf_counter()
        filtered = prefilter_all()
        pre_ms += (time.perf_counter() - t1) * 1e3
        sols = c.h.solve_batch(params, filtered, seeds)
    barrier(c)
    e2e_ms = (time.perf_counter() - t0) * 1e3
    lat = []
    for i in range(8):
        t0 = time.perf_counter()
        params.seed = seeds[i]
        c.h.solve(params, prefilter(i))
        lat.append((time.perf_counter() - t0) * 1e3)
    dev_max, e2e_max = max_over_ranks(c, r["dev_ms"], e2e_ms)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, solution_arrays(r["sols"]), c.rank)
    if c.rank != 0:
        return None
    errs = [c.synth.rotation_error(s.R, p["R"]) for s, p in zip(sols, cases)]
    line = {"metric": "registrations/s", "value": trials * steps * c.world / (dev_max / 1e3), "unit": "registrations/s",
            "n_gpus": c.world, "steps": steps, "warmup": W, "ms_per_step": dev_max / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64+f32",
            "data": "synthetic (bunny vertices shipped by the reference)",
            "config": {"workload": f"bunny: configs[0], bun_zipper_res3 (1889 vertices), random rigid transform, +-0.05 "
                                   f"noise, 90% gross outliers, {trials} trials per GPU per step advanced as one batch; "
                                   f"e2e times what the reference times (PSULVSB.cc:309-329): histogram pre-filter + "
                                   f"mask_filter + solve, host buffers",
                       "median_rotation_error_rad": float(np.median(errs)),
                       "mean_final_inliers": float(np.mean([s.final_inlier_count for s in sols])),
                       "mean_C_after_prefilter": float(np.mean([p.src.shape[1] for p in probs])),
                       "ticks_per_step": float(np.mean(r["ticks"])),
                       "prefilter_ms_per_step": pre_ms / steps},
            "e2e": {"value": trials * steps * c.world / (e2e_max / 1e3), "unit": "registrations/s",
                    "h2d_bytes_per_step": int(sum(p.nbytes for p in probs)) * c.world,
                    "d2h_bytes_per_step": ctypes.sizeof(capi.Solution) * trials * c.world},
            "latency_ms_single": {"wall_ms": float(np.median(lat[3:])),
                                  "what": "pre-filter + psulvsb_solve of ONE trial, host buffers (median of 5)"},
            "gpu_launches": int(r["launches"])}
    if not args.no_cpu_baseline:
        from oracle import oracle as O
        from oracle import prefilter as PF

        n_cpu = 32
        t0 = time.perf_counter()
        bad = 0
        for i in range(n_cpu):
            p = cases[i]
            keep, _ = PF.histogram_outlier_removal(normals[i][0], normals[i][1])
            src_r, dst_r, rmap = PF.mask_filter(p["src"], p["dst"], keep)
            po = O.default_params(seed=seeds[i], **PARAM_KW)
            ref, _ = O.solve(po, src_r, dst_r, p["src"], p["dst"], keep, rmap, trace_cap=1)
            s = sols[i]
            if (ref.valid, ref.final_inlier_count, ref.local_iters) != (s.valid, s.final_inlier_count, s.local_iters) or \
                    (ref.valid and c.synth.rotation_error(s.R, O.solution_R(ref)) > 1e-5):
                bad += 1
        tcpu = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": n_cpu / tcpu, "unit": "registrations/s", "cores": 1, "kind": "port",
                                "sample": f"the first {n_cpu} trials: numpy pre-filter + CPU oracle, {tcpu:.1f} s"}
        line["parity"] = {"checked": n_cpu, "mismatch": bad,
                          "fields": "valid, final_inlier_count, local_iters exact; R < 1e-5 rad"}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="cfgA", choices=["cfgA", "cfgB", "cfgC", "cfgD", "bunny"])
    ap.add_argument("--batch", type=int, default=592,
                    help="cfgA: fragment pairs per GPU per step (default: four per SM of a 148-SM B200; the library "
                         "advances them as two lock-step chunks of 296 on two engines)")
    ap.add_argument("--chunk", type=int, default=0, help="registrations per lock-step chunk (0: library default)")
    ap.add_argument("--lanes", type=int, default=0, help="chunks in flight at once (0: library default)")
    ap.add_argument("--debug", default="", help="name=value[,name=value] for psulvsb_debug_set")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="cfgA: skip stages / variants (kernel tuning runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy "
                         "(float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; it does not apply to --impl reference")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    c = setup(args)
    if args.config in ("cfgA", "cfgC"):
        line, params = run_cfgA(args, c, CFGC_PAIRS if args.config == "cfgC" else 0)
        if args.config == "cfgA" and not args.no_extras:
            stages = {"k1_100k": stage_k1(c), "k4_1Mx50k": stage_k4(c)[0]}
            n_check = 0 if args.no_cpu_baseline else 16
            variants = {
                "mode2_prefilter_selfupdate": run_variant(
                    c, params, "cfg-A pairs through the emulated pre-filter (keeps 60% of the inliers, 30% of the "
                               "outliers: C ~ 1600 of M = 5000), self-update active", 2, "fpfh", args.batch, 3, n_check),
                "gross_outliers": run_variant(
                    c, params, "cfg-A pairs with gross outliers (dst += +-U[5,10] per axis, PSULVSB.cc:200-220)", 1,
                    "gross", args.batch, 3, n_check),
            }
            if line is not None:
                line["stages"] = stages
                line["variants"] = variants
    elif args.config == "cfgB":
        line = run_cfgB(args, c)
    elif args.config == "cfgD":
        line = run_cfgD(args, c)
    else:
        line = run_bunny(args, c)
    rc = 0
    if c.rank == 0 and line is not None:
        print(json.dumps(line), flush=True)
        par = [line.get("parity")] + [v.get("parity") for v in (line.get("variants") or {}).values() if v]
        if any(p and p.get("mismatch", 0) > 0 for p in par):
            print("bench.py: GPU results differ from the CPU oracle (see `parity`)", file=sys.stderr)
            rc = 3
    if c.world > 1:
        c.dist.barrier()
        c.dist.destroy_process_group()
    c.h.close()
    sys.exit(rc)


if __name__ == "__main__":
    main()
