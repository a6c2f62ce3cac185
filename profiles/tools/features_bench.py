"""Times the correspondence stage (csrc/k8_features.cu) on one GPU: FPFH (radius normals + SPFH + FPFH, with the grid
build) at N = 5 000 and 50 000 points of the seeded synthetic surface (synth.make_surface), and the two-way descriptor
nearest neighbour (the matcher's kernel) at 5k x 5k and 50k x 50k.  CUDA events around back-to-back calls after a
warm-up, at least `--min-seconds` of timed work per line; the device name, power limit and SM clock are read in the
same run.  The NN rate is reported against the FP32-pipe roofline of DESIGN.md section 6 (SMs x 128 lanes x SM clock)
with the difference form's unit cost: 66 FP32 lane operations per distance (33 FADD halves + 33 FFMA halves; the 34th,
padding dimension is not counted).

    python profiles/tools/features_bench.py [--out profiles/r3_features_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import psulvsb_b200  # noqa: E402,F401
from psulvsb_b200 import features, stages, synth  # noqa: E402

UNIT_SLOTS = 66


def smi(query):
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=" + query, "--format=csv,noheader,nounits", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return ""


def timed(fn, min_seconds):
    import torch

    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    reps, ms = 1, 0.0
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= 1000.0 * min_seconds:
            return ms / reps, reps
        reps = max(reps * 2, int(reps * 1.2 * 1000.0 * min_seconds / max(ms, 1e-3)))


def mean_neighbours(P, r):
    from scipy.spatial import cKDTree

    t = cKDTree(P.T)
    return float(np.mean([len(x) for x in t.query_ball_point(P.T, r)]))


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_features_bench.json"))
    ap.add_argument("--min-seconds", type=float, default=1.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("features_bench: no CUDA device (nothing is measured without one)")
    res = {"device": torch.cuda.get_device_name(0), "power_limit_w": smi("power.limit"),
           "sm_clock_max_mhz": smi("clocks.max.sm"), "sms": torch.cuda.get_device_properties(0).multi_processor_count,
           "fpfh": [], "nn": []}
    # radii scale with the spacing (1 / sqrt(N)) so that both sizes see about the same neighbourhoods
    for n in (5000, 50000):
        P = synth.make_surface(n, 1)
        s = (5000.0 / n) ** 0.5
        rn, rf = 0.06 * s, 0.1 * s
        d = stages.to_device_points(P)
        ms, reps = timed(lambda: features.fpfh_device(d, rn, rf), args.min_seconds)
        res["fpfh"].append({"n": n, "normal_radius": rn, "feature_radius": rf, "ms": ms, "reps": reps,
                            "points_per_s": n / ms * 1e3, "mean_normal_neighbours": mean_neighbours(P, rn),
                            "mean_feature_neighbours": mean_neighbours(P, rf)})
        print(json.dumps(res["fpfh"][-1]), flush=True)
    clock = smi("clocks.sm")
    res["sm_clock_during_mhz"] = clock
    f_mhz = float(clock) if clock else float(res["sm_clock_max_mhz"] or 1965)
    roof = res["sms"] * 128 * f_mhz * 1e6 / UNIT_SLOTS
    for n in (5000, 50000):
        P = synth.make_surface(n, 1)
        s = (5000.0 / n) ** 0.5
        fs, _ = features.fpfh_device(stages.to_device_points(P), 0.06 * s, 0.1 * s)
        R, _ = synth.random_rigid(np.random.default_rng(2))
        ft, _ = features.fpfh_device(stages.to_device_points(R @ P), 0.06 * s, 0.1 * s)
        ms, reps = timed(lambda: features.nearest_neighbours_device(fs, ft), args.min_seconds)
        rate = n * n / ms * 1e3
        res["nn"].append({"n_src": n, "n_tgt": n, "ms": ms, "reps": reps, "distances_per_s": rate,
                          "roofline_distances_per_s": roof, "of_roofline": rate / roof})
        print(json.dumps(res["nn"][-1]), flush=True)
    res["when"] = time.strftime("%Y-%m-%d %H:%M:%S")
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("device", "power_limit_w", "sm_clock_during_mhz")}))


if __name__ == "__main__":
    main()
