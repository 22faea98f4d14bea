"""Times the Tanks and Temples trajectory alignment (K9 trajectory alignment: csrc/pointcloud.cu, mvs_b200/registration.py) at the
toolbox's defaults, 100,000 RANSAC hypotheses, on oracle/tnt_align.py's orbit scene at 400 and 1600 cameras, and one run of the
vectorised fp64 oracle on the host cores -> one JSON file.

    python tools/bench_tnt_align.py --out profiles/r10_bench_tnt_align.json [--rounds 5]

Timing: a warm-up call per size, then rounds that alternate the two sizes; per round CUDA events around the whole call
(align_trajectory from the poses to the returned dict) and, inside it, events around the two kernels (ops.EVENTS); "host" is the
whole call minus the kernels (the centres, the uploads, the launch and the one read-back).  Median and range over the rounds.  Also
the card's name and power limit, read in the same run, and the result against the planted similarity and the oracle's choice."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "deep-multiview-depth-estimation_b200"), os.path.join(ROOT, "oracle")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import tnt_align as oracle  # noqa: E402
import tnt_register  # noqa: E402
from mvs_b200 import ops, registration  # noqa: E402

N_HYP = 100_000
SIZES = (400, 1600)


def _summary(v):
    return {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "rounds_ms": [float(t) for t in v]}


def timed_call(sc):
    ops.EVENTS = {}
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    r = registration.align_trajectory(sc["poses"], sc["reference"], sc["gt_trans"], max_iteration=N_HYP)
    t1.record()
    t1.synchronize()
    kern = float(sum(a.elapsed_time(b) for a, b, _ in ops.EVENTS["pc_ransac_align"]))
    ops.EVENTS = None
    whole = t0.elapsed_time(t1)
    return r, whole, kern


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--no-host", action="store_true", help="skip the host oracle run")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_tnt_align needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    scenes = {n: oracle.orbit_scene(n=n) for n in SIZES}
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "hypotheses": N_HYP,
           "timing": "CUDA events; a warm-up call per size; rounds alternate the sizes; median and range",
           "workload": "oracle/tnt_align.py orbit_scene(n): 1.3 turns, ~40 units across, noise 0.01, 15 % outliers displaced 1-3 units",
           "sizes": {}}
    for n in SIZES:
        timed_call(scenes[n])
    rounds = {n: {"whole": [], "kernels": [], "host": []} for n in SIZES}
    results = {}
    for _ in range(a.rounds):
        for n in SIZES:
            r, whole, kern = timed_call(scenes[n])
            rounds[n]["whole"].append(whole)
            rounds[n]["kernels"].append(kern)
            rounds[n]["host"].append(whole - kern)
            results[n] = r
    for n in SIZES:
        r = results[n]
        ang, sc, tr = tnt_register.similarity_error(r["transformation"], scenes[n]["S_true"])
        res["sizes"][str(n)] = {"cameras": n, "pair_tests": N_HYP * n, "whole_call": _summary(rounds[n]["whole"]),
                                "kernels": _summary(rounds[n]["kernels"]), "host": _summary(rounds[n]["host"]),
                                "hypothesis": r["hypothesis"], "inliers": r["inliers"], "planted_inliers": int((~scenes[n]["outlier"]).sum()),
                                "inlier_rmse": r["inlier_rmse"],
                                "error_vs_planted": {"rotation_rad": ang, "scale": sc, "translation": tr}}
        print(n, json.dumps(res["sizes"][str(n)])[:600], flush=True)
    if not a.no_host:
        sc = scenes[SIZES[0]]
        t0 = time.perf_counter()
        want = oracle.align(sc["poses"], sc["reference"], sc["gt_trans"], n_hyp=N_HYP)
        dt = time.perf_counter() - t0
        res["host_oracle_fp64"] = {"note": "oracle/tnt_align.py: per-hypothesis numpy Umeyama, vectorised numpy scoring; one run",
                                   "cameras": SIZES[0], "s": dt, "host_cpus": os.cpu_count(), "hypothesis": want["hypothesis"],
                                   "gpu_hypothesis": results[SIZES[0]]["hypothesis"], "oracle_gap": want["gap"]}
        print("host", json.dumps(res["host_oracle_fp64"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1, default=float)


if __name__ == "__main__":
    main()
