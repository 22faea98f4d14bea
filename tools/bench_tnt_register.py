"""Times the Tanks and Temples registration (K9 registration: csrc/pointcloud.cu, mvs_b200/registration.py) on tools/bench_tnt_eval.py's
T&T-sized scene with a planted perturbation of its alignment, and one iteration of the fp64 oracle's ICP on the host cores as the
stand-in for Open3D (which is not used here) -> one JSON file.

    python tools/bench_tnt_register.py --out profiles/r09_bench_tnt_register.json [--rounds 3] [--scale 1.0]

Workload: bench_tnt_eval.workload (about 20 M ground-truth and 10 M reconstruction points, tau = 0.01), its alignment A perturbed to
T0 = P A with P a similarity of 3 degrees about an oblique axis through the crop's centre, scale 1.02 and a shift of 3 tau per axis.
Timing: CUDA events around whole calls after a warm-up call, median and range over --rounds; per stage of one call, events around
each launch (ops.EVENTS) summed by kernel, and the host's share (SVD, composition, the per-iteration read-back and launch issue) as
the stage's wall time minus its kernel time.  Also: the card's name and power limit, the error of the result against the planted
perturbation, and precision / recall / F-score under A, T0 and the registered transform."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "deep-multiview-depth-estimation_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tools")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench_tnt_eval  # noqa: E402
import tnt_register as oracle  # noqa: E402
from mvs_b200 import ops, registration, tanks  # noqa: E402

TAU = bench_tnt_eval.TAU


def _summary(v):
    return {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "rounds_ms": [float(t) for t in v]}


def _events_ms(ev):
    torch.cuda.synchronize()
    return {k: float(sum(a.elapsed_time(b) for a, b, _ in v)) for k, v in ev.items()}, {k: len(v) for k, v in ev.items()}


def staged(x, gt, crop, T0, tau):
    """register_tanks_and_temples stage by stage (the same calls), with every kernel bracketed by events."""
    gs, _ = tanks.crop_points(gt, crop, None)
    T, out = T0, []
    for method, param, d_max in (("voxel", tau, 80 * tau), ("voxel", tau / 2, 20 * tau), ("uniform", None, 2 * tau)):
        torch.cuda.synchronize()
        ops.EVENTS = {}
        t0 = time.perf_counter()
        xs, _ = tanks.crop_points(x, crop, T)
        if method == "voxel":
            s64 = tanks.voxel_down_sample(xs, param)[0]
            t64, t32 = tanks.voxel_down_sample(gs, param)[:2]
        else:
            s64 = xs[::registration.uniform_rate(xs.shape[0])].contiguous()
            t64 = gs[::registration.uniform_rate(gs.shape[0])].contiguous()
            t32 = t64.float()
        grid = registration.build_grid(t32)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        prep, _ = _events_ms(ops.EVENTS)
        ops.EVENTS = {}
        r = registration.icp_point_to_point(s64, t64, d_max, target_grid=grid)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        kern, launches = _events_ms(ops.EVENTS)
        ops.EVENTS = None
        T = r["transformation"] @ T
        icp_ms = (t2 - t1) * 1e3
        out.append({"method": method, "n_down": s64.shape[0], "m_down": t64.shape[0], "iterations": r["iterations"],
                    "correspondences": r["correspondences"], "prepare_wall_ms": (t1 - t0) * 1e3, "prepare_kernels_ms": prep,
                    "icp_wall_ms": icp_ms, "search_ms": kern.get("pc_nearest_index", 0.0), "sums_ms": kern.get("pc_icp_sums", 0.0),
                    "transform_ms": kern.get("pc_transform64", 0.0), "launches": launches,
                    "host_solve_and_readback_ms": icp_ms - sum(kern.values())})
    return T, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--no-host", action="store_true", help="skip the host oracle iteration")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_tnt_register needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    dev = torch.device("cuda:0")
    x, gt, crop, A = bench_tnt_eval.workload(dev, a.scale)
    c = np.array([20.0, 12.5, 0.0])
    P = oracle.similarity(oracle.rotation([0.4, -0.3, 1.0], 3.0), 1.02, np.zeros(3))
    P[:3, 3] = c - P[:3, :3] @ c + 3 * TAU
    T0 = P @ A
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None,
           "timing": "CUDA events; warm-up call first; whole calls and stage-by-stage calls alternate over rounds; median and range",
           "workload": {"n": int(x.shape[0]), "m": int(gt.shape[0]), "tau": TAU, "A": A.tolist(), "T0": T0.tolist(),
                        "perturbation": "3 deg about (0.4, -0.3, 1) through (20, 12.5, 0), scale 1.02, shift 3 tau per axis"}}
    reg = registration.register_tanks_and_temples(x, gt, crop, T0, TAU)            # warm-up
    whole, stages = [], []
    for _ in range(a.rounds):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0.record()
        reg = registration.register_tanks_and_temples(x, gt, crop, T0, TAU)
        t1.record()
        t1.synchronize()
        whole.append(t0.elapsed_time(t1))
        T_staged, st = staged(x, gt, crop, T0, TAU)
        stages.append(st)
    res["whole_call"] = _summary(whole)
    keys = ("prepare_wall_ms", "icp_wall_ms", "search_ms", "sums_ms", "transform_ms", "host_solve_and_readback_ms")
    res["stages"] = [{**{k: v for k, v in stages[-1][i].items() if k not in keys},
                      **{k: _summary([r[i][k] for r in stages]) for k in keys}} for i in range(3)]
    res["staged_equals_whole"] = bool(np.array_equal(T_staged, reg["transformation"]))
    res["registration"] = [{k: (v.tolist() if isinstance(v, np.ndarray) else v) for k, v in s.items()} for s in reg["stages"]]
    ang, sc, tr = oracle.similarity_error(reg["transformation"], A)
    ang0, sc0, tr0 = oracle.similarity_error(T0, A)
    res["error_vs_planted"] = {"before": {"rotation_rad": ang0, "scale": sc0, "translation": tr0},
                               "after": {"rotation_rad": ang, "scale": sc, "translation": tr}}
    res["scores"] = {}
    for name, T in (("exact", A), ("init", T0), ("registered", reg["transformation"])):
        e = tanks.evaluate_tanks_and_temples(x, gt, crop, T, TAU)
        res["scores"][name] = {k: e[k] for k in ("precision", "recall", "fscore")}
    print(json.dumps({k: v for k, v in res.items() if k != "workload"}, default=str)[:4000], flush=True)
    if not a.no_host:
        # one ICP iteration of the oracle (one cKDTree correspondence search on all cores + the Umeyama update + the next search)
        # on stage 3's inputs, the stand-in for Open3D's per-iteration cost
        T2 = np.array(reg["stages"][1]["transformation"])
        xs, _ = tanks.crop_points(x, crop, T2)
        gs, _ = tanks.crop_points(gt, crop, None)
        s = xs[::registration.uniform_rate(xs.shape[0])].cpu().numpy()
        t = gs[::registration.uniform_rate(gs.shape[0])].cpu().numpy()
        t0 = time.perf_counter()
        from scipy.spatial import cKDTree
        tree = cKDTree(t.astype(np.float32).astype(np.float64))
        t_tree = time.perf_counter() - t0
        t0 = time.perf_counter()
        oracle.icp(s, t, 2 * TAU, max_iteration=1)
        dt = time.perf_counter() - t0
        del tree
        res["host_oracle_fp64"] = {"note": "oracle/tnt_register.py, numpy + cKDTree on all cores, a stand-in for Open3D: one ICP "
                                           "iteration (two searches, one update) on stage 3's inputs, tree build included",
                                   "s": dt, "tree_build_s": t_tree, "host_cpus": os.cpu_count(), "n": len(s), "m": len(t)}
        print("host", json.dumps(res["host_oracle_fp64"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1, default=float)


if __name__ == "__main__":
    main()
