"""Times the K9 Tanks and Temples evaluation (csrc/pointcloud.cu, mvs_b200/tanks.py) on a synthetic T&T-sized scene, and the fp64
oracle pipeline on the host cores as the stand-in for the toolbox (whose Open3D is not used here) -> one JSON file.

    python tools/bench_tnt_eval.py --out profiles/r08_bench_tnt_eval.json [--rounds 5] [--scale 1.0]

Workload (seeded, metres): a wavy terrain z = 0.5 sin(x / 3) cos(y / 4) over 40 x 25 m; the ground truth samples it uniformly (about
20 M points, about 7 mm apart); the reconstruction samples x < 36 m of it (about 10 M points) with 3 mm Gaussian noise per axis and
5 % outliers spread over the box, given in a frame a similarity transform maps to the ground truth's.  tau = 0.01.  The crop volume
(orthogonal axis z, a concave hexagon, z in [-1, 1.5]) cuts part of both clouds.  --scale multiplies both point counts.

Timing: CUDA events around whole calls after a warm-up, median and range over --rounds; per stage, events around each stage of one
call run stage by stage, over the same rounds.  Also: the card's name and power limit, and how many `< tau` decisions differ between
the GPU (fp32 distances) and the oracle on the un-rounded fp64 down-sampled points."""
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

import tnt_eval as oracle  # noqa: E402
from mvs_b200 import evaluation, tanks  # noqa: E402

TAU = 0.01
LX, LY = 40.0, 25.0
POLYGON = [[1.0, 1.0, 0.0], [30.0, 2.0, 0.0], [38.0, 12.0, 0.0], [20.0, 10.0, 0.0], [28.0, 23.0, 0.0], [2.0, 22.0, 0.0]]


def _terrain(g, n, dev, x_max=LX):
    x = torch.rand(n, generator=g, device=dev, dtype=torch.float64) * x_max
    y = torch.rand(n, generator=g, device=dev, dtype=torch.float64) * LY
    return torch.stack([x, y, 0.5 * torch.sin(x / 3) * torch.cos(y / 4)], 1)


def workload(dev, scale):
    g = torch.Generator(device=dev).manual_seed(0)
    m, n = int(20_000_000 * scale), int(10_000_000 * scale)
    gt = _terrain(g, m, dev).float().contiguous()
    n_out = int(0.05 * n)
    rec = _terrain(g, n - n_out, dev, 36.0) + 0.003 * torch.randn(n - n_out, 3, generator=g, device=dev, dtype=torch.float64)
    lo, hi = torch.tensor([0.0, 0.0, -2.0], device=dev, dtype=torch.float64), torch.tensor([LX, LY, 2.0], device=dev, dtype=torch.float64)
    rec = torch.cat([rec, lo + torch.rand(n_out, 3, generator=g, device=dev, dtype=torch.float64) * (hi - lo)])
    c, s = np.cos(0.3), np.sin(0.3)
    A = np.eye(4)
    A[:3, :3] = 1.25 * np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
    A[:3, 3] = [2.0, -1.0, 0.5]
    Ai = torch.from_numpy(np.linalg.inv(A[:3, :3])).to(dev)
    rec_in = ((rec - torch.from_numpy(A[:3, 3]).to(dev)) @ Ai.T).float().contiguous()
    crop = tanks._crop_volume("Z", -1.0, 1.5, POLYGON)
    return rec_in, gt, crop, A


class Events:
    def __init__(self):
        self.ms = {}

    def stage(self, name):
        ev = self

        class _S:
            def __enter__(self):
                self.a = torch.cuda.Event(enable_timing=True)
                self.a.record()

            def __exit__(self, *exc):
                b = torch.cuda.Event(enable_timing=True)
                b.record()
                b.synchronize()
                ev.ms.setdefault(name, []).append(self.a.elapsed_time(b))
        return _S()


def staged_call(x, gt, crop, A, tau, ev):
    """evaluate_tanks_and_temples stage by stage, each bracketed by events (the same calls in the same order)."""
    edges = tanks.histogram_edges(tau)
    with ev.stage("crop"):
        xs, _ = tanks.crop_points(x, crop, A)
        gs, _ = tanks.crop_points(gt, crop, None)
    with ev.stage("keys"):
        kx, kg = tanks.voxel_keys(xs, tau / 2), tanks.voxel_keys(gs, tau / 2)
    with ev.stage("sort_and_means"):
        s64, s32, _ = tanks.voxel_means(xs, kx)
        t64, t32, _ = tanks.voxel_means(gs, kg)
    cap = tanks.search_cap(tau, tanks.STRETCH, edges)
    with ev.stage("grids"):
        g_t, g_s = evaluation.build_grid(t32), evaluation.build_grid(s32)
    with ev.stage("search_rec_to_gt"):
        d_s = evaluation.nearest_distance(s32, t32, cap, grid=g_t)
    with ev.stage("search_gt_to_rec"):
        d_t = evaluation.nearest_distance(t32, s32, cap, grid=g_s)
    with ev.stage("statistics"):
        counts = tanks.statistics(d_s, d_t, tau, edges)
    return counts, s64, t64, d_s, d_t


def _summary(v):
    return {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "rounds_ms": [float(t) for t in v]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--no-host", action="store_true", help="skip the host oracle run")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_tnt_eval needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    dev = torch.device("cuda:0")
    x, gt, crop, A = workload(dev, a.scale)
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None,
           "timing": "CUDA events; warm-up call first; whole calls and stage-by-stage calls alternate over rounds; median and range",
           "workload": {"n": int(x.shape[0]), "m": int(gt.shape[0]), "tau": TAU, "stretch": tanks.STRETCH, "polygon": POLYGON,
                        "axis": "Z", "axis_min": -1.0, "axis_max": 1.5, "transform": A.tolist()}}
    out = tanks.evaluate_tanks_and_temples(x, gt, crop, A, TAU, return_details=True)          # warm-up
    whole, ev = [], Events()
    for _ in range(a.rounds):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0.record()
        r = tanks.evaluate_tanks_and_temples(x, gt, crop, A, TAU)
        t1.record()
        t1.synchronize()
        whole.append(t0.elapsed_time(t1))
        staged = staged_call(x, gt, crop, A, TAU, ev)
    res["whole_call"] = _summary(whole)
    res["stages"] = {k: _summary(v) for k, v in ev.ms.items()}
    res["stages_sum_median_ms"] = float(sum(np.median(v) for v in ev.ms.values()))
    res["result"] = {k: (v.tolist() if isinstance(v, np.ndarray) else v) for k, v in r.items()
                     if k not in ("edges", "cum_precision", "cum_recall")}
    res["staged_equals_whole"] = bool(staged[0][0] == r["n_precision"] and staged[0][1] == r["m_recall"])
    print(json.dumps({k: v for k, v in res.items() if k != "workload"}, default=str)[:3000], flush=True)
    if not a.no_host:
        xc, gc = x.cpu().numpy(), gt.cpu().numpy()
        del staged
        torch.cuda.empty_cache()
        t0 = time.perf_counter()
        w = oracle.evaluate(xc, gc, tuple(crop), A, TAU, round_fp32=False)
        dt = time.perf_counter() - t0
        d_s, d_t = out["d_s"].cpu().double().numpy(), out["d_t"].cpu().double().numpy()
        same = np.array_equal(out["xyz_down"].cpu().numpy(), w["xyz_down"]) and np.array_equal(out["gt_down"].cpu().numpy(), w["gt_down"])
        res["host_oracle_fp64"] = {
            "s": dt, "host_cpus": os.cpu_count(), "note": "oracle/tnt_eval.py (numpy + cKDTree on all cores), the stand-in for the toolbox",
            "down_sampled_clouds_bit_identical": bool(same),
            "tau_decisions_differ_rec_to_gt": int(np.sum((d_s < TAU) != (w["d_s"] < TAU))) if same else None,
            "tau_decisions_differ_gt_to_rec": int(np.sum((d_t < TAU) != (w["d_t"] < TAU))) if same else None,
            "precision": w["precision"], "recall": w["recall"], "fscore": w["fscore"]}
        print("host", json.dumps(res["host_oracle_fp64"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1, default=float)


if __name__ == "__main__":
    main()
