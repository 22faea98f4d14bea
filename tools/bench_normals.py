"""Times K10 (csrc/pointcloud.cu pc_knn_kernel, mvs_b200/normals.py) on the two workloads users run it on -> one JSON file.

    python tools/bench_normals.py --out profiles/r11_bench_normals.json [--rounds 5]

Workloads:
  tnt    the toolbox's use: the down-sampled clouds of tools/bench_tnt_eval.py's scene (reconstruction and ground truth), k = 20,
         canonical sign, and the whole write_evaluation_files call on that evaluation.
  fused  tools/bench_fusion.py's cfg4-size cloud (49 views of 296 x 400, fuse_depth_maps), k = 30, oriented by point_viewpoints.

Per cloud: the search alone (k_nearest, dist and index written) against estimate_normals, and estimate_normals on grids of 1/2, 1
and 2 x the edge of the KNN_CELLS_PER_POINT rule; every grid is built outside the timed window.  Timing: CUDA events around each
call after a warm-up per shape; the compared forms alternate over --rounds rounds; median and range.  The card's name and power
limit are read in the same run.  One host run of the fp64 oracle (oracle/pc_normals.py) on a subsample, its size stated."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "deep-multiview-depth-estimation_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tools")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench_tnt_eval  # noqa: E402
import fusion as fusion_oracle  # noqa: E402
import pc_normals as oracle  # noqa: E402
import mvs_b200  # noqa: E402
from mvs_b200 import evaluation, tanks  # noqa: E402


def _ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def _alternate(fns, rounds):
    for fn in fns.values():
        fn()                                                        # warm-up of this shape
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            out[k].append(_ms(fn))
    return {k: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "rounds_ms": v}
            for k, v in out.items()}


def bench_cloud(x, k, views, rounds):
    g = evaluation.build_grid(x, cells_per_point=evaluation.KNN_CELLS_PER_POINT)
    grids = {1.0: g}
    for f in (0.5, 2.0):
        try:
            grids[f] = evaluation.build_grid(x, cell=g.cell * f)
        except mvs_b200.MvsB200Error as e:                          # a finer grid over the kernels' cell bound
            print(f"cell {f}x: {e}", flush=True)
    alt = [f for f in (0.5, 2.0) if f in grids]
    fns = {"pc_knn_alone": lambda: mvs_b200.k_nearest(x, x, k, grid=g),
           "pc_normals": lambda: mvs_b200.estimate_normals(x, k, viewpoints=views, grid=g)}
    for f in alt:
        fns[f"pc_normals_cell_{f}x"] = (lambda gg: lambda: mvs_b200.estimate_normals(x, k, viewpoints=views, grid=gg))(grids[f])
    times = _alternate(fns, rounds)
    same = all(torch.equal(mvs_b200.estimate_normals(x, k, viewpoints=views, grid=grids[f]),
                           mvs_b200.estimate_normals(x, k, viewpoints=views, grid=g)) for f in alt)
    zero = int((mvs_b200.estimate_normals(x, k, viewpoints=views, grid=g) == 0).all(1).sum())
    return {"points": int(x.shape[0]), "k": k, "viewpoints": views is not None, "cell_1x": g.cell,
            "cells": {str(f): {"cell": grids[f].cell, "blocks": grids[f].nb} for f in grids}, "kernels": times,
            "normals_identical_across_cells": bool(same), "zero_normals": zero}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0, help="multiplies the tnt workload's point counts")
    ap.add_argument("--host-sample", type=int, default=20000)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_normals needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    dev = torch.device("cuda:0")
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None,
           "timing": "CUDA events per call after a warm-up per shape; forms alternate over rounds; median and range; grids prebuilt",
           "list_storage": "shared memory [slot][thread] (the register form was not built)"}
    x, gt, crop, A = bench_tnt_eval.workload(dev, a.scale)
    ev = tanks.evaluate_tanks_and_temples(x, gt, crop, A, bench_tnt_eval.TAU, return_details=True)
    del x, gt
    rec32, gt32 = ev["xyz_down"].float().contiguous(), ev["gt_down"].float().contiguous()
    res["tnt_reconstruction"] = bench_cloud(rec32, tanks.NORMALS_KNN, None, a.rounds)
    print(json.dumps(res["tnt_reconstruction"])[:1500], flush=True)
    res["tnt_ground_truth"] = bench_cloud(gt32, tanks.NORMALS_KNN, None, a.rounds)
    print(json.dumps(res["tnt_ground_truth"])[:1500], flush=True)
    with tempfile.TemporaryDirectory() as d:
        res["write_evaluation_files"] = _alternate({"whole_call": lambda: tanks.write_evaluation_files(d, "Bench", ev)}, a.rounds)
    sub = np.random.default_rng(0).choice(rec32.shape[0], a.host_sample, replace=False)
    pts = rec32[torch.from_numpy(np.sort(sub)).to(dev)].cpu().numpy()
    t0 = time.perf_counter()
    want = oracle.normals(pts, tanks.NORMALS_KNN)
    t_host = time.perf_counter() - t0
    got = mvs_b200.estimate_normals(torch.from_numpy(pts).to(dev), tanks.NORMALS_KNN).cpu().numpy()
    sure = (want["nbr"] >= 1e-4) & (want["eigengap"] >= 1e-3) & (want["count"] >= 3)
    res["host_oracle"] = {"sample_points": int(a.host_sample), "sample": "uniform without replacement from the down-sampled reconstruction",
                          "s": t_host, "host_cpus": os.cpu_count(), "max_angle_rad_where_sure": float(oracle.angle(got[sure], want["normal"][sure]).max()),
                          "sure_share": float(sure.mean())}
    print("host", json.dumps(res["host_oracle"]), flush=True)
    del ev, rec32, gt32
    torch.cuda.empty_cache()
    N, h, w = 49, 296, 400
    s = fusion_oracle.analytic_scene(N, h, w, seed=0, focal=1.5 * w)
    rng = np.random.default_rng(1)
    depth = torch.from_numpy((s["depth"] * (1 + 2e-3 * rng.standard_normal(s["depth"].shape))).astype(np.float32))[:, None].to(dev)
    conf = torch.from_numpy(rng.uniform(0.5, 1.0, (N, 1, h, w)).astype(np.float32)).to(dev)
    colours = torch.from_numpy(rng.uniform(size=(N, 3, h, w)).astype(np.float32)).to(dev)
    src = [[(i + k) % N for k in (1, -1, 2, -2, 3, -3, 4, -4, 5, -5)] for i in range(N)]
    xyz, _, masks = mvs_b200.fuse_depth_maps(depth, conf, colours, s["K"], s["R"], s["T"], src)
    views = mvs_b200.point_viewpoints(masks, s["R"], s["T"])
    res["fused_cfg4"] = bench_cloud(xyz, 30, views, a.rounds)
    nrm = mvs_b200.estimate_normals(xyz, 30, viewpoints=views).double()
    ang = torch.atan2(torch.linalg.cross(nrm, torch.from_numpy(s["n0"]).to(dev).expand_as(nrm)).norm(dim=1),
                      (nrm @ torch.from_numpy(s["n0"]).to(dev)).abs())
    res["fused_cfg4"]["median_angle_to_disk_normal_rad"] = float(ang.median())
    res["fused_cfg4"]["facing_emitting_camera_share"] = float(((nrm * (views - xyz.double())).sum(1) > 0).double().mean())
    print(json.dumps(res["fused_cfg4"])[:1500], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1, default=float)


if __name__ == "__main__":
    main()
