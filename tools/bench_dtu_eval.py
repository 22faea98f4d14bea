"""Times the K8 point-cloud evaluation (csrc/pointcloud.cu) on a synthetic DTU-sized scan, and the host references -> one JSON file.

    python tools/bench_dtu_eval.py --out profiles/r05_bench_dtu_eval.json

Workload (seeded, DTU units = mm, BB 400 x 400 x 300): the ground truth is a hemisphere of radius 120 plus a ground ring (r 120..170)
sampled uniformly at 25 points / mm^2 (about 0.2 mm spacing); the data clouds sample the same surface at two sizes (about 2.1 M
points, the cfg4 size of bench_fusion, and about 10 M) with 1 mm Gaussian noise per axis and 3 % outliers spread over the box
(many beyond max_dist).  The observability mask (Res = 1 mm) holds the voxels within 15 mm of the surface.  Timing: CUDA events
around whole calls (each ends in a device synchronise or a read-back), warm-up first, compared forms alternating over rounds."""
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

import pointcloud_eval as oracle  # noqa: E402
from mvs_b200 import _lib, evaluation  # noqa: E402
from mvs_b200.ops import _stream  # noqa: E402

R_SPHERE, R_GROUND, DENSITY = 120.0, 170.0, 25.0
BB = np.array([[-200.0, -200.0, -50.0], [200.0, 200.0, 250.0]])
RES = 1.0
L2_BYTES = 126e6


def _surface(g, n, dev):
    """n points uniform by area on the hemisphere + the ground ring."""
    a_sph, a_gnd = 2 * np.pi * R_SPHERE ** 2, np.pi * (R_GROUND ** 2 - R_SPHERE ** 2)
    ns = int(n * a_sph / (a_sph + a_gnd))
    z = torch.rand(ns, generator=g, device=dev, dtype=torch.float64) * R_SPHERE
    phi = torch.rand(ns, generator=g, device=dev, dtype=torch.float64) * 2 * np.pi
    rho = torch.sqrt(R_SPHERE ** 2 - z * z)
    sph = torch.stack([rho * torch.cos(phi), rho * torch.sin(phi), z], 1)
    ng = n - ns
    r = torch.sqrt(torch.rand(ng, generator=g, device=dev, dtype=torch.float64) * (R_GROUND ** 2 - R_SPHERE ** 2) + R_SPHERE ** 2)
    phi = torch.rand(ng, generator=g, device=dev, dtype=torch.float64) * 2 * np.pi
    gnd = torch.stack([r * torch.cos(phi), r * torch.sin(phi), torch.zeros_like(r)], 1)
    return torch.cat([sph, gnd])


def workload(dev):
    g = torch.Generator(device=dev).manual_seed(0)
    area = 2 * np.pi * R_SPHERE ** 2 + np.pi * (R_GROUND ** 2 - R_SPHERE ** 2)
    stl = _surface(g, int(area * DENSITY), dev).float().contiguous()
    data = {}
    for name, n in (("2.1M", 2_100_000), ("10M", 10_000_000)):
        n_out = int(0.03 * n)
        pts = _surface(g, n - n_out, dev) + torch.randn(n - n_out, 3, generator=g, device=dev, dtype=torch.float64)
        lo, hi = torch.tensor(BB[0], device=dev), torch.tensor(BB[1], device=dev)
        out = lo + torch.rand(n_out, 3, generator=g, device=dev, dtype=torch.float64) * (hi - lo)
        data[name] = torch.cat([pts, out]).float().contiguous()
    shape = tuple(int(v) for v in np.floor((BB[1] - BB[0]) / RES) + 1)
    ax = [torch.arange(s, device=dev, dtype=torch.float64) * RES + BB[0, a] for a, s in enumerate(shape)]
    X, Y, Z = torch.meshgrid(*ax, indexing="ij")
    rr = torch.sqrt(X * X + Y * Y + Z * Z)
    mask = ((rr - R_SPHERE).abs() < 15) | ((Z.abs() < 15) & (rr < R_GROUND + 15))
    del X, Y, Z, rr
    return stl, data, mask


def _time(fn, reps=1):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        r = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps, r                  # ms per call


def _alternate(fns, rounds):
    for f in fns.values():
        _time(f)
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            out[k].append(_time(f)[0])
    return {k: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v)), "rounds_ms": v}
            for k, v in out.items()}


def bench_size(name, x, stl, mask, rounds):
    dev = x.device
    res = {"n_data": int(x.shape[0]), "m_stl": int(stl.shape[0])}
    # thinning: total (grid + neighbour lists + rounds + bookkeeping) and its rounds
    t_thin, (kept, n_rounds) = _time(lambda: evaluation.thin(x, evaluation.DST, seed=0))
    t_thin2, _ = _time(lambda: evaluation.thin(x, evaluation.DST, seed=0))
    q = x[kept].contiguous()
    res.update(thin_ms=[t_thin, t_thin2], thin_rounds=n_rounds, n_reduced=int(q.shape[0]))
    # grid over the ground truth at the chosen cell and at half and twice that cell, alternated; then the search on each
    cell0, nb0 = evaluation.cell_size(*(v.cpu().tolist() for v in torch.aminmax(stl, dim=0)), stl.shape[0])
    grids = {}

    def grid(c):
        def f():
            grids[c] = evaluation.build_grid(stl, cell=c)
        return f
    sizes = {"0.5x": 0.5 * cell0, "chosen": cell0, "2x": 2 * cell0}
    res["cell_mm"] = sizes
    res["grid_stl"] = _alternate({k: grid(c) for k, c in sizes.items()}, rounds)
    md = evaluation.MAX_DIST

    def search(c):
        return lambda: evaluation.nearest_distance(q, stl, md, grid=grids[c])
    res["nearest_data_to_stl"] = _alternate({k: search(c) for k, c in sizes.items()}, rounds)
    dq = evaluation.build_grid(q)
    res["grid_reduced_data"] = _alternate({"chosen": lambda: evaluation.build_grid(q)}, rounds)
    res["cell_reduced_data_mm"] = dq.cell
    res["nearest_stl_to_data"] = _alternate({"chosen": lambda: evaluation.nearest_distance(stl, q, md, grid=dq)}, rounds)
    d = [evaluation.nearest_distance(q, stl, md, grid=grids[c]) for c in sizes.values()]
    res["cell_sizes_agree_bitwise"] = bool(all(torch.equal(d[0], e) for e in d[1:]))
    res["queries_per_s"] = {"data_to_stl": q.shape[0] / res["nearest_data_to_stl"]["chosen"]["median_ms"] * 1e3,
                            "stl_to_data": stl.shape[0] / res["nearest_stl_to_data"]["chosen"]["median_ms"] * 1e3}
    # the whole call (seeded order)
    bb, plane = BB, [0.0, 0.0, 1.0, 1e-3]
    res["evaluate_point_cloud"] = _alternate({"whole": lambda: evaluation.evaluate_point_cloud(x, stl, mask, bb, RES, plane)}, rounds)
    out = evaluation.evaluate_point_cloud(x, stl, mask, bb, RES, plane)
    res["result"] = out
    # minimal bytes: what each pass must read and write once (the gathers of neighbouring points are not counted)
    n, m, k = x.shape[0], stl.shape[0], q.shape[0]
    res["bytes_min"] = {"nearest_data_to_stl": k * (12 + 4) + m * 16, "nearest_stl_to_data": m * (12 + 4) + k * 16,
                        "grid_stl": m * (12 + 4) + m * (4 + 8 + 12 + 4 + 16)}
    res["GBps_at_median"] = {"nearest_data_to_stl": res["bytes_min"]["nearest_data_to_stl"] / res["nearest_data_to_stl"]["chosen"]["median_ms"] / 1e6,
                             "nearest_stl_to_data": res["bytes_min"]["nearest_stl_to_data"] / res["nearest_stl_to_data"]["chosen"]["median_ms"] / 1e6}
    ws = n * 12 + n * 16 + m * 12 + m * 16
    res["working_set_bytes"] = ws
    res["exceeds_l2_126MB"] = bool(ws > L2_BYTES)
    return res, q


def host_refs(q, stl):
    """The numpy oracle on a subset of 200 queries (brute force against the whole ground truth), and scipy's cKDTree (all
    cores) on the whole reduced cloud in both directions when scipy is present."""
    out = {}
    qs, s = q[:200].cpu().numpy(), stl.cpu().numpy()
    t0 = time.perf_counter()
    oracle.nearest(qs, s)
    dt = time.perf_counter() - t0
    out["numpy_oracle"] = {"queries": 200, "targets": int(s.shape[0]), "s": dt, "s_per_query": dt / 200,
                           "note": "a subset, brute force; not the MATLAB scripts"}
    try:
        from scipy.spatial import cKDTree
    except ImportError:
        out["ckdtree"] = "scipy not installed: not measured"
        return out
    qa = q.cpu().numpy()
    t0 = time.perf_counter()
    ts = cKDTree(s)
    t1 = time.perf_counter()
    ts.query(qa, k=1, distance_upper_bound=evaluation.MAX_DIST, workers=-1)
    t2 = time.perf_counter()
    tq = cKDTree(qa)
    t3 = time.perf_counter()
    tq.query(s, k=1, distance_upper_bound=evaluation.MAX_DIST, workers=-1)
    t4 = time.perf_counter()
    out["ckdtree"] = {"build_stl_s": t1 - t0, "query_data_to_stl_s": t2 - t1, "build_data_s": t3 - t2, "query_stl_to_data_s": t4 - t3,
                      "workers": "all", "host_cpus": os.cpu_count()}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dtu_eval needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    dev = torch.device("cuda:0")
    stl, data, mask = workload(dev)
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None,
           "timing": "CUDA events around whole calls after a warm-up; compared forms alternate over rounds; median of rounds",
           "workload": {"bb": BB.tolist(), "res": RES, "mask_shape": list(mask.shape), "m_stl": int(stl.shape[0]),
                        "dst": evaluation.DST, "max_dist": evaluation.MAX_DIST, "block": evaluation.BLOCK}}
    q = None
    for name, x in data.items():
        res[name], q_ = bench_size(name, x, stl, mask, a.rounds)
        if q is None:
            q = q_
        print(name, json.dumps({k: v for k, v in res[name].items() if k != "result"}, default=str)[:1500], flush=True)
    res["host_2.1M"] = host_refs(q, stl)
    print("host", json.dumps(res["host_2.1M"]))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1, default=float)


if __name__ == "__main__":
    main()
