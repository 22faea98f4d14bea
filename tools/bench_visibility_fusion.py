"""Times visibility fusion against K7's fusion on bench_fusion's workload (CUDA events, alternating rounds) -> one JSON file.

    python tools/bench_visibility_fusion.py --out profiles/r06_bench_visibility_fusion.json

Workload: exactly tools/bench_fusion.py's.  49 views (DTU's view count), each with the ring of sources i+-1 ... i+-5 (MVSNet's 10),
of a synthetic scene (oracle.fusion.analytic_scene plus 0.2 % depth noise) at the cfg1 depth size 128 x 160 and the cfg4 size
296 x 400, views in index order.  The inputs fit in the 126 MB L2, so repeated calls read them from L2: the times are L2-resident
times.  Recorded per size: the whole visibility_fusion and fuse_depth_maps calls (alternated); the N = 49 per-view check launches
of visibility_fusion back to back, timed from before the first to after the last (the used state is zeroed outside the window),
alternated with K7's single check launch over all views; and the points each function emits."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "deep-multiview-depth-estimation_b200"), os.path.join(ROOT, "oracle"), os.path.dirname(__file__)]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import fusion as oracle  # noqa: E402
from bench_fusion import _alternate  # noqa: E402
from mvs_b200 import _lib, fusion  # noqa: E402
from mvs_b200.ops import _stream  # noqa: E402


def _stats(v):
    return {"median_us": float(np.median(v)), "min_us": float(np.min(v)), "max_us": float(np.max(v)), "rounds_us": v}


def bench(h, w, N=49, S=10, reps=20, rounds=7):
    dev = torch.device("cuda:0")
    s = oracle.analytic_scene(N, h, w, seed=0, focal=1.5 * w)          # bench_fusion's scene, inputs and sources
    rng = np.random.default_rng(1)
    depth = (s["depth"] * (1 + 2e-3 * rng.standard_normal(s["depth"].shape))).astype(np.float32)
    conf = rng.uniform(0.5, 1.0, depth.shape).astype(np.float32)
    colours = rng.uniform(size=(N, 3, h, w)).astype(np.float32)
    src = [[(i + k) % N for k in (1, -1, 2, -2, 3, -3, 4, -4, 5, -5)] for i in range(N)]
    t = lambda a, c=1: torch.from_numpy(a).reshape(N, c, h, w).to(dev)       # noqa: E731
    d, c, col = t(depth), t(conf), t(colours, 3)
    cam = (s["K"], s["R"], s["T"])

    whole = _alternate({"visibility_fusion": lambda: fusion.visibility_fusion(d, c, col, *cam, src),
                        "fuse_depth_maps": lambda: fusion.fuse_depth_maps(d, c, col, *cam, src)}, reps, rounds)

    dd, cc, cams, srct, mask, count, fused, blocks = fusion._prepare(d, c, *cam, src, "sweep")
    used = torch.zeros((N, h, w), dtype=torch.uint8, device=dev)

    def checks_vis():
        for r in range(N):
            _lib.call("mvsb200_fusion_visibility", dd.data_ptr(), cc.data_ptr(), cams.data_ptr(), srct.data_ptr(), N, S, h, w, 0.8, 1.0,
                      0.01, 3, r, used.data_ptr(), mask.data_ptr(), count.data_ptr(), fused.data_ptr(), blocks.data_ptr(), _stream())

    def check_k7():
        _lib.call("mvsb200_fusion_check", dd.data_ptr(), cc.data_ptr(), cams.data_ptr(), srct.data_ptr(), N, S, h, w, 0.8, 1.0, 0.01, 3,
                  mask.data_ptr(), count.data_ptr(), fused.data_ptr(), blocks.data_ptr(), _stream())

    def timed(fn):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in ev:
            used.zero_()
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        return float(np.mean([a.elapsed_time(b) for a, b in ev])) * 1e3

    timed(checks_vis), timed(check_k7)                                 # warm-up
    rec = {"visibility_checks_49_launches": [], "k7_check_1_launch": []}
    for _ in range(rounds):
        rec["visibility_checks_49_launches"].append(timed(checks_vis))
        rec["k7_check_1_launch"].append(timed(check_k7))
    checks = {k: _stats(v) for k, v in rec.items()}

    pts_v = fusion.visibility_fusion(d, c, col, *cam, src)[0].shape[0]
    pts_k = fusion.fuse_depth_maps(d, c, col, *cam, src)[0].shape[0]
    px = N * h * w
    return {"views": N, "sources": S, "h": h, "w": w, "order": "index", "ctas_per_view_launch": -(-h * w // 128),
            "points_visibility_fusion": pts_v, "points_fuse_depth_maps": pts_k, "point_ratio": pts_v / pts_k,
            "input_bytes": int(px * 4 * 2 + px * 12), "fits_l2_126MB": bool(px * 4 * 2 + px * 12 < 126e6), "l2_resident": True,
            "whole_call": whole, "checks": checks,
            "per_view_check_us_at_median": checks["visibility_checks_49_launches"]["median_us"] / N}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_visibility_fusion needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None,
           "timing": "CUDA events; whole calls: `reps` back-to-back calls per round, the two functions alternating; checks: one event "
                     "pair per pass, mean over `reps` passes per round, alternating; median and range of the rounds",
           "cfg1": bench(128, 160), "cfg4": bench(296, 400)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: ({q: res[k][q] for q in ("points_visibility_fusion", "points_fuse_depth_maps", "per_view_check_us_at_median")}
                          | {"whole": {n: v["median_us"] for n, v in res[k]["whole_call"].items()},
                             "checks": {n: v["median_us"] for n, v in res[k]["checks"].items()}}
                          if k.startswith("cfg") else res[k]) for k in res}, default=str))


if __name__ == "__main__":
    main()
