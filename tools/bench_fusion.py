"""Times the K7 consistency check and compaction kernels, the fp64 oracle on the host, and K4 with / without the confidence
(CUDA events, alternating rounds) -> one JSON file.

    python tools/bench_fusion.py --out profiles/r04_bench_fusion.json

Fusion workload: 49 views with 10 sources each (DTU's view count, MVSNet's source count) of a synthetic scene
(oracle.fusion.analytic_scene plus 0.2 % depth noise) at the cfg1 depth size 128 x 160 and the cfg4 size 296 x 400.  The inputs
(depth, confidence and colour maps of 49 views, "input_bytes") fit in the 126 MB L2, so repeated launches read them from L2:
the times are L2-resident times."""
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

import fusion as oracle  # noqa: E402
from mvs_b200 import _lib, fusion  # noqa: E402
from mvs_b200.ops import _stream  # noqa: E402


def _events(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / reps            # us per call


def _alternate(fns, reps, rounds):
    for f in fns.values():
        _events(f, 5)
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            out[k].append(_events(f, reps))
    return {k: {"median_us": float(np.median(v)), "min_us": float(np.min(v)), "max_us": float(np.max(v)), "rounds_us": v}
            for k, v in out.items()}


def bench_fusion(h, w, N=49, S=10, reps=200, rounds=5):
    dev = torch.device("cuda:0")
    s = oracle.analytic_scene(N, h, w, seed=0, focal=1.5 * w)          # the disk fills most of every view, as at 64 px
    rng = np.random.default_rng(1)
    depth = (s["depth"] * (1 + 2e-3 * rng.standard_normal(s["depth"].shape))).astype(np.float32)
    conf = rng.uniform(0.5, 1.0, depth.shape).astype(np.float32)
    colours = rng.uniform(size=(N, 3, h, w)).astype(np.float32)
    src = [[(i + k) % N for k in (1, -1, 2, -2, 3, -3, 4, -4, 5, -5)] for i in range(N)]
    t = lambda a, c=1: torch.from_numpy(a).reshape(N, c, h, w).to(dev)       # noqa: E731
    d, c, col = t(depth), t(conf), t(colours, 3)
    mask, count, fused, blocks, cams = fusion._check(d, c, s["K"], s["R"], s["T"], src, "sweep", 0.8, 1.0, 0.01, 3)
    srct = torch.from_numpy(fusion.source_table(src, N)).to(dev)
    offsets = torch.cumsum(blocks, 0) - blocks
    M = int(offsets[-1] + blocks[-1])
    xyz = torch.empty((M, 3), device=dev)
    rgb = torch.empty((M, 3), device=dev)

    def check():
        _lib.call("mvsb200_fusion_check", d.data_ptr(), c.data_ptr(), cams.data_ptr(), srct.data_ptr(), N, S, h, w, 0.8, 1.0, 0.01, 3,
                  mask.data_ptr(), count.data_ptr(), fused.data_ptr(), blocks.data_ptr(), _stream())

    def emit():
        _lib.call("mvsb200_fusion_emit", mask.data_ptr(), fused.data_ptr(), col.data_ptr(), cams.data_ptr(), offsets.data_ptr(), N, h, w,
                  xyz.data_ptr(), rgb.data_ptr(), _stream())

    def whole():
        fusion.fuse_depth_maps(d, c, col, s["K"], s["R"], s["T"], src)

    times = _alternate({"check": check, "emit": emit}, reps, rounds)
    times.update(_alternate({"fuse_depth_maps_end_to_end": whole}, 20, rounds))
    px = N * h * w
    # bytes the check needs at least: depth + conf of every reference pixel read, mask + count + fused written; the source taps
    # (4 per consistent source) are re-reads of the same maps from L2 / L1
    check_bytes = px * (4 + 4 + 1 + 4 + 4)
    emit_bytes = px * (1 + 4) + M * (12 + 12 + 12)
    n_ref = 4                                             # the oracle on the first 4 reference views (others get no sources)
    src_o = [r if i < n_ref else [-1] * S for i, r in enumerate(src)]
    t0 = time.perf_counter()
    oracle.check(depth, conf, s["K"], s["R"], s["T"], src_o, "sweep")
    t_or = time.perf_counter() - t0
    return {"views": N, "sources": S, "h": h, "w": w, "points": M, "kept_fraction": M / px,
            "input_bytes": int(px * 4 * 2 + px * 12), "fits_l2_126MB": bool(px * 4 * 2 + px * 12 < 126e6), "l2_resident": True,
            "kernels": times, "check_bytes_min": check_bytes, "emit_bytes_min": emit_bytes,
            "check_GBps_at_median": check_bytes / times["check"]["median_us"] / 1e3,
            "emit_GBps_at_median": emit_bytes / times["emit"]["median_us"] / 1e3,
            "oracle_host_s_for_4_reference_views": t_or, "oracle_host_s_per_reference_view": t_or / n_ref,
            "host_cpus": os.cpu_count()}


def bench_k4(B=1, D=192, h=128, w=160, reps=200, rounds=7):
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(0)
    x = torch.randn(B, D, h, w, generator=g).to(dev)
    depths = (425.0 + 2.5 * torch.arange(D, dtype=torch.float32)).repeat(B, 1).contiguous().to(dev)
    prob = torch.empty_like(x)
    ranks = torch.empty(B, 5, h, w, dtype=torch.int32, device=dev)
    depth = torch.empty(B, h, w, device=dev)
    conf = torch.empty(B, h, w, device=dev)

    def plain():
        _lib.call("mvsb200_softmax_depth_fwd", x.data_ptr(), 1, depths.data_ptr(), prob.data_ptr(), ranks.data_ptr(), depth.data_ptr(),
                  B, D, h, w, 5, _stream())

    def with_conf():
        _lib.call("mvsb200_softmax_depth_conf_fwd", x.data_ptr(), 1, depths.data_ptr(), prob.data_ptr(), ranks.data_ptr(), depth.data_ptr(),
                  conf.data_ptr(), B, D, h, w, 5, _stream())

    def standalone():
        _lib.call("mvsb200_depth_confidence", prob.data_ptr(), depth.data_ptr(), depths.data_ptr(), conf.data_ptr(), B, D, h, w, _stream())

    r = _alternate({"softmax_depth_fwd": plain, "softmax_depth_conf_fwd": with_conf, "depth_confidence_standalone": standalone}, reps, rounds)
    return {"B": B, "D": D, "h": h, "w": w, "kernels": r}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fusion needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None,
           "timing": "CUDA events around `reps` back-to-back launches, rounds alternate between the compared forms; median of rounds",
           "fusion_cfg1": bench_fusion(128, 160), "fusion_cfg4": bench_fusion(296, 400), "k4_cfg1": bench_k4()}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v["kernels"] if isinstance(v, dict) and "kernels" in v else v) for k, v in res.items()}, default=str)[:3000])


if __name__ == "__main__":
    main()
