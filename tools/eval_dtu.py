"""DTU accuracy / completeness of one reconstructed scan (mvs_b200.evaluate_point_cloud on the GPU).

    python tools/eval_dtu.py --ply scan1.ply --dtu /data/dtu_eval --scan 1 [--out result.json]

--dtu is the directory of DTU's evaluation data: Points/stl/stl{scan:03d}_total.ply, ObsMask/ObsMask{scan}_10.mat and
ObsMask/Plane{scan}.mat (INTEGRATION.md §2).  Prints one JSON line: accuracy, completeness, overall (mm), the medians and counts."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "deep-multiview-depth-estimation_b200"))

import torch  # noqa: E402

import mvs_b200  # noqa: E402
from mvs_b200 import evaluation  # noqa: E402


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--ply", required=True, help="the reconstruction (binary little-endian or ASCII PLY)")
    ap.add_argument("--dtu", required=True, help="DTU's evaluation directory (Points/stl, ObsMask)")
    ap.add_argument("--scan", type=int, required=True)
    ap.add_argument("--out", help="also write the result as JSON to this file")
    ap.add_argument("--dst", type=float, default=evaluation.DST)
    ap.add_argument("--max-dist", type=float, default=evaluation.MAX_DIST)
    ap.add_argument("--block", type=float, default=evaluation.BLOCK)
    ap.add_argument("--seed", type=int, default=0, help="seed of the thinning's visiting order (a CPU torch.Generator)")
    ap.add_argument("--device", default="cuda:0")
    a = ap.parse_args(argv)
    xyz, _ = mvs_b200.read_ply(a.ply)
    stl, obs_mask, bb, res, plane = mvs_b200.load_dtu_eval(a.dtu, a.scan)
    dev = torch.device(a.device)
    r = mvs_b200.evaluate_point_cloud(xyz.to(dev), stl.to(dev), obs_mask, bb, res, plane, dst=a.dst, max_dist=a.max_dist,
                                      block=a.block, seed=a.seed)
    r = {"scan": a.scan, "ply": a.ply, **r}
    print(json.dumps(r))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(r, f, indent=1)


if __name__ == "__main__":
    main()
