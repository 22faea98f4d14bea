"""Tanks and Temples precision, recall and F-score of one reconstructed scene (mvs_b200.evaluate_tanks_and_temples on the GPU).

    python tools/eval_tnt.py --ply Barn.ply --tnt /data/tnt --scene Barn --tau 0.01 [--out result.json]

    python tools/eval_tnt.py --ply Barn.ply --tnt /data/tnt --scene Barn --tau 0.01 --traj Barn.log [--seed 0]

    python tools/eval_tnt.py --ply Barn.ply --tnt /data/tnt --scene Barn --tau 0.01 [--register | --traj Barn.log] --write out/

--tnt is the directory of T&T's evaluation data, one sub-directory per scene with {scene}.ply, {scene}.json and {scene}_trans.txt,
and for --traj also {scene}_COLMAP_SfM.log and, for a trajectory of every video frame, {scene}_mapping_reference.txt
(INTEGRATION.md §2).  --traj runs the toolbox's whole chain: the RANSAC alignment of the reconstruction's camera trajectory (a .log
file in the reconstruction's frame) to T&T's COLMAP one mapped by {scene}_trans.txt (mvs_b200.align_trajectory, draws seeded by
--seed), then the three ICP stages from that alignment, then the evaluation; it implies --register and excludes --init.  Without
--traj the reconstruction must be in the frame of T&T's COLMAP cameras, or --init must map it near the ground truth.  --register
refines that alignment with the toolbox's three ICP stages (mvs_b200.register_tanks_and_temples) and evaluates under the refined
transform, as the toolbox does; without it {scene}_trans.txt (or --init) is used as given.  --tau is the scene's threshold (the
toolbox's table of per-scene values is not shipped).  Prints one JSON line: precision, recall, fscore, the counts, and the
histogram edges and cumulative curves; with --register also a `registration` record (the refined transform and, per stage, its
sizes, iterations, fitness, rmse and transform); with --traj also an `alignment` record (the RANSAC transform, fitness, rmse,
inliers, the winning hypothesis and its sample, the correspondence count and the seed).  --write DIR also writes the toolbox's
per-scene files into DIR (mvs_b200.write_evaluation_files): {scene}.precision.ply and {scene}.recall.ply, the down-sampled clouds
with normals and coloured by distance, and {scene}.precision.txt, {scene}.recall.txt and {scene}.prf_tau_plotstr.txt."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "deep-multiview-depth-estimation_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import mvs_b200  # noqa: E402
from mvs_b200 import tanks  # noqa: E402


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--ply", required=True, help="the reconstruction (binary little-endian or ASCII PLY)")
    ap.add_argument("--tnt", required=True, help="T&T's evaluation directory ({scene}/{scene}.ply, .json, _trans.txt)")
    ap.add_argument("--scene", required=True)
    ap.add_argument("--tau", type=float, required=True, help="the scene's distance threshold, in the ground truth's units")
    ap.add_argument("--stretch", type=float, default=tanks.STRETCH, help="the histograms span [0, stretch * tau)")
    ap.add_argument("--out", help="also write the result as JSON to this file")
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--register", action="store_true", help="refine the alignment with the toolbox's three ICP stages first")
    ap.add_argument("--init", help="a 4 x 4 text file to start from instead of {scene}_trans.txt")
    ap.add_argument("--traj", help="the reconstruction's camera trajectory (.log): align it to T&T's first (implies --register)")
    ap.add_argument("--seed", type=int, help="the seed of the alignment's RANSAC draws (with --traj; default 0)")
    ap.add_argument("--write", metavar="DIR", help="also write the toolbox's coloured precision / recall clouds and curves to DIR")
    a = ap.parse_args(argv)
    if a.traj and a.init:
        ap.error("--traj and --init exclude each other: --traj computes the initial alignment")
    if a.seed is not None and not a.traj:
        ap.error("--seed applies to --traj only")
    if a.write is not None and (not a.write or (os.path.exists(a.write) and not os.path.isdir(a.write))):
        ap.error(f"--write needs a directory, got {a.write!r}")
    xyz, _ = mvs_b200.read_ply(a.ply)
    gt, crop, trans = mvs_b200.load_tnt_eval(a.tnt, a.scene)
    if a.init:
        trans = np.loadtxt(a.init, dtype=np.float64)
    dev = torch.device(a.device)
    xyz, gt = xyz.to(dev), gt.to(dev)
    reg = align = None
    if a.traj:
        _, poses = mvs_b200.read_trajectory(a.traj)
        ref, mapping = mvs_b200.load_tnt_trajectory(a.tnt, a.scene)
        with torch.cuda.device(dev):
            align = mvs_b200.align_trajectory(poses, ref, trans, mapping=mapping, seed=a.seed or 0)
        trans = align["transformation"]
    if a.register or a.traj:
        reg = mvs_b200.register_tanks_and_temples(xyz, gt, crop, trans, a.tau)
        trans = reg["transformation"]
    r = mvs_b200.evaluate_tanks_and_temples(xyz, gt, crop, trans, a.tau, stretch=a.stretch, return_details=a.write is not None)
    if a.write is not None:
        with torch.cuda.device(dev):
            mvs_b200.write_evaluation_files(a.write, a.scene, r, stretch=a.stretch)
        for k in ("xyz_down", "gt_down", "d_s", "d_t"):
            del r[k]
    r = {"scene": a.scene, "ply": a.ply, **{k: v.tolist() if isinstance(v, np.ndarray) else v for k, v in r.items()}}
    if align is not None:
        r["alignment"] = {**{k: v.tolist() if isinstance(v, np.ndarray) else v for k, v in align.items()}, "seed": a.seed or 0}
    if reg is not None:
        r["registration"] = {"transformation": reg["transformation"].tolist(), "init": reg["init"].tolist(),
                             "stages": [{k: v.tolist() if isinstance(v, np.ndarray) else v for k, v in st.items()} for st in reg["stages"]]}
    print(json.dumps(r))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(r, f, indent=1)


if __name__ == "__main__":
    main()
