"""The Tanks and Temples trajectory alignment (K9 trajectory alignment: csrc/pointcloud.cu, mvs_b200/registration.py) on the GPU
against the fp64 oracle (oracle/tnt_align.py): the draws bit for bit, every hypothesis's transform and inlier count, the selection
and its tie rule, determinism and seeds, empty and degenerate inputs, the whole chain alignment -> registration -> evaluation from
fused depth maps in a far-off frame, and the command-line tool."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import fusion as fusion_oracle
import tnt_align as oracle
import tnt_eval
import tnt_register
import mvs_b200
from mvs_b200 import tanks

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_HYP = 20000


@pytest.fixture(scope="module")
def orbit():
    sc = oracle.orbit_scene()
    want = oracle.align(sc["poses"], sc["reference"], sc["gt_trans"], n_hyp=N_HYP)
    got = mvs_b200.align_trajectory(sc["poses"], sc["reference"], sc["gt_trans"], max_iteration=N_HYP, return_details=True)
    return sc, want, got


def test_draws_equal_the_oracle(orbit):
    sc, want, got = orbit
    assert got["samples"].dtype == torch.int32
    assert np.array_equal(got["samples"].cpu().numpy(), want["draws"])
    # a seed near 2^64 wraps the counter the same way on both sides
    r = mvs_b200.align_trajectory(sc["poses"], sc["reference"], sc["gt_trans"], max_iteration=500, seed=2 ** 64 - 5, return_details=True)
    assert np.array_equal(r["samples"].cpu().numpy(), oracle.draws(2 ** 64 - 5, 500, 6, len(sc["poses"])))


def test_every_hypothesis_against_the_oracle(orbit):
    sc, want, got = orbit
    T = got["transforms"].cpu().numpy()
    good, error2 = got["good"].cpu().numpy(), got["error2"].cpu().numpy()
    solved = ~np.isnan(want["transforms"][:, 0, 0])
    assert np.array_equal(~np.isnan(T).any((1, 2)), solved)
    assert (good[~solved] == 0).all() and (error2[~solved] == 0).all()
    cond = want["cond"] >= 1e-3
    ref = want["transforms"][:, :3]
    rel = np.abs(T - ref).max((1, 2)) / np.abs(ref).max((1, 2))
    print("hypotheses", N_HYP, "solved", int(solved.sum()), "conditioned", int(cond.sum()), "max rel transform error",
          float(rel[cond].max()))
    assert cond.sum() > 0.9 * N_HYP and (rel[cond] <= 1e-9).all()
    sure = want["margin"] >= 1e-6
    same = good == want["good"]
    print("margin >= 1e-6", int(sure.sum()), "good equal", int(same.sum()), "unequal with margin", int((~same & sure).sum()))
    assert same[sure].all()
    assert same.mean() >= 0.999
    both = same & solved
    assert (np.abs(error2[both] - want["error2"][both]) <= 1e-9 * np.maximum(want["error2"][both], 1e-300)).all()


def test_selection_against_the_oracle(orbit):
    sc, want, got = orbit
    h, hw = got["hypothesis"], want["hypothesis"]
    print("gpu", h, got["inliers"], got["inlier_rmse"], "oracle", hw, want["inliers"], want["inlier_rmse"], "gap", want["gap"])
    if want["gap"] >= 1e-6:
        assert h == hw
    else:
        assert got["inliers"] == want["inliers"] and abs(got["inlier_rmse"] - want["inlier_rmse"]) <= 1e-9 * want["inlier_rmse"]
    good, error2 = got["good"].cpu().numpy(), got["error2"].cpu().numpy()
    assert h == oracle.select(good, error2)                        # the rule on the kernel's own scores
    assert got["inliers"] == good[h] and got["fitness"] == good[h] / len(sc["poses"])
    assert got["inlier_rmse"] == math.sqrt(error2[h] / good[h])
    assert got["sample"] == want["draws"][h].tolist() and got["n_correspondences"] == len(sc["poses"])
    T = np.eye(4)
    T[:3] = got["transforms"][h].cpu().numpy()
    assert got["transformation"].tobytes() == T.tobytes()             # the matrix the kernel scored
    ang, sc_err, _ = tnt_register.similarity_error(got["transformation"], sc["S_true"])
    assert ang <= 1e-2 and sc_err <= 1e-2 and got["inliers"] == (~sc["outlier"]).sum()


def test_six_cameras_ties_go_to_the_first():
    six = oracle.orbit_scene(n=6, seed=1, outliers=0.0)
    got = mvs_b200.align_trajectory(six["poses"], six["reference"], six["gt_trans"], return_details=True)
    good, error2 = got["good"].cpu().numpy(), got["error2"].cpu().numpy()
    s = got["samples"].cpu().numpy()
    h = got["hypothesis"]
    tied = np.flatnonzero((good == good[h]) & (error2 == error2[h]))
    repeats = np.flatnonzero((s == s[h]).all(1))
    print("winner", h, "exactly tied", len(tied), "identical draws", len(repeats))
    assert len(repeats) > 1 and tied[0] == h and len(tied) > 1
    assert h == oracle.select(good, error2) and oracle.select(good, error2, tie="last") == tied[-1] > h
    T = got["transforms"].cpu().numpy()
    assert all(T[k].tobytes() == T[h].tobytes() for k in repeats)     # identical draws, identical bits
    want = oracle.align(six["poses"], six["reference"], six["gt_trans"])
    assert want["hypothesis"] == np.flatnonzero((want["good"] == want["good"][want["hypothesis"]])
                                                & (want["error2"] == want["error2"][want["hypothesis"]]))[0]


def test_two_runs_and_another_seed(orbit):
    sc, _, got = orbit
    again = mvs_b200.align_trajectory(sc["poses"], sc["reference"], sc["gt_trans"], max_iteration=N_HYP, return_details=True)
    for k in ("good", "error2", "transforms", "samples"):
        assert again[k].cpu().numpy().tobytes() == got[k].cpu().numpy().tobytes(), k
    assert again["transformation"].tobytes() == got["transformation"].tobytes()
    other = mvs_b200.align_trajectory(sc["poses"], sc["reference"], sc["gt_trans"], seed=7)
    ang, s_err, tr = tnt_register.similarity_error(other["transformation"], sc["S_true"])
    print("seed 7", other["hypothesis"], ang, s_err, tr)
    assert other["hypothesis"] != got["hypothesis"] and ang <= 1e-2 and s_err <= 1e-2 and other["inliers"] == got["inliers"]


def test_empty_degenerate_and_refusals(orbit):
    sc = orbit[0]
    P, ref, G = sc["poses"], sc["reference"], sc["gt_trans"]
    none = mvs_b200.align_trajectory(P, ref[:0], G, return_details=True)
    assert np.array_equal(none["transformation"], np.eye(4)) and none["hypothesis"] == -1 and none["n_correspondences"] == 0
    assert int(none["good"].abs().sum()) == 0 and none["fitness"] == 0 and none["inlier_rmse"] == 0
    zero = mvs_b200.align_trajectory(P, ref, G, max_iteration=0)
    assert zero["hypothesis"] == -1 and np.array_equal(zero["transformation"], np.eye(4))
    # two pairs: no draw holds 3 distinct indices
    two = mvs_b200.align_trajectory(P[:2], ref[:2], G, max_iteration=1000, return_details=True)
    assert two["hypothesis"] == -1 and int(two["good"].abs().sum()) == 0 and bool(torch.isnan(two["transforms"]).all())
    # every centre to register the same point: zero source variance, Eigen's 0 / 0 scale, no inlier
    same = P.copy()
    same[:, :3, 3] = 1.0
    r = mvs_b200.align_trajectory(same, ref, G, max_iteration=1000, return_details=True)
    assert r["hypothesis"] == -1 and int(r["good"].abs().sum()) == 0
    with pytest.raises(mvs_b200.MvsB200Error, match="needs its pair"):
        mvs_b200.align_trajectory(P[:10], ref, G)
    with pytest.raises(mvs_b200.MvsB200Error, match="mapping is needed"):
        mvs_b200.align_trajectory(np.concatenate([P] * 5), ref, G)
    lib = mvs_b200.load_library()
    assert lib.mvsb200_pc_ransac_align(None, None, 1, 1, 6, 0.04, 1, 0, None, None, None, None, None, None) == -1
    x = torch.zeros((8, 3), dtype=torch.float64, device=DEV)
    g, e, t, rec = (torch.zeros(n, dtype=d, device=DEV) for n, d in ((1, torch.int32), (1, torch.float64), (12, torch.float64),
                                                                       (80, torch.float64)))
    for args, msg in (((8, 1, 2, 0.04), b"ransac_n"), ((8, 1, 65, 0.04), b"ransac_n"), ((8, 1, 6, 0.0), b"max_dist2"),
                      ((0, 1, 6, 0.04), b"correspondences"), ((8, 0, 6, 0.04), b"hypotheses")):
        assert lib.mvsb200_pc_ransac_align(x.data_ptr(), x.data_ptr(), *args, 1, 0, g.data_ptr(), e.data_ptr(), t.data_ptr(), None,
                                           rec.data_ptr(), None) == -1
        assert msg in lib.mvsb200_last_error()


# the fused-disk scene of tests/test_gpu_tnt_register.py: one disk and its GT lattice on three planes 70-120 degrees apart
PLACEMENTS = (([1.0, 0.0, 0.0], 0.0, [0.0, 0.0, 0.0]), ([1.0, 0.2, 0.0], 80.0, [9.0, 1.0, 2.0]), ([0.1, 1.0, 0.3], -75.0, [2.0, 9.0, -1.5]))


def _placements(centre):
    out = []
    for ax, deg, o in PLACEMENTS:
        Q = tnt_register.rotation(ax, deg) if deg else np.eye(3)
        out.append(tnt_register.similarity(Q, 1.0, np.asarray(o) - Q @ centre))
    return out


def _place(x, centre):
    return np.concatenate([tnt_eval.transform(x, P) for P in _placements(centre)])


@pytest.fixture(scope="module")
def far_scene():
    s = fusion_oracle.analytic_scene(6, 48, 64, normal="sweep", seed=0)
    depth = torch.from_numpy(s["depth"].astype(np.float32))[:, None].to(DEV)
    src = [[j for j in range(6) if j != i] for i in range(6)]
    xyz, _, _ = mvs_b200.fuse_depth_maps(depth, torch.ones_like(depth), torch.rand(6, 3, 48, 64, device=DEV), s["K"], s["R"], s["T"],
                                         src, conf_min=0.0, reproj_px=1e3, rel_depth=1.0, min_views=1)
    r, n0, centre = s["radius"], s["n0"], s["centre"]
    a0 = np.cross(n0, [0.0, 1.0, 0.0])
    a0 /= np.linalg.norm(a0)
    b0 = np.cross(n0, a0)
    colmap = _place(xyz.double().cpu().numpy(), centre)                   # the reconstruction in T&T's COLMAP frame
    step = 0.01 * r
    k = np.arange(-int(r / step) - 1, int(r / step) + 2) * step
    u, v = (a.ravel() for a in np.meshgrid(k, k, indexing="ij"))
    on = u * u + v * v <= r * r
    A = tnt_register.similarity(tnt_register.rotation([0.3, 1.0, -0.5], 40.0), 1.7, [3.0, -1.0, 2.0])      # _trans.txt
    gt = tnt_eval.transform(_place(centre + u[on, None] * a0 + v[on, None] * b0, centre), A).astype(np.float32)
    lo, hi = gt.min(0) - 1, gt.max(0) + 1
    crop = tanks._crop_volume("y", lo[1], hi[1], [[lo[0], 0, lo[2]], [hi[0], 0, lo[2]], [hi[0], 0, hi[2]], [lo[0], 0, hi[2]]])
    tau = 0.05 * 1.7 * r / 4
    # the user's own frame: a large rotation, scale 0.6 and a far shift
    W = tnt_register.similarity(tnt_register.rotation([0.7, -0.2, 0.4], 150.0), 0.6, [300.0, -120.0, 80.0])
    rec = tnt_eval.transform(colmap, W).astype(np.float32)
    cams = mvs_b200.camera_poses(s["R"], s["T"])
    ref = np.concatenate([P @ cams for P in _placements(centre)])        # T&T's COLMAP trajectory
    user = W @ ref
    user[:, :3, :3] /= 0.6                                                # camera-to-world poses of the user's frame
    return {"rec": rec, "gt": gt, "crop": crop, "tau": tau, "A": A, "W": W, "ref": ref, "user": user}


def test_end_to_end_from_a_far_off_frame(far_scene):
    f = far_scene
    xg, gg = torch.from_numpy(f["rec"]).to(DEV), torch.from_numpy(f["gt"]).to(DEV)
    exact = f["A"] @ np.linalg.inv(f["W"])
    f_exact = mvs_b200.evaluate_tanks_and_temples(xg, gg, f["crop"], exact, f["tau"])["fscore"]
    f_trans = mvs_b200.evaluate_tanks_and_temples(xg, gg, f["crop"], f["A"], f["tau"])["fscore"]
    al = mvs_b200.align_trajectory(f["user"], f["ref"], f["A"])
    reg = mvs_b200.register_tanks_and_temples(xg, gg, f["crop"], al["transformation"], f["tau"])
    f_reg = mvs_b200.evaluate_tanks_and_temples(xg, gg, f["crop"], reg["transformation"], f["tau"])["fscore"]
    print("alignment", al["hypothesis"], al["inliers"], al["inlier_rmse"], tnt_register.similarity_error(al["transformation"], exact),
          "fscore exact", f_exact, "trans only", f_trans, "aligned + registered", f_reg)
    assert al["inliers"] == len(f["ref"]) == 18
    assert abs(f_reg - f_exact) <= 0.01 and f_trans <= 0.02


def test_eval_tnt_tool_with_traj(tmp_path, far_scene):
    f = far_scene
    d = tmp_path / "Synth"
    d.mkdir()
    mvs_b200.write_ply(str(d / "Synth.ply"), f["gt"])
    axis, amin, amax, poly = f["crop"]
    with open(d / "Synth.json", "w") as fh:
        json.dump({"class_name": "SelectionPolygonVolume", "orthogonal_axis": axis, "axis_min": amin, "axis_max": amax,
                   "bounding_polygon": poly.tolist(), "version_major": 1, "version_minor": 0}, fh)
    np.savetxt(str(d / "Synth_trans.txt"), f["A"], fmt="%.17g")
    mvs_b200.write_trajectory(str(d / "Synth_COLMAP_SfM.log"), f["ref"])
    traj = str(tmp_path / "rec.log")
    mvs_b200.write_trajectory(traj, f["user"])
    ply = str(tmp_path / "rec.ply")
    mvs_b200.write_ply(ply, f["rec"])
    out = str(tmp_path / "r.json")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "eval_tnt.py"), "--ply", ply, "--tnt", str(tmp_path), "--scene",
                        "Synth", "--tau", str(f["tau"]), "--traj", traj, "--seed", "3", "--out", out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = json.load(open(out))
    assert json.loads(r.stdout.strip().splitlines()[-1]) == got
    al = mvs_b200.align_trajectory(mvs_b200.read_trajectory(traj)[1], f["ref"], f["A"], seed=3)
    assert np.array_equal(np.array(got["alignment"]["transformation"]), al["transformation"]) and got["alignment"]["seed"] == 3
    assert got["alignment"]["hypothesis"] == al["hypothesis"] and got["alignment"]["inliers"] == 18
    assert np.array_equal(np.array(got["registration"]["init"]), al["transformation"]) and len(got["registration"]["stages"]) == 3
    xg, gg = torch.from_numpy(f["rec"]).to(DEV), torch.from_numpy(f["gt"]).to(DEV)
    reg = mvs_b200.register_tanks_and_temples(xg, gg, f["crop"], al["transformation"], f["tau"])
    assert got["fscore"] == mvs_b200.evaluate_tanks_and_temples(xg, gg, f["crop"], reg["transformation"], f["tau"])["fscore"]
    assert got["fscore"] > 0.5
