"""The Tanks and Temples trajectory alignment without a GPU: the trajectory and mapping readers and writer with their refusals, the
toolbox's mapping rule and point pairing, the fp64 oracle (oracle/tnt_align.py) recovering a planted similarity, each of its
mutation switches changing the outcome, the counter-based draws pinned to SplitMix64's published sequence, and the command-line
tool's argument rules."""
import os
import subprocess
import sys

import numpy as np
import pytest

import tnt_align as oracle
import tnt_register
import mvs_b200
from mvs_b200 import registration, tanks

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def orbit():
    return oracle.orbit_scene()


def test_trajectory_round_trip(tmp_path, orbit):
    p = str(tmp_path / "a.log")
    mvs_b200.write_trajectory(p, orbit["poses"])
    meta, poses = mvs_b200.read_trajectory(p)
    assert poses.tobytes() == orbit["poses"].tobytes()
    n = len(poses)
    assert np.array_equal(meta, np.stack([np.arange(n), np.arange(n), np.arange(1, n + 1)], 1)) and meta.dtype == np.int64
    mvs_b200.write_trajectory(p, orbit["poses"][:3], metadata=[[7, 8, 9]] * 3)
    assert mvs_b200.read_trajectory(p)[0].tolist() == [[7, 8, 9]] * 3
    # the toolbox's writer: tab- and space-separated fixed-point values, a trailing blank line
    with open(p, "w") as f:
        f.write("0 0 1\n1.000000000000 0.000000000000 0.000000000000 2.5\n0\t1 0 0\n0 0 1 -3\n0 0 0 1\n\n")
    meta, poses = mvs_b200.read_trajectory(p)
    assert meta.tolist() == [[0, 0, 1]] and poses[0, :3, 3].tolist() == [2.5, 0.0, -3.0]


@pytest.mark.parametrize("text, match", [
    ("0 0 1\n1 0 0 0\n0 1 0 0\n0 0 1 0\n", "short"),
    ("0 0 1\n1 0 0 0\n0 1 0 0\n0 0 1 0\n0 0 0 1\n0 1 2\n1 0 0 0\n", "short"),
    ("0 0 1\n1 0 0 0\n0 1 x 0\n0 0 1 0\n0 0 0 1\n", "numbers expected"),
    ("0 0 1\n1 0 0 0\n0 1 0\n0 0 1 0\n0 0 1 0\n0 0 0 1\n", "short|4 finite"),
    ("0 0 1\n1 0 0 0\n0 1 0 nan\n0 0 1 0\n0 0 0 1\n", "finite"),
    ("0 0 1.5\n1 0 0 0\n0 1 0 0\n0 0 1 0\n0 0 0 1\n", "integers"),
    ("0 0\n1 0 0 0\n0 1 0 0\n0 0 1 0\n0 0 0 1\n", "3 integers"),
    ("0 0 1\n1 0 0 0\n0 1 0 0\n0 0 1 0\n0 0 1e-9 1\n", "0 0 0 1"),
])
def test_trajectory_refusals(tmp_path, text, match):
    p = tmp_path / "bad.log"
    p.write_text(text)
    with pytest.raises(mvs_b200.MvsB200Error, match=match):
        mvs_b200.read_trajectory(str(p))


def test_mapping_reader_and_refusals(tmp_path):
    p = tmp_path / "m.txt"
    p.write_text("3\n5000\n0 11\n1 2000\n2 4999\n")
    m = mvs_b200.read_mapping(str(p))
    assert m.n_total == 5000 and m.rows.tolist() == [[0, 11], [1, 2000], [2, 4999]] and m.rows.dtype == np.int64
    for text, match in (("4\n5000\n0 11\n1 2000\n2 4999\n", "n_sampled is 4 but 3"), ("2\n5000\n0 11\n1 2000\n2 4999\n", "n_sampled"),
                        ("1\n5000\n0 1.5\n", "integers"), ("1\n5000\n0 1 2\n", "2 integers"), ("1\n", "first two lines"),
                        ("x\n5\n", "integers")):
        p.write_text(text)
        with pytest.raises(mvs_b200.MvsB200Error, match=match):
            mvs_b200.read_mapping(str(p))


def test_load_tnt_trajectory(tmp_path, orbit):
    d = tmp_path / "Synth"
    d.mkdir()
    with pytest.raises(mvs_b200.MvsB200Error, match="not found"):
        mvs_b200.load_tnt_trajectory(str(tmp_path), "Synth")
    mvs_b200.write_trajectory(str(d / "Synth_COLMAP_SfM.log"), orbit["reference"])
    ref, mapping = mvs_b200.load_tnt_trajectory(str(tmp_path), "Synth")
    assert ref.tobytes() == orbit["reference"].tobytes() and mapping is None
    (d / "Synth_mapping_reference.txt").write_text("2\n10\n0 3\n1 7\n")
    assert mvs_b200.load_tnt_trajectory(str(tmp_path), "Synth")[1].rows.tolist() == [[0, 3], [1, 7]]


def test_camera_poses_invert_the_extrinsics():
    rng = np.random.default_rng(2)
    R = oracle._rotations(rng, 5)
    T = rng.normal(size=(5, 3)) * 4
    P = mvs_b200.camera_poses(R, T)
    for k in range(5):
        E = np.eye(4)
        E[:3, :3], E[:3, 3] = R[k], T[k]
        assert np.abs(P[k] @ E - np.eye(4)).max() < 1e-12
    assert np.array_equal(P[:, 3], np.tile([0.0, 0.0, 0.0, 1.0], (5, 1)))
    assert np.array_equal(mvs_b200.camera_poses(R, T[..., None]), P)
    with pytest.raises(mvs_b200.MvsB200Error, match="R"):
        mvs_b200.camera_poses(R[:, :2], T)


def _dense(n, sparse, rng):
    """A dense trajectory of n poses whose frames 3, 6, 9, ... (1-based) are the sparse poses; every other frame is far off."""
    dense = oracle.poses_at(rng.uniform(500, 600, (n, 3)), rng)
    frames = 3 * np.arange(1, len(sparse) + 1)
    dense[frames - 1] = sparse
    return dense, np.stack([np.arange(len(sparse)), frames], 1)


def test_mapping_is_used_above_1600_poses(orbit):
    rng = np.random.default_rng(3)
    sparse, ref, G = orbit["poses"][:200], orbit["reference"][:200], orbit["gt_trans"]
    for n in (1600, 1601):
        dense, rows = _dense(n, sparse, rng)
        src, tgt = registration.trajectory_points(dense, ref, G, tanks.Mapping(n, rows))
        want = sparse[:, :3, 3] if n > 1600 else dense[:200, :3, 3]
        assert np.array_equal(src, want), n
        assert np.array_equal(tgt, oracle.points(dense, ref, G, rows)[1])
        assert np.array_equal(src, oracle.points(dense, ref, G, rows)[0])
    with pytest.raises(mvs_b200.MvsB200Error, match="mapping is needed"):
        registration.trajectory_points(dense, ref, G)
    bad = rows.copy()
    bad[5, 1] = 0
    with pytest.raises(mvs_b200.MvsB200Error, match="1-based"):
        registration.trajectory_points(dense, ref, G, bad)


def test_pairing_and_refusals(orbit):
    P, ref, G = orbit["poses"], orbit["reference"], orbit["gt_trans"]
    src, tgt = registration.trajectory_points(np.concatenate([P, P[:7]]), ref, G)      # extra poses are ignored
    assert np.array_equal(src, P[:, :3, 3])
    c = ref[:, :3, 3]
    assert np.array_equal(tgt, np.stack([((G[r, 0] * c[:, 0] + G[r, 1] * c[:, 1]) + G[r, 2] * c[:, 2]) + G[r, 3] for r in range(3)], 1))
    with pytest.raises(mvs_b200.MvsB200Error, match="needs its pair"):
        registration.trajectory_points(P[:-1], ref, G)
    with pytest.raises(mvs_b200.MvsB200Error, match="affine"):
        registration.trajectory_points(P, ref, np.ones((4, 4)))
    with pytest.raises(mvs_b200.MvsB200Error, match="finite"):
        registration.trajectory_points(P * np.nan, ref, G)
    with pytest.raises(mvs_b200.MvsB200Error, match=r"\[n, 4, 4\]"):
        registration.trajectory_points(P[:, :3], ref, G)
    for kw, match in ((dict(ransac_n=2), "ransac_n"), (dict(ransac_n=65), "ransac_n"), (dict(max_iteration=-1), "max_iteration"),
                      (dict(seed=-1), "seed"), (dict(seed=2 ** 64), "seed"), (dict(max_correspondence_distance=0.0), "max_corr")):
        with pytest.raises(mvs_b200.MvsB200Error, match=match):
            mvs_b200.align_trajectory(P, ref, G, **kw)


def test_draws_are_splitmix64():
    # SplitMix64 from state 0: its published first outputs, and the same stream for any split into hypotheses
    first = [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4, 0x06C45D188009454F, 0xF88BB8A8724C81EC]
    k = np.arange(1, 5, dtype=np.uint64)
    assert [int(v) for v in oracle.splitmix64(k * oracle.GOLDEN)] == first
    n = 2 ** 31 - 1
    assert oracle.draws(0, 1, 4, n)[0].tolist() == [v % n for v in first]
    assert np.array_equal(oracle.draws(0, 4, 6, 400)[2:], oracle.draws(0, 2, 6, 400, first=2))
    assert oracle.draws(0, 2, 6, 400).tolist() == [[335, 100, 79, 44, 347, 90], [113, 140, 99, 390, 201, 326]]
    assert not np.array_equal(oracle.draws(1, 2, 6, 400), oracle.draws(0, 2, 6, 400))


def test_oracle_recovers_a_planted_similarity(orbit):
    r = oracle.align(orbit["poses"], orbit["reference"], orbit["gt_trans"], n_hyp=3000)
    ang, sc, tr = tnt_register.similarity_error(r["transformation"], orbit["S_true"])
    print("rotation", ang, "scale", sc, "translation", tr, "inliers", r["inliers"], "hypothesis", r["hypothesis"])
    assert ang <= 1e-2 and sc <= 1e-2
    src, tgt = oracle.points(orbit["poses"], orbit["reference"], orbit["gt_trans"])
    g, _, _ = oracle.score(src, tgt, r["transformation"][None], 0.2)
    q = oracle.tnt_eval.transform(src, r["transformation"])
    inl = ((q - tgt) ** 2).sum(1) < 0.04
    assert np.array_equal(inl, ~orbit["outlier"]) and g[0] == r["inliers"] == (~orbit["outlier"]).sum()
    assert r["fitness"] == r["inliers"] / len(src)


def test_mutations_change_the_outcome(orbit):
    P, ref, G, S = orbit["poses"], orbit["reference"], orbit["gt_trans"], orbit["S_true"]
    base = oracle.align(P, ref, G, n_hyp=3000)
    for kw in (dict(apply_gt_trans=False), dict(swap=True)):
        e = tnt_register.similarity_error(oracle.align(P, ref, G, n_hyp=3000, **kw)["transformation"], S)
        print(kw, e)
        assert e[0] > 0.1 or e[1] > 0.1, kw
    fit = oracle.align(P, ref, G, n_hyp=3000, select_by="fitness")
    assert fit["inliers"] == base["inliers"] and fit["hypothesis"] < base["hypothesis"] and fit["inlier_rmse"] > base["inlier_rmse"]
    # the 0-based reading of the mapping pairs the reference with the far-off frames next to the sampled ones
    rng = np.random.default_rng(4)
    dense, rows = _dense(2000, P, rng)
    good = oracle.align(dense, ref, G, rows, n_hyp=1000)
    bad = oracle.align(dense, ref, G, rows, n_hyp=1000, mapping_base=0)
    assert good["inliers"] == base["inliers"] and bad["inliers"] < good["inliers"] / 4
    # six cameras: 6^6 = 46656 samples, so 100000 draws repeat some; exact ties go to the first
    six = oracle.orbit_scene(n=6, seed=1, outliers=0.0)
    first = oracle.align(six["poses"], six["reference"], six["gt_trans"], n_hyp=100000)
    last = oracle.align(six["poses"], six["reference"], six["gt_trans"], n_hyp=100000, tie="last")
    a, b = first["hypothesis"], last["hypothesis"]
    assert b > a and first["good"][a] == first["good"][b] and first["error2"][a] == first["error2"][b]


def test_tool_argument_rules(tmp_path):
    tool = os.path.join(ROOT, "tools", "eval_tnt.py")
    base = [sys.executable, tool, "--ply", "x.ply", "--tnt", str(tmp_path), "--scene", "S", "--tau", "0.01"]
    r = subprocess.run(base + ["--traj", "a.log", "--init", "t.txt"], capture_output=True, text=True)
    assert r.returncode == 2 and "--traj" in r.stderr and "--init" in r.stderr
    r = subprocess.run(base + ["--seed", "3"], capture_output=True, text=True)
    assert r.returncode == 2 and "--seed" in r.stderr
    r = subprocess.run([sys.executable, tool, "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--traj" in r.stdout and "--seed" in r.stdout
