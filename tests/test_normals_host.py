"""K10 on the host: the normals oracle (oracle/pc_normals.py) against analytic normals and under its mutations, the hot_r table,
write_ply with normals, the Tanks and Temples curve files, the C ABI's refusals and eval_tnt.py's --write rule (no GPU needed)."""
import ctypes
import math
import os
import struct
import sys

import numpy as np
import pytest

import mvs_b200
from mvs_b200 import _lib, tanks

pytest.importorskip("scipy.spatial")
import pc_normals as oracle  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lattice_plane():
    """Integer points i (2, -1, 0) + j (2, 0, -1) of the plane x + 2y + 2z = 0, exact in fp32; normal (1, 2, 2) / 3."""
    i, j = (a.ravel() for a in np.meshgrid(np.arange(-4, 5), np.arange(-4, 5), indexing="ij"))
    return (i[:, None] * np.array([2, -1, 0]) + j[:, None] * np.array([2, 0, -1])).astype(np.float32), np.array([1.0, 2.0, 2.0]) / 3


def test_oracle_normals_are_analytic_on_noise_free_surfaces():
    p, want = _lattice_plane()
    got = oracle.normals(p, 12)
    assert (got["count"] == 12).all()
    assert oracle.angle(got["normal"], np.tile(want, (len(p), 1))).max() < 1e-9
    assert np.allclose(got["normal"], want, atol=1e-12)             # canonical sign: y and z tie at 2/3, y (first) is positive
    # sphere of radius 5: the pole and a symmetric ring (3, 0, 4), ... -> the radial normal at the pole
    sph = np.array([[0, 0, 5], [3, 0, 4], [-3, 0, 4], [0, 3, 4], [0, -3, 4]], np.float32)
    got = oracle.normals(sph, 5)
    assert oracle.angle(got["normal"][:1], [[0.0, 0.0, 1.0]])[0] < 1e-9 and got["normal"][0, 2] > 0
    # cylinder x^2 + y^2 = 25: (5, 0, 0) and its symmetric neighbours (4, +-3, .), (5, 0, +-1) -> the radial normal (1, 0, 0)
    cyl = np.array([[5, 0, 0], [4, 3, 0], [4, -3, 0], [5, 0, 1], [5, 0, -1], [4, 3, 1], [4, -3, 1], [4, 3, -1], [4, -3, -1]], np.float32)
    got = oracle.normals(cyl, 9)
    assert oracle.angle(got["normal"][:1], [[1.0, 0.0, 0.0]])[0] < 1e-9 and got["normal"][0, 0] > 0


def test_oracle_zero_normals_below_three_neighbours_and_for_coincident_points():
    p = np.array([[0, 0, 0], [1, 0, 0], [5, 5, 5], [5, 5, 5], [5, 5, 5]], np.float32)
    got = oracle.normals(p, 3, max_dist=2.0)
    assert (got["count"][:2] == 2).all() and (got["normal"][:2] == 0).all()        # capped: 2 neighbours
    assert (got["count"][2:] == 3).all() and (got["normal"][2:] == 0).all()        # trace 0


def test_mutation_exclude_self():
    rng = np.random.default_rng(0)
    p, _ = oracle.surface("plane", 200, rng)
    a, _, _ = oracle.knn(p, p, 5)
    b, _, _ = oracle.knn(p, p, 5, exclude_self=True)
    assert (a[:, 0] == np.arange(len(p))).all() and not (b == np.arange(len(p))[:, None]).any()


def test_mutation_ties_larger():
    g = np.stack(np.meshgrid(*[np.arange(-2, 3)] * 3, indexing="ij"), -1).reshape(-1, 3).astype(np.float32)
    q = np.zeros((1, 3), np.float32)
    # the centre, then 6 points at d^2 = 1: k = 4 cuts that tie group, and the smaller rows win
    a, d, _ = oracle.knn(q, g, 4)
    b, _, _ = oracle.knn(q, g, 4, ties_larger=True)
    ones = np.nonzero(oracle.d2_fp32(q, g) == 1)[0]
    assert list(a[0, 1:]) == sorted(ones)[:3] and list(b[0, 1:]) == sorted(ones)[::-1][:3] and d[0, 0] == 0


def test_mutation_cumulant_at_1e4():
    rng = np.random.default_rng(1)
    p, want = oracle.surface("plane", 400, rng, scale=0.05, offset=(1e4, -1e4, 1e4))
    good = oracle.normals(p, 20)
    bad = oracle.normals(p, 20, cumulant=True)
    ok = good["count"] >= 3
    assert np.median(oracle.angle(good["normal"][ok], want[ok])) < 1e-3
    with np.errstate(invalid="ignore"):                              # the cancelled cumulants leave zero normals too
        wrong = np.nan_to_num(oracle.angle(bad["normal"][ok], want[ok]), nan=np.pi / 2)
    assert np.median(wrong) > 0.1


def test_mutation_flip_on_zero_dot():
    i, j = (a.ravel() for a in np.meshgrid(np.arange(-4, 5), np.arange(-4, 5), indexing="ij"))
    p = np.c_[i, j, np.zeros_like(i)].astype(np.float32)
    v = np.array([10.0, 3.0, 0.0])                                  # in the plane z = 0: n . (v - p) = 0 exactly
    good = oracle.normals(p, 12, viewpoints=v)
    bad = oracle.normals(p, 12, viewpoints=v, flip_le=True)
    assert (good["orient"] == 0).all()
    assert (good["normal"] == [0.0, 0.0, 1.0]).all() and (bad["normal"] == [0.0, 0.0, -1.0]).all()


def test_mutation_canonical_on_the_smallest_component():
    # the plane with normal (-1, 2, 6) / sqrt(41): the largest component (z) is positive, the smallest (x) negative
    i, j = (a.ravel() for a in np.meshgrid(np.arange(-3, 4), np.arange(-3, 4), indexing="ij"))
    p = (i[:, None] * np.array([2, 1, 0]) + j[:, None] * np.array([6, 0, 1])).astype(np.float32)
    want = np.array([-1.0, 2.0, 6.0]) / math.sqrt(41)
    good = oracle.normals(p, 10)
    bad = oracle.normals(p, 10, canon_smallest=True)
    assert np.allclose(good["normal"], want, atol=1e-9) and np.allclose(bad["normal"], -want, atol=1e-9)


def test_hot_r_table_knots_and_index_rule():
    t = tanks.hot_r_table()
    assert t.shape == (256, 3) and np.array_equal(t[0], [1.0, 1.0, 1.0]) and np.allclose(t[-1], [0.0416, 0.0, 0.0])
    hot = t[::-1]
    i = np.arange(256)
    # the segments: red 0.0416 -> 1 over [0, 0.365079], green 0 -> 1 over [0.365079, 0.746032], blue 0 -> 1 over [0.746032, 1]
    assert np.allclose(hot[:, 0], np.minimum(0.0416 + (1 - 0.0416) * i / (0.365079 * 255), 1.0), atol=1e-12)
    assert np.allclose(hot[:, 1], np.clip((i - 0.365079 * 255) / ((0.746032 - 0.365079) * 255), 0, 1), atol=1e-12)
    assert np.allclose(hot[:, 2], np.clip((i - 0.746032 * 255) / ((1 - 0.746032) * 255), 0, 1), atol=1e-12)
    assert hot[93, 0] < 1.0 and hot[94, 0] == 1.0 and hot[190, 1] < 1.0 and hot[191, 1] == 1.0
    # matplotlib's index rule: int(x * 256), 1.0 -> 255; a rounding rule moves x = 128.6 / 256 to another row
    x = np.array([0.0, 1.0, 0.5, 128.6 / 256, 255.99 / 256])
    assert np.array_equal(tanks.hot_r(x), t[[0, 255, 128, 128, 255]])
    assert not np.array_equal(t[128], t[int(np.rint(128.6))])
    # distances: +inf and anything >= 3 tau take the last row
    assert np.array_equal(tanks.distance_colours([0.0, 0.03, np.inf, 0.015], 0.01), t[[0, 255, 255, 128]])


def test_write_ply_with_normals_and_unchanged_without(tmp_path):
    xyz = np.array([[1.0, 2.0, 3.0], [-1.5, 0.25, 8.0]], np.float32)
    rgb = np.array([[0.0, 0.5, 1.0], [1.0, 0.2, 0.0]])
    nrm = np.array([[0.0, 0.0, 1.0], [0.6, -0.8, 0.0]], np.float32)
    mvs_b200.write_ply(str(tmp_path / "a.ply"), xyz, rgb)
    head = b"ply\nformat binary_little_endian 1.0\nelement vertex 2\n"
    c8 = [[0, 128, 255], [255, 51, 0]]
    want = head + b"property float x\nproperty float y\nproperty float z\nproperty uchar red\nproperty uchar green\nproperty uchar blue\n" \
        b"end_header\n" + b"".join(struct.pack("<3f3B", *p, *c) for p, c in zip(xyz.tolist(), c8))
    assert (tmp_path / "a.ply").read_bytes() == want
    mvs_b200.write_ply(str(tmp_path / "b.ply"), xyz, rgb, normals=nrm)
    want = head + b"property float x\nproperty float y\nproperty float z\nproperty float nx\nproperty float ny\nproperty float nz\n" \
        b"property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n" + \
        b"".join(struct.pack("<6f3B", *p, *n, *c) for p, n, c in zip(xyz.tolist(), nrm.tolist(), c8))
    assert (tmp_path / "b.ply").read_bytes() == want
    got_xyz, got_rgb = mvs_b200.read_ply(str(tmp_path / "b.ply"))
    assert np.array_equal(got_xyz.numpy(), xyz) and got_rgb.numpy().tolist() == c8
    with pytest.raises(mvs_b200.MvsB200Error, match="normals"):
        mvs_b200.write_ply(str(tmp_path / "c.ply"), xyz, normals=nrm[:1])


def test_curve_files(tmp_path):
    r = {"precision": 0.75, "recall": 0.5, "fscore": 0.6, "tau": 0.01, "cum_precision": np.array([0.1, 0.5, 0.75]),
         "cum_recall": np.array([0.2, 0.3, 0.5])}
    paths = tanks.write_curves(str(tmp_path), "Barn", r)
    assert [os.path.basename(p) for p in paths] == ["Barn.precision.txt", "Barn.recall.txt", "Barn.prf_tau_plotstr.txt"]
    assert np.array_equal(np.loadtxt(paths[0]), r["cum_precision"]) and np.array_equal(np.loadtxt(paths[1]), r["cum_recall"])
    assert np.array_equal(np.loadtxt(paths[2]), [0.75, 0.5, 0.6, 0.01, 5.0])
    with pytest.raises(mvs_b200.MvsB200Error, match="return_details"):
        mvs_b200.write_evaluation_files(str(tmp_path), "Barn", r)


def test_c_abi_refuses_k_and_view_mode():
    lib = mvs_b200.load_library()
    p = ctypes.c_void_p(256)
    args = [p, 0, p, p, p, 0.0, 0.0, 0.0, 1.0, 1, 1, 1, 0.0, math.inf]
    for k in (0, 33):
        assert lib.mvsb200_pc_knn(*args, k, p, p, None) == -1 and b"1 <= k <= 32" in lib.mvsb200_last_error()
        assert lib.mvsb200_pc_normals(*args, k, None, 0, p, None) == -1
    assert lib.mvsb200_pc_knn(*args, 32, p, p, None) == 0                               # n = 0: nothing to launch
    assert lib.mvsb200_pc_normals(*args, 20, None, 1, p, None) == -1 and b"viewpoints" in lib.mvsb200_last_error()
    assert lib.mvsb200_pc_normals(*args, 20, None, 3, p, None) == -1
    args[13] = float("nan")
    assert lib.mvsb200_pc_knn(*args, 4, p, p, None) == -1
    assert _lib.PC_KNN_MAX == 32


def test_eval_tnt_write_argument_rules(tmp_path, capsys):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import eval_tnt
    finally:
        sys.path.pop(0)
    f = tmp_path / "a_file"
    f.write_text("x")
    base = ["--ply", "x.ply", "--tnt", str(tmp_path), "--scene", "S", "--tau", "0.01"]
    for bad in (["--write", str(f)], ["--write", ""], ["--write"]):
        with pytest.raises(SystemExit) as e:
            eval_tnt.main(base + bad)
        assert e.value.code == 2
    assert "--write" in capsys.readouterr().err
