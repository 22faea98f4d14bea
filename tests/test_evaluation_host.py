"""The DTU point-cloud evaluation without a GPU: the fp64 oracle's thinning, coverage and mask rules against independent
definitions, read_ply, load_dtu_eval on a synthetic DTU directory, and the refusals that need no device."""
import itertools
import os

import numpy as np
import pytest
import torch

import pointcloud_eval as oracle
import mvs_b200
from mvs_b200 import evaluation


def _clustered(rng, n, dst):
    c = rng.uniform(-1, 1, (max(n // 20, 1), 3))
    return (c[rng.integers(0, len(c), n)] + rng.normal(0, 1.5 * dst, (n, 3))).astype(np.float32)


def _lfmis(x, dst, order):
    """The lexicographically first maximal independent set of the "within dst" graph in `order`, by its definition: the set S
    with no two members within dst such that every point outside S has a member of S within dst that comes earlier in `order`
    -- found by brute force over all subsets of a tiny cloud."""
    n = len(x)
    d = np.sqrt(((x[:, None].astype(np.float64) - x[None].astype(np.float64)) ** 2).sum(-1))
    adj = (d <= dst) & ~np.eye(n, dtype=bool)
    rank = np.empty(n, int)
    rank[order] = np.arange(n)
    found = []
    for bits in itertools.product([0, 1], repeat=n):
        S = np.array(bits, bool)
        if (adj & S[:, None] & S[None]).any():
            continue
        if all(S[i] or (adj[i] & S & (rank < rank[i])).any() for i in range(n)):
            found.append(np.nonzero(S)[0])
    assert len(found) == 1
    return found[0]


def test_parallel_rounds_equal_the_sequential_greedy():
    rng = np.random.default_rng(0)
    for trial in range(30):
        dst = 0.2
        kind = trial % 3
        if kind == 0:
            x = rng.uniform(-1, 1, (300, 3)).astype(np.float32)
        elif kind == 1:
            x = _clustered(rng, 300, dst)
        else:                                   # exact duplicates
            x = rng.uniform(-1, 1, (60, 3)).astype(np.float32)
            x = x[rng.integers(0, 60, 300)]
        order = rng.permutation(len(x))
        nb, _ = oracle.neighbours(x, dst)
        seq = oracle.thin_sequential(x, dst, order, nb)
        par, rounds = oracle.thin_rounds(x, dst, order, nb)
        assert np.array_equal(seq, par) and rounds >= 1
        # maximal and independent
        keep = np.zeros(len(x), bool)
        keep[seq] = True
        for i in range(len(x)):
            assert keep[i] != bool(keep[nb[i]].any())


def test_greedy_is_the_lexicographically_first_maximal_independent_set():
    rng = np.random.default_rng(1)
    for trial in range(25):
        n = int(rng.integers(3, 11))
        x = rng.uniform(0, 0.5, (n, 3)).astype(np.float32)
        if trial % 5 == 0:
            x[1] = x[0]
        order = rng.permutation(n)
        want = _lfmis(x, 0.2, order)
        assert np.array_equal(oracle.thin_sequential(x, 0.2, order), want)
        assert np.array_equal(oracle.thin_rounds(x, 0.2, order)[0], want)


def test_coverage_rule_equals_the_literal_block_loop():
    rng = np.random.default_rng(2)
    bb = np.array([[-10.0, 5.0, 0.0], [130.0, 61.0, 59.0]])
    block = 60.0
    q = rng.uniform(-40, 220, (4000, 3))
    # points on the block edges, on BB[0] and on the last block's far face
    edges = np.array([[-10.0, 5.0, 0.0], [50.0, 65.0, 60.0], [170.0, 64.0, 59.0], [169.999, 64.999, 59.999], [-10.0001, 6.0, 1.0]])
    q = np.concatenate([q, edges])
    cov, margin = oracle.covered(q, bb, block)
    assert np.array_equal(cov, oracle.covered_literal(q, bb, block))
    assert cov.any() and (~cov).any()
    assert np.array_equal(cov[-5:], [True, False, False, True, False])
    got = evaluation.covered(torch.from_numpy(q), bb, block).numpy()
    assert np.array_equal(got, cov)


def test_round_half_away_and_voxel_edges():
    x = torch.tensor([0.5, -0.5, 1.5, -1.5, -0.4, 2.5, 0.49999999], dtype=torch.float64)
    assert evaluation.round_half_away(x).tolist() == [1.0, -1.0, 2.0, -2.0, -0.0, 3.0, 0.0]
    assert oracle.round_half_away(x.numpy().astype(np.float64)).tolist() == [1.0, -1.0, 2.0, -2.0, -0.0, 3.0, 0.0]
    # voxel-index edges: Res = 0.25 (exact), BB[0] = 0, mask 4 x 4 x 4 all true
    mask = np.ones((4, 4, 4), bool)
    bb = np.array([[0.0, 0.0, 0.0], [1.0, 1.0, 1.0]])
    res = 0.25
    idx = np.array([-0.5, -0.4, 0.0, 3.0, 3.4, 3.5, 2.5])           # (q - BB0) / Res on the x axis
    q = np.stack([idx * res, np.full(7, 0.5), np.full(7, 0.5)], 1)
    want = [False, True, True, True, True, False, True]
    got, margin = oracle.in_mask(q, mask, bb, res)
    assert got.tolist() == want
    assert evaluation.in_mask(torch.from_numpy(q), torch.from_numpy(mask), bb, res).tolist() == want
    assert margin[0] == 0 and margin[5] == 0 and margin[1] > 0


def test_read_ply_round_trip_ascii_mixed_types_and_refusals(tmp_path):
    rng = np.random.default_rng(3)
    xyz = rng.normal(0, 100, (257, 3)).astype(np.float32)
    rgb = rng.uniform(0, 1, (257, 3)).astype(np.float32)
    p = str(tmp_path / "a.ply")
    mvs_b200.write_ply(p, torch.from_numpy(xyz), torch.from_numpy(rgb))
    x2, c2 = mvs_b200.read_ply(p)
    assert x2.dtype == torch.float32 and np.array_equal(x2.numpy().view(np.int32), xyz.view(np.int32))
    assert np.array_equal(c2.numpy(), np.clip(np.rint(rgb.astype(np.float64) * 255), 0, 255).astype(np.uint8))
    mvs_b200.write_ply(p, xyz)
    x3, c3 = mvs_b200.read_ply(p)
    assert c3 is None and np.array_equal(x3.numpy(), xyz)
    # ASCII with extra properties of mixed types, a comment and an element before the vertices
    a = str(tmp_path / "b.ply")
    with open(a, "w") as f:
        f.write("ply\nformat ascii 1.0\ncomment made by hand\nelement camera 1\nproperty float fx\nelement vertex 3\n"
                "property double x\nproperty short id\nproperty float y\nproperty uchar red\nproperty float z\n"
                "property uchar green\nproperty uchar blue\nproperty int flags\nend_header\n500.0\n"
                "1.5 7 2.5 10 -3.25 20 30 -1\n0.1 -2 0.2 0 0.3 255 1 0\n4 0 5 1 6 2 3 9\n")
    xa, ca = mvs_b200.read_ply(a)
    assert np.array_equal(xa.numpy(), np.array([[1.5, 2.5, -3.25], [0.1, 0.2, 0.3], [4, 5, 6]], np.float32))
    assert ca.tolist() == [[10, 20, 30], [0, 255, 1], [1, 2, 3]]
    # binary with mixed types: double x, int16 id, float y/z, uint32 flags
    b = str(tmp_path / "c.ply")
    rec = np.zeros(5, dtype=[("x", "<f8"), ("id", "<i2"), ("y", "<f4"), ("z", "<f4"), ("flags", "<u4")])
    rec["x"], rec["y"], rec["z"] = np.arange(5) + 0.5, -np.arange(5), 2.0
    with open(b, "wb") as f:
        f.write(b"ply\nformat binary_little_endian 1.0\nelement vertex 5\nproperty double x\nproperty short id\nproperty float y\n"
                b"property float z\nproperty uint flags\nelement face 0\nproperty list uchar int vertex_indices\nend_header\n")
        f.write(rec.tobytes())
    xb, cb = mvs_b200.read_ply(b)
    assert cb is None and np.array_equal(xb.numpy(), np.stack([rec["x"], rec["y"], rec["z"]], 1).astype(np.float32))
    bad = {"big": "ply\nformat binary_big_endian 1.0\nelement vertex 1\nproperty float x\nproperty float y\nproperty float z\nend_header\n",
           "list": "ply\nformat ascii 1.0\nelement vertex 1\nproperty float x\nproperty float y\nproperty float z\n"
                   "property list uchar int idx\nend_header\n1 2 3 1 0\n",
           "noz": "ply\nformat ascii 1.0\nelement vertex 1\nproperty float x\nproperty float y\nend_header\n1 2\n"}
    for key, text in bad.items():
        q = str(tmp_path / f"{key}.ply")
        with open(q, "w") as f:
            f.write(text)
        with pytest.raises(mvs_b200.MvsB200Error, match={"big": "big-endian", "list": "list property", "noz": "no property 'z'"}[key]):
            mvs_b200.read_ply(q)


def test_load_dtu_eval_on_a_synthetic_directory(tmp_path):
    sio = pytest.importorskip("scipy.io")
    rng = np.random.default_rng(4)
    os.makedirs(tmp_path / "Points" / "stl")
    os.makedirs(tmp_path / "ObsMask")
    stl = rng.uniform(0, 50, (100, 3)).astype(np.float32)
    mvs_b200.write_ply(str(tmp_path / "Points" / "stl" / "stl024_total.ply"), stl)
    mask = rng.uniform(size=(6, 7, 8)) > 0.5
    bb = np.array([[-1.0, -2.0, -3.0], [60.0, 70.0, 80.0]])
    sio.savemat(str(tmp_path / "ObsMask" / "ObsMask24_10.mat"), {"ObsMask": mask, "BB": bb, "Res": 10.0})
    sio.savemat(str(tmp_path / "ObsMask" / "Plane24.mat"), {"P": np.array([[0.1], [0.2], [0.9], [-5.0]])})
    s, m, b, r, p = mvs_b200.load_dtu_eval(str(tmp_path), 24)
    assert np.array_equal(s.numpy(), stl) and m.dtype == torch.bool and np.array_equal(m.numpy(), mask)
    assert np.array_equal(b, bb) and r == 10.0 and np.array_equal(p, [0.1, 0.2, 0.9, -5.0])
    with pytest.raises(mvs_b200.MvsB200Error, match="not found"):
        mvs_b200.load_dtu_eval(str(tmp_path), 25)


def test_refusals_without_a_device():
    x = torch.rand(10, 3)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.thin_points(x)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.nearest_distance(x, x, 1.0)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.evaluate_point_cloud(x, x, np.ones((2, 2, 2), bool), np.zeros((2, 3)), 1.0, [0, 0, 1, 0])
    with pytest.raises(mvs_b200.MvsB200Error, match="permutation"):
        evaluation._order([0, 0, 1], 0, 3)
    with pytest.raises(mvs_b200.MvsB200Error, match="permutation"):
        evaluation._order([0, 1], 0, 3)
    with pytest.raises(mvs_b200.MvsB200Error, match="permutation"):
        evaluation._order([0.0, 1.0, 2.0], 0, 3)
    assert evaluation._order([2, 0, 1], 0, 3).tolist() == [2, 0, 1]
    assert torch.equal(evaluation._order(None, 5, 100), evaluation._order(None, 5, 100))
    for v in (0, -1, float("nan"), float("inf")):
        with pytest.raises(mvs_b200.MvsB200Error, match="must be > 0"):
            evaluation._positive(v, "dst")


def test_cell_size_rule_is_bounded():
    cell, nb = evaluation.cell_size([0, 0, 0], [400, 400, 300], 3_000_000)
    assert 512 * np.prod(nb) <= evaluation.CELL_BUDGET and cell > 0
    cell, nb = evaluation.cell_size([0, 0, 0], [0, 0, 0], 5)            # one point, repeated
    assert nb == [1, 1, 1]
    cell, nb = evaluation.cell_size([0, 0, 0], [100, 100, 0], 10_000, min_cell=0.5)   # a flat cloud
    assert cell >= 0.5 and 512 * np.prod(nb) <= evaluation.CELL_BUDGET
