"""The Tanks and Temples evaluation without a GPU: the crop-volume reader and the file loader, the C ABI's argument refusals, and the
fp64 oracle (oracle/tnt_eval.py) against independent restatements of its steps."""
import ctypes
import json

import numpy as np
import pytest
import torch

import tnt_eval as oracle
import mvs_b200
from mvs_b200 import tanks

SQUARE = [[0.0, 0.0, 0.0], [2.0, 0.0, 0.0], [2.0, 2.0, 0.0], [0.0, 2.0, 0.0]]


def _write(path, **kw):
    d = {"class_name": "SelectionPolygonVolume", "orthogonal_axis": "Y", "axis_min": -1.5, "axis_max": 2.25,
         "bounding_polygon": SQUARE, "version_major": 1, "version_minor": 0}
    d.update(kw)
    for k in [k for k, v in d.items() if v is None]:
        del d[k]
    with open(path, "w") as f:
        json.dump(d, f)
    return str(path)


@pytest.mark.parametrize("letter", ["X", "y", "z", "Z"])
def test_crop_volume_round_trip(tmp_path, letter):
    poly = [[0.1, -3.0, 7.25], [1.5, 2.0, -0.5], [-2.0, 0.3, 1.0], [0.0, 0.0, 1e-3]]
    c = mvs_b200.read_crop_volume(_write(tmp_path / "c.json", orthogonal_axis=letter, axis_min=-0.75, axis_max=3.5,
                                         bounding_polygon=poly))
    assert isinstance(c, mvs_b200.CropVolume)
    assert c.axis == letter.upper() and c.axis_min == -0.75 and c.axis_max == 3.5
    assert c.polygon.dtype == np.float64 and np.array_equal(c.polygon, np.array(poly))


@pytest.mark.parametrize("bad, match", [
    (dict(class_name="AxisAlignedBoundingBox"), "class_name"),
    (dict(class_name=None), "class_name"),
    (dict(bounding_polygon=None), "no bounding_polygon"),
    (dict(axis_min=None), "no axis_min"),
    (dict(orthogonal_axis="w"), "orthogonal_axis"),
    (dict(orthogonal_axis="xy"), "orthogonal_axis"),
    (dict(axis_max=float("inf")), "axis_max must be finite"),
    (dict(bounding_polygon=[[0, 0, 0], [1, float("nan"), 0], [1, 1, 0]]), "bounding_polygon must be finite"),
    (dict(bounding_polygon=[[0, 0, 0], [1, 0, 0]]), r"\[k, 3\]"),
    (dict(bounding_polygon=[[0, 0], [1, 0], [1, 1]]), r"\[k, 3\]"),
    (dict(bounding_polygon=[[float(i), float(i * i), 0.0] for i in range(1025)]), r"\[k, 3\]"),
])
def test_crop_volume_refusals(tmp_path, bad, match):
    with pytest.raises(mvs_b200.MvsB200Error, match=match):
        mvs_b200.read_crop_volume(_write(tmp_path / "c.json", **bad))


def test_crop_volume_not_json(tmp_path):
    p = tmp_path / "c.json"
    p.write_text("{not json")
    with pytest.raises(mvs_b200.MvsB200Error, match="not JSON"):
        mvs_b200.read_crop_volume(str(p))


def test_load_tnt_eval_names_the_missing_file(tmp_path):
    d = tmp_path / "Barn"
    d.mkdir()
    with pytest.raises(mvs_b200.MvsB200Error, match=r"Barn\.ply not found"):
        mvs_b200.load_tnt_eval(str(tmp_path), "Barn")
    gt = np.random.default_rng(0).normal(size=(50, 3)).astype(np.float32)
    mvs_b200.write_ply(str(d / "Barn.ply"), gt)
    with pytest.raises(mvs_b200.MvsB200Error, match=r"Barn\.json not found"):
        mvs_b200.load_tnt_eval(str(tmp_path), "Barn")
    _write(d / "Barn.json")
    with pytest.raises(mvs_b200.MvsB200Error, match=r"Barn_trans\.txt not found"):
        mvs_b200.load_tnt_eval(str(tmp_path), "Barn")
    A = np.array([[0.0, -2.0, 0.0, 1.5], [2.0, 0.0, 0.0, -0.25], [0.0, 0.0, 2.0, 3.0], [0.0, 0.0, 0.0, 1.0]])
    np.savetxt(str(d / "Barn_trans.txt"), A)
    g, crop, trans = mvs_b200.load_tnt_eval(str(tmp_path), "Barn")
    assert np.array_equal(g.numpy(), gt) and crop.axis == "Y" and np.array_equal(trans, A)
    np.savetxt(str(d / "Barn_trans.txt"), A[:3])
    with pytest.raises(mvs_b200.MvsB200Error, match="4 x 4"):
        mvs_b200.load_tnt_eval(str(tmp_path), "Barn")


def test_transform_refusals_and_identity():
    assert tanks._affine(None) is None and tanks._affine(np.eye(4)) is None
    A = np.eye(4)
    A[0, 3] = 0.5
    assert tanks._affine(A).tolist() == [1, 0, 0, 0.5, 0, 1, 0, 0, 0, 0, 1, 0]
    P = np.eye(4)
    P[3, 2] = 1e-9
    with pytest.raises(mvs_b200.MvsB200Error, match="affine"):
        tanks._affine(P)
    with pytest.raises(mvs_b200.MvsB200Error, match="finite"):
        tanks._affine(np.full((4, 4), np.nan))
    with pytest.raises(mvs_b200.MvsB200Error, match="4 x 4"):
        tanks._affine(np.eye(3))


def test_cpu_tensors_are_refused():
    crop = tanks._crop_volume("z", -1, 1, SQUARE)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.evaluate_tanks_and_temples(torch.zeros(4, 3), torch.zeros(4, 3), crop, None, 0.01)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.voxel_down_sample(torch.zeros(4, 3, dtype=torch.float64), 0.1)


def test_abi_refuses_bad_polygons_and_axes():
    lib = mvs_b200.load_library()
    buf = ctypes.c_void_p(16)                   # never dereferenced: argument checks come before any CUDA call
    a = (ctypes.c_double * 12)(*([1.0] + [0.0] * 11))
    for k, axis, match in ((2, 1, b"3 to 1024"), (1025, 1, b"3 to 1024"), (4, 3, b"axis"), (4, -1, b"axis")):
        rc = lib.mvsb200_pc_transform_crop(buf, 10, a, buf, k, axis, 0.0, 1.0, buf, buf, None)
        assert rc == -1
        assert match in lib.mvsb200_last_error()
    bad = (ctypes.c_double * 12)(*([float("nan")] + [0.0] * 11))
    assert lib.mvsb200_pc_transform_crop(buf, 10, bad, buf, 4, 1, 0.0, 1.0, buf, buf, None) == -1
    assert b"finite" in lib.mvsb200_last_error()
    assert lib.mvsb200_pc_voxel_keys(buf, 10, 0.0, 0.0, 0.0, 0.1, 1 << 31, 1 << 31, 1 << 1, buf, None) == -1
    assert b"2^62" in lib.mvsb200_last_error()
    assert lib.mvsb200_pc_voxel_keys(buf, 10, 0.0, 0.0, 0.0, 0.0, 1, 1, 1, buf, None) == -1


# ---- the oracle against independent restatements ------------------------------------------------------------------------------------

CONCAVE = [[0.0, 0.0], [4.0, 0.0], [4.0, 3.0], [2.5, 3.0], [2.5, 1.0], [1.5, 1.0], [1.5, 3.0], [0.0, 3.0]]   # a U, horizontal edges


def _polygon(axis, uv):
    """[k, 3] vertices with the (u, v) columns of `axis` set to uv and the w column junk (CropInPolygon never reads it)."""
    u, v, w = oracle.AXES[axis]
    b = np.zeros((len(uv), 3))
    b[:, u], b[:, v] = np.asarray(uv)[:, 0], np.asarray(uv)[:, 1]
    b[:, w] = np.arange(len(uv)) * 7.5
    return b


@pytest.mark.parametrize("axis", ["x", "y", "z"])
def test_oracle_crop_matches_the_winding_number(axis):
    rng = np.random.default_rng(1)
    p = rng.uniform(-1, 5, (20000, 3))
    poly = _polygon(axis, CONCAVE)
    got, margin = oracle.crop(p, axis, 0.5, 4.0, poly)
    want = oracle.inside_winding(p, axis, 0.5, 4.0, poly)
    away = margin > 1e-3
    assert away.mean() > 0.95 and np.array_equal(got[away], want[away])
    assert 0.1 < got.mean() < 0.6


def test_oracle_crop_mutations_differ_on_planted_points():
    poly = _polygon("z", CONCAVE)
    # on a vertex v-level (p_v = 1 = b_v of the U's inner bottom), on an edge's v-range end, on axis_min / axis_max
    p = np.array([[0.5, 3.0, 1.0], [2.0, 1.0, 1.0], [1.0, 0.0, 1.0], [1.0, 2.0, 0.5], [1.0, 2.0, 4.0]])
    base = oracle.crop(p, "z", 0.5, 4.0, poly)[0]
    assert base.tolist() == [True, True, False, True, True]
    assert not np.array_equal(oracle.crop(p, "z", 0.5, 4.0, poly, closed_both=True)[0], base)
    assert not np.array_equal(oracle.crop(p, "z", 0.5, 4.0, poly, exclusive_bounds=True)[0], base)


def test_oracle_voxel_step_matches_a_dict():
    rng = np.random.default_rng(2)
    p = np.concatenate([rng.normal(0, 0.3, (3000, 3)), rng.uniform(-0.01, 0.01, (500, 3)) + 0.123])
    voxel = 0.05
    mean, counts, keys = oracle.voxel_down_sample(p, voxel)
    want = oracle.voxel_down_sample_dict(p, voxel)
    assert len(mean) == len(want) and counts.sum() == len(p) and np.all(np.diff(keys) > 0)
    got = {tuple(np.floor((m - (p.min(0) - voxel * 0.5)) / voxel).astype(int)): m for m in mean}
    assert got.keys() == want.keys()
    for k, m in want.items():
        assert np.array_equal(got[k], m)                # the dict adds in input order from 0: the same bits
    # the mutations change something
    assert not np.array_equal(oracle.voxel_down_sample(p, voxel, half_offset=False)[1], counts)
    assert not np.array_equal(oracle.voxel_down_sample(p, voxel, summation="pairwise")[0], mean)


def test_oracle_curves_follow_np_histogram_semantics():
    tau = 0.01
    e = oracle.histogram_edges(tau)
    assert len(e) >= 499 and e[0] == 0 and e[-1] < 5 * tau
    rng = np.random.default_rng(3)
    d_s = np.concatenate([rng.uniform(0, 6 * tau, 5000), e[[0, 7, 100, -1]], [np.inf, np.inf]])
    d_t = rng.uniform(0, 3 * tau, 3000)
    P, R, F, edges, cum_s, cum_t = oracle.f1_histo(tau, 5, d_s, d_t)
    # a literal count: [e_k, e_k+1) and the last bin closed; values outside [e_0, e_K] dropped
    K = len(e) - 1
    hist = np.zeros(K, np.int64)
    for d in d_s:
        for k in range(K):
            if e[k] <= d < e[k + 1] or (k == K - 1 and d == e[K]):
                hist[k] += 1
                break
    assert np.array_equal(cum_s, np.cumsum(hist).astype(float) / len(d_s))
    assert hist[-1] >= 1 and cum_s[-1] < 1
    assert P == np.sum(d_s < tau) / len(d_s) and R == np.sum(d_t < tau) / len(d_t)
    assert F == 2 * R * P / (R + P)
    # the device histogram's formula on the host: searchsorted(right) - 1, clamped, then the range filter
    idx = np.minimum(np.searchsorted(e, d_s, side="right") - 1, K - 1)
    ok = (d_s >= e[0]) & (d_s <= e[-1])
    assert np.array_equal(np.bincount(idx[ok], minlength=K), hist)


def test_fscore_edge_cases():
    z = oracle.f1_histo(0.01, 5, np.zeros(0), np.ones(5))
    assert z[:3] == (0.0, 0.0, 0.0) and all(np.array_equal(a, [0]) for a in z[3:])
    far = oracle.f1_histo(0.01, 5, np.full(4, np.inf), np.full(3, 0.02))
    assert far[:3] == (0.0, 0.0, 0.0) and far[4][-1] == 0 and far[5][-1] == 1
    one = oracle.f1_histo(0.01, 5, np.zeros(3), np.full(2, 0.005))
    assert one[:3] == (1.0, 1.0, 1.0)
    half = oracle.f1_histo(0.01, 5, np.array([0.0, 0.02]), np.zeros(2))
    assert half[:3] == (0.5, 1.0, 2 * 1.0 * 0.5 / 1.5)


def test_search_cap_is_above_every_counted_distance():
    for tau in (0.01, 0.003, 0.05, 0.3, 1.0, 7.0, 1e-4):
        for stretch in (5, 1, 2.5):
            e = tanks.histogram_edges(tau, stretch)
            cap = tanks.search_cap(tau, stretch, e)
            assert cap == float(np.float32(cap)) and cap > stretch * tau and cap > e[-1]
