"""K10 on the GPU (csrc/pointcloud.cu pc_knn_kernel) against the fp64 oracle (oracle/pc_normals.py): k-nearest neighbourhoods with
planted ties and caps, consistency with K8's nearest_neighbour, normals on noisy surfaces at several scales and offsets, an end
to end run from fused depth maps, and the Tanks and Temples files."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import fusion as fusion_oracle
import mvs_b200
from mvs_b200 import tanks

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytest.importorskip("scipy.spatial")
import pc_normals as oracle  # noqa: E402


def _g(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(DEV)


def _check_knn(q, t, k, max_dist=math.inf):
    d, idx = mvs_b200.k_nearest(_g(q), _g(t), k, max_dist)
    d, idx = d.cpu().numpy().astype(np.float64), idx.cpu().numpy()
    want_i, want_d, margin = oracle.knn(q, t, k, max_dist)
    pad = want_i < 0
    assert np.array_equal(idx < 0, pad) and np.isinf(d[pad]).all()
    ok = ~pad
    assert np.allclose(d[ok], want_d[ok], rtol=1e-6, atol=0)
    sure = margin >= 1e-4
    assert sure.mean() > 0.5
    assert all(set(idx[i][idx[i] >= 0]) == set(want_i[i][want_i[i] >= 0]) for i in np.nonzero(sure)[0])
    # order: exact wherever consecutive listed distances are 1e-4 apart
    gaps = np.diff(want_d, axis=1) / np.maximum(want_d[:, 1:], 1e-30)
    clear = np.concatenate([np.ones((len(q), 1), bool), gaps >= 1e-4], 1) & np.concatenate([gaps >= 1e-4, np.ones((len(q), 1), bool)], 1)
    clear &= sure[:, None] & ok
    assert np.array_equal(idx[clear], want_i[clear])
    return d, idx


@pytest.mark.parametrize("k", [1, 20, 32])
def test_k_nearest_against_the_oracle(k):
    rng = np.random.default_rng(k)
    t = rng.uniform(-1, 1, (20000, 3)).astype(np.float32)
    t[:10000, 2] *= 0.01                                              # a slab and a box: sparse and dense cells
    q = np.r_[t[:2000], rng.uniform(-1.5, 1.5, (2000, 3))].astype(np.float32)
    _check_knn(q, t, k)
    _check_knn(q, t, k, max_dist=0.08)                                # capped: many rows padded
    a = mvs_b200.k_nearest(_g(q), _g(t), k, 0.08)
    b = mvs_b200.k_nearest(_g(q), _g(t), k, 0.08)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_k_nearest_ties_go_to_the_smaller_rows():
    g = np.stack(np.meshgrid(*[np.arange(-4, 5)] * 3, indexing="ij"), -1).reshape(-1, 3).astype(np.float32)
    rng = np.random.default_rng(3)
    t = g[rng.permutation(len(g))]
    q = g[np.abs(g).max(1) <= 2]
    # k = 4: the centre and 3 of the 6 points at d^2 = 1; k = 10: the 7 of d^2 <= 1 and 3 of the 12 at d^2 = 2
    for k in (4, 10, 20):
        d, idx = mvs_b200.k_nearest(_g(q), _g(t), k)
        want_i, want_d, _ = oracle.knn(q, t, k)
        assert np.array_equal(idx.cpu().numpy(), want_i) and np.allclose(d.cpu().numpy(), want_d, rtol=1e-6, atol=0)


def test_k_equal_one_is_nearest_neighbour_bit_for_bit():
    rng = np.random.default_rng(4)
    t = _g(rng.uniform(-1, 1, (50000, 3)))
    q = _g(rng.uniform(-1.2, 1.2, (20000, 3)))
    for cap in (0.02, 1e3):
        d1, i1 = mvs_b200.nearest_neighbour(q, t, cap)
        dk, ik = mvs_b200.k_nearest(q, t, 1, cap)
        assert torch.equal(d1, dk[:, 0]) and torch.equal(i1, ik[:, 0])


def test_k_nearest_refusals_and_empty_inputs():
    x = _g(np.zeros((4, 3)))
    for k in (0, 33, 2.5):
        with pytest.raises(mvs_b200.MvsB200Error, match="k must be"):
            mvs_b200.k_nearest(x, x, k)
    with pytest.raises(mvs_b200.MvsB200Error, match="max_dist"):
        mvs_b200.k_nearest(x, x, 3, 0.0)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.k_nearest(x.cpu(), x, 3)
    with pytest.raises(mvs_b200.MvsB200Error, match="finite"):
        mvs_b200.k_nearest(_g([[np.nan, 0, 0]]), x, 3)
    d, i = mvs_b200.k_nearest(x, x[:0], 5)
    assert d.shape == (4, 5) and torch.isinf(d).all() and (i == -1).all()
    d, i = mvs_b200.k_nearest(x, x[:2], 5)                            # fewer points than k
    assert (i[:, :2] >= 0).all() and (i[:, 2:] == -1).all()


@pytest.mark.parametrize("kind,scale,offset", [("plane", 1.0, (0, 0, 0)), ("sphere", 1.0, (0.5, -2, 3)), ("cylinder", 2.0, (0, 0, 0)),
                                               ("sphere", 2.0, (1e4, -1e4, 1e4)), ("cylinder", 50.0, (-300, 20, 1e4)),
                                               ("plane", 5.0, (1e4, 1e4, -1e4))])
def test_estimate_normals_against_the_oracle(kind, scale, offset):
    rng = np.random.default_rng(int(scale * 100) + len(kind))
    p, _ = oracle.surface(kind, 6000, rng, scale, offset, noise=2e-3)
    v = np.asarray(offset) + rng.uniform(-3, 3, (len(p), 3)) * scale
    for k, cap, views in ((30, math.inf, None), (20, math.inf, v), (12, 0.06 * scale, v[0])):
        got = mvs_b200.estimate_normals(_g(p), k, max_dist=cap, viewpoints=views).cpu().numpy().astype(np.float64)
        want = oracle.normals(p, k, cap, views)
        none = want["count"] < 3
        assert (got[none] == 0).all() and (np.abs(got[~none]).sum(1) > 0).all()
        sure = (want["nbr"] >= 1e-4) & (want["eigengap"] >= 1e-3) & ~none
        assert sure.mean() > 0.5
        with np.errstate(invalid="ignore"):
            ang = oracle.angle(got[sure], want["normal"][sure])
        assert ang.max() <= 1e-6, (kind, k, float(ang.max()))
        signs = sure & (want["canon"] >= 1e-6) & (want["orient"] >= 1e-6)
        assert ((got[signs] * want["normal"][signs]).sum(1) > 0).all()
        assert np.allclose(np.linalg.norm(got[~none], axis=1), 1.0, atol=1e-6)


def test_zero_normals_for_caps_and_coincident_points():
    p = np.array([[0, 0, 0], [1, 0, 0], [5, 5, 5], [5, 5, 5], [5, 5, 5], [9, 9, 9], [9, 9, 9.5], [9, 9.5, 9], [9.5, 9, 9]], np.float32)
    got = mvs_b200.estimate_normals(_g(p), 4, max_dist=2.0).cpu().numpy()
    assert (got[:5] == 0).all() and (np.abs(got[5:]).sum(1) > 0).all()
    a = mvs_b200.estimate_normals(_g(p), 4)
    assert torch.equal(a, mvs_b200.estimate_normals(_g(p), 4))
    with pytest.raises(mvs_b200.MvsB200Error, match="viewpoints"):
        mvs_b200.estimate_normals(_g(p), 4, viewpoints=np.zeros((2, 3)))


def _disk_cloud():
    s = fusion_oracle.analytic_scene(6, 48, 64, normal="sweep", seed=0)
    depth = torch.from_numpy(s["depth"].astype(np.float32))[:, None].to(DEV)
    src = [[j for j in range(6) if j != i] for i in range(6)]
    xyz, rgb, masks = mvs_b200.fuse_depth_maps(depth, torch.ones_like(depth), torch.rand(6, 3, 48, 64, device=DEV), s["K"], s["R"],
                                               s["T"], src, conf_min=0.0, reproj_px=1e3, rel_depth=1.0, min_views=1)
    return s, xyz, rgb, masks


def test_end_to_end_fused_disk(tmp_path):
    s, xyz, rgb, masks = _disk_cloud()
    views = mvs_b200.point_viewpoints(masks, s["R"], s["T"])
    assert views.shape == (xyz.shape[0], 3) and views.dtype == torch.float64
    C = fusion_oracle.centres(s["R"], s["T"])
    counts = masks.reshape(6, -1).sum(1).cpu().numpy()
    assert np.array_equal(views.cpu().numpy(), np.repeat(C, counts, 0))
    nrm = mvs_b200.estimate_normals(xyz, viewpoints=views)
    n = nrm.cpu().numpy().astype(np.float64)
    p = xyz.cpu().numpy().astype(np.float64)
    # the disk is exact in the depth maps, so the fused points leave its plane by fp32 rounding only (measured: all 17,048 points
    # within 5.8e-6 rad, median 1.4e-6 rad)
    ang = oracle.angle(n, np.tile(s["n0"], (len(n), 1)))
    share = float((ang < 1e-3).mean())
    print({"points": len(n), "share_within_1e-3_rad": share, "median_rad": float(np.median(ang)), "max_rad": float(ang.max())})
    assert share >= 0.99
    assert ((n * (views.cpu().numpy() - p)).sum(1) > 0).all()       # every normal faces the camera that emitted its point
    want = oracle.normals(xyz.cpu().numpy(), 30, viewpoints=views.cpu().numpy())
    sure = (want["nbr"] >= 1e-4) & (want["eigengap"] >= 1e-3)
    assert oracle.angle(n[sure], want["normal"][sure]).max() <= 1e-6
    path = str(tmp_path / "disk.ply")
    mvs_b200.write_ply(path, xyz, rgb, normals=nrm)
    raw = open(path, "rb").read()
    body = raw[raw.index(b"end_header\n") + len(b"end_header\n"):]
    rec = np.frombuffer(body, dtype=[("p", "<f4", 3), ("n", "<f4", 3), ("c", "u1", 3)])
    assert np.array_equal(rec["n"], nrm.cpu().numpy()) and np.array_equal(rec["p"], xyz.cpu().numpy())


def _tnt_files_check(d, scene, out):
    for name, pts, dist in (("precision", out["xyz_down"], out["d_s"]), ("recall", out["gt_down"], out["d_t"])):
        raw = open(os.path.join(d, f"{scene}.{name}.ply"), "rb").read()
        body = raw[raw.index(b"end_header\n") + len(b"end_header\n"):]
        rec = np.frombuffer(body, dtype=[("p", "<f4", 3), ("n", "<f4", 3), ("c", "u1", 3)])
        assert len(rec) == (out["n_down"] if name == "precision" else out["m_down"])
        p32 = pts.float()
        assert np.array_equal(rec["p"], p32.cpu().numpy())
        assert np.array_equal(rec["n"], mvs_b200.estimate_normals(p32, 20).cpu().numpy())
        col = tanks.distance_colours(dist.double().cpu().numpy(), out["tau"])
        assert np.array_equal(rec["c"], np.clip(np.rint(col * 255.0), 0, 255).astype(np.uint8))
    assert np.array_equal(np.loadtxt(os.path.join(d, f"{scene}.precision.txt")), out["cum_precision"])
    assert np.array_equal(np.loadtxt(os.path.join(d, f"{scene}.recall.txt")), out["cum_recall"])
    assert np.array_equal(np.loadtxt(os.path.join(d, f"{scene}.prf_tau_plotstr.txt")),
                          [out["precision"], out["recall"], out["fscore"], out["tau"], 5.0])


def test_tanks_and_temples_files_and_tool(tmp_path):
    s, xyz, _, _ = _disk_cloud()
    r, n0, centre = s["radius"], s["n0"], s["centre"]
    a0 = np.cross(n0, [0.0, 1.0, 0.0])
    a0 /= np.linalg.norm(a0)
    b0 = np.cross(n0, a0)
    step = 0.01 * r
    k = np.arange(-int(1.1 * r / step) - 1, int(1.1 * r / step) + 2) * step
    u, v = (a.ravel() for a in np.meshgrid(k, k, indexing="ij"))
    on = u * u + v * v <= (1.1 * r) ** 2
    gt = (centre + u[on, None] * a0 + v[on, None] * b0).astype(np.float32)
    lo, hi = gt.min(0) - 1, gt.max(0) + 1
    crop = tanks._crop_volume("y", lo[1], hi[1], [[lo[0], 0, lo[2]], [hi[0], 0, lo[2]], [hi[0], 0, hi[2]], [lo[0], 0, hi[2]]])
    tau = 0.05
    out = mvs_b200.evaluate_tanks_and_temples(xyz, _g(gt), crop, None, tau, return_details=True)
    paths = mvs_b200.write_evaluation_files(str(tmp_path / "w"), "Disk", out)
    assert len(paths) == 5 and all(os.path.exists(p) for p in paths)
    _tnt_files_check(str(tmp_path / "w"), "Disk", out)
    # the tool: the same files, and the JSON without --write unchanged
    d = tmp_path / "Disk"
    d.mkdir()
    import json
    mvs_b200.write_ply(str(d / "Disk.ply"), gt)
    with open(d / "Disk.json", "w") as f:
        json.dump({"class_name": "SelectionPolygonVolume", "orthogonal_axis": "y", "axis_min": crop.axis_min, "axis_max": crop.axis_max,
                   "bounding_polygon": crop.polygon.tolist(), "version_major": 1, "version_minor": 0}, f)
    np.savetxt(str(d / "Disk_trans.txt"), np.eye(4), fmt="%.17g")
    ply = str(tmp_path / "rec.ply")
    mvs_b200.write_ply(ply, xyz)
    tool = os.path.join(ROOT, "tools", "eval_tnt.py")
    base = [sys.executable, tool, "--ply", ply, "--tnt", str(tmp_path), "--scene", "Disk", "--tau", str(tau)]
    plain = subprocess.run(base, capture_output=True, text=True)
    wrote = subprocess.run(base + ["--write", str(tmp_path / "t")], capture_output=True, text=True)
    assert plain.returncode == 0 and wrote.returncode == 0, plain.stderr + wrote.stderr
    assert plain.stdout.strip().splitlines()[-1] == wrote.stdout.strip().splitlines()[-1]
    _tnt_files_check(str(tmp_path / "t"), "Disk", out)
