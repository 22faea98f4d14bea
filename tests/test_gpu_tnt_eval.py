"""The Tanks and Temples evaluation (K9, csrc/pointcloud.cu) on the GPU against the fp64 oracle (oracle/tnt_eval.py): bit-exact
transform, crop and voxel means, the capped distances against cKDTree, the whole call on a scene whose every decision has a clear
margin, an end-to-end run from fused depth maps, mutation checks, determinism and refusals."""
import json
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch

import fusion as fusion_oracle
import tnt_eval as oracle
import mvs_b200
from mvs_b200 import tanks

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytest.importorskip("scipy.spatial")


def _g(a, dtype=np.float32):
    return torch.from_numpy(np.ascontiguousarray(a, dtype)).to(DEV)


def _rotation(rng):
    q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    return q * np.sign(np.linalg.det(q))


def _similarity(rng, scale, shift):
    A = np.eye(4)
    A[:3, :3] = scale * _rotation(rng)
    A[:3, 3] = shift
    return A


CONVEX = [[-1.0, -1.5], [2.0, -1.0], [2.5, 1.0], [0.5, 2.5], [-1.5, 1.0]]
CONCAVE = [[-2.0, -2.0], [2.0, -2.0], [2.0, 2.0], [0.5, 2.0], [0.5, -0.5], [-0.5, -0.5], [-0.5, 2.0], [-2.0, 2.0]]   # a U
AMIN, AMAX = -1.25, 1.75


def _crop_volume(axis, uv):
    u, v, w = oracle.AXES[axis]
    b = np.zeros((len(uv), 3))
    b[:, u], b[:, v] = np.asarray(uv)[:, 0], np.asarray(uv)[:, 1]
    b[:, w] = 99.0                                      # never read
    return tanks._crop_volume(axis.upper(), AMIN, AMAX, b)


def _planted(axis, uv):
    """Points (in the frame after the transform) on the vertex v-levels and the edges' v-range ends, and on axis_min / axis_max."""
    u, v, w = oracle.AXES[axis]
    uv = np.asarray(uv)
    pts = []
    for bu, bv in uv:
        for du in (-0.25, 0.0, 0.25):
            for pw in (0.5, AMIN, AMAX):
                p = np.zeros(3)
                p[u], p[v], p[w] = bu + du, bv, pw
                pts.append(p)
    for pw in (AMIN, AMAX, np.nextafter(AMIN, -1), np.nextafter(AMAX, 2)):
        p = np.zeros(3)
        p[u], p[v], p[w] = 1.0, 0.0, pw
        pts.append(p)
    return np.array(pts)


def _case(axis, poly, tf, rng):
    uv = CONVEX if poly == "convex" else CONCAVE
    crop = _crop_volume(axis, uv)
    planted = _planted(axis, uv)
    if tf == "identity":
        A, x_planted = None, planted
    elif tf == "dyadic":                                    # exact in both directions: the planted points land on their levels
        P = np.array([[0.0, 2.0, 0.0], [0.0, 0.0, -2.0], [2.0, 0.0, 0.0]])
        A = np.eye(4)
        A[:3, :3], A[:3, 3] = P, [0.5, -0.25, 0.125]
        x_planted = (planted - A[:3, 3]) @ np.linalg.inv(P).T
    else:                                                   # a scaled rigid transform
        A = _similarity(rng, 1.7, [0.3, -0.2, 0.1])
        x_planted = (planted - A[:3, 3]) @ np.linalg.inv(A[:3, :3]).T
    if A is None:
        x_rand = rng.uniform(-3, 3, (50000, 3))
    else:
        x_rand = (rng.uniform(-3, 3, (50000, 3)) - A[:3, 3]) @ np.linalg.inv(A[:3, :3]).T
    x = np.concatenate([x_rand, x_planted]).astype(np.float32)
    return x, crop, A, len(x_rand)


@pytest.mark.parametrize("poly", ["convex", "concave"])
@pytest.mark.parametrize("tf", ["identity", "dyadic", "rigid"])
@pytest.mark.parametrize("axis", ["x", "y", "z"])
def test_crop_is_bit_exact(axis, tf, poly):
    rng = np.random.default_rng(zlib.crc32(f"{axis}{tf}{poly}".encode()))
    x, crop, A, n_rand = _case(axis, poly, tf, rng)
    got, kept = mvs_b200.crop_points(_g(x), crop, A)
    x64 = x.astype(np.float64)
    xt = x64 if A is None else oracle.transform(x64, A)
    want, _ = oracle.crop(xt, crop.axis, crop.axis_min, crop.axis_max, crop.polygon)
    assert np.array_equal(kept.cpu().numpy(), np.nonzero(want)[0])
    assert np.array_equal(got.cpu().numpy(), xt[want])               # fp64 bits
    assert 0.05 < want[:n_rand].mean() < 0.7
    # the planted points are the ones every mutation is judged on
    if tf != "rigid":
        pl = slice(n_rand, None)
        for mut in (dict(closed_both=True), dict(exclusive_bounds=True)):
            m = oracle.crop(xt, crop.axis, crop.axis_min, crop.axis_max, crop.polygon, **mut)[0]
            assert not np.array_equal(m[pl], want[pl]), mut
    if tf == "dyadic":
        before = oracle.crop(x64, crop.axis, crop.axis_min, crop.axis_max, crop.polygon)[0]
        assert not np.array_equal(before, want)                       # crop before transform


def _voxel_cloud(rng, voxel):
    """Clusters of thousands of points inside single voxels, a spread, a point at the origin fixing vmin = -voxel / 2, and points
    where floor((p - vmin) / voxel) and floor((p - vmin) * (1 / voxel)) disagree."""
    dense = [rng.uniform(-0.3 * voxel, 0.3 * voxel, (4000, 3)) + np.array([4, 7, 2]) * voxel,
             rng.uniform(-0.45 * voxel, 0.45 * voxel, (2500, 3)) + np.array([40, 3, 9]) * voxel]
    spread = rng.uniform(0, 60 * voxel, (30000, 3))
    vmin = 0.0 - voxel * 0.5
    cand = []
    for k in range(1, 60):
        c = vmin + k * voxel
        for t in range(-3, 4):
            q = c
            for _ in range(abs(t)):
                q = np.nextafter(q, np.inf if t > 0 else -np.inf)
            if np.floor((q - vmin) / voxel) != np.floor((q - vmin) * (1.0 / voxel)):
                cand.append(q)
    cand = np.array(cand)
    assert len(cand) >= 3
    odd = np.stack([cand, np.full_like(cand, 0.37 * voxel * 60), np.full_like(cand, 0.5 * voxel * 60)], 1)
    return np.concatenate([[[0.0, 0.0, 0.0]], dense[0], spread, dense[1], odd])


@pytest.mark.parametrize("voxel", [0.1, 0.005, 0.0137])
def test_voxel_down_sample_is_bit_exact(voxel):
    rng = np.random.default_rng(int(voxel * 1e4))
    p = _voxel_cloud(rng, voxel)
    mean, mean32, counts = mvs_b200.voxel_down_sample(_g(p, np.float64), voxel)
    want, wcounts, _ = oracle.voxel_down_sample(p, voxel)
    assert counts.max() >= 2500
    assert np.array_equal(counts.cpu().numpy(), wcounts)
    assert np.array_equal(mean.cpu().numpy(), want)
    assert np.array_equal(mean32.cpu().numpy(), want.astype(np.float32))
    for mut in (dict(summation="pairwise"), dict(divide=False), dict(half_offset=False)):
        m, c, _ = oracle.voxel_down_sample(p, voxel, **mut)
        assert m.shape != want.shape or not np.array_equal(m, want) or not np.array_equal(c, wcounts), mut


def _check_distances(got, q32, t32, cap):
    want = oracle.nearest(q32.astype(np.float64), t32.astype(np.float64), cap)
    g = got.cpu().double().numpy()
    sure = np.abs(oracle.nearest(q32, t32, np.inf) - cap) / cap >= 1e-4
    assert np.array_equal(np.isfinite(g)[sure], np.isfinite(want)[sure])
    both = np.isfinite(g) & np.isfinite(want)
    assert both.sum() > 100
    assert np.max(np.abs(g[both] - want[both]) / np.maximum(want[both], 1e-30)) <= 1e-6


def _noisy_scene(rng, n_gt=60000, n_rec=40000):
    """A bumpy surface, a reconstruction of part of it with noise and outliers, in metres."""
    def surf(n):
        xy = rng.uniform(-2, 2, (n, 2))
        return np.concatenate([xy, 0.2 * np.sin(2 * xy[:, :1]) * np.cos(3 * xy[:, 1:])], 1)
    gt = surf(n_gt)
    rec = surf(n_rec)[: n_rec] * [0.8, 1.0, 1.0] + rng.normal(0, 0.004, (n_rec, 3))
    rec[: n_rec // 20] = rng.uniform(-2, 2, (n_rec // 20, 3))
    return gt.astype(np.float32), rec.astype(np.float32)


def test_distances_against_ckdtree():
    rng = np.random.default_rng(5)
    gt, rec = _noisy_scene(rng)
    crop = _crop_volume("z", CONCAVE)
    tau = 0.02
    out = mvs_b200.evaluate_tanks_and_temples(_g(rec), _g(gt), crop, None, tau, return_details=True)
    cap = tanks.search_cap(tau, 5, tanks.histogram_edges(tau))
    s32, t32 = out["xyz_down"].float().cpu().numpy(), out["gt_down"].float().cpu().numpy()
    _check_distances(out["d_s"], s32, t32, cap)
    _check_distances(out["d_t"], t32, s32, cap)
    # the GPU's histograms are np.histogram of its own distances, exactly
    for d, cum, n in ((out["d_s"], out["cum_precision"], out["n_down"]), (out["d_t"], out["cum_recall"], out["m_down"])):
        h = np.histogram(d.cpu().numpy(), out["edges"])[0]
        assert np.array_equal(cum, np.cumsum(h).astype(float) / n)
    assert np.array_equal(out["edges"], np.arange(0, tau * 5, tau / 100))
    assert 0.2 < out["precision"] < 1 and 0.2 < out["recall"] < 1


def _lattice_scene(rng, A):
    """GT: a 30 x 30 lattice of pitch 0.1 on z = 0; the reconstruction: one point above 70 % of the sites at heights (k + 1/2) tau / 100
    (k < 700, so some beyond the cap), and outliers 0.3 above; given to the evaluation in the frame A maps to the GT's.  Every
    distance is one height, half a bin from every edge, from tau and from the cap; every point is alone in its voxel."""
    tau = 0.01
    i, j = np.meshgrid(np.arange(30), np.arange(30), indexing="ij")
    gt = np.stack([0.1 * i.ravel(), 0.1 * j.ravel(), np.zeros(900)], 1).astype(np.float32)
    sites = rng.permutation(900)[:630]
    h = (rng.integers(0, 700, 630) + 0.5) * tau / 100
    rec = np.concatenate([gt[sites].astype(np.float64) + np.stack([np.zeros(630), np.zeros(630), h], 1),
                          gt[rng.permutation(900)[:40]].astype(np.float64) + [0.03, 0.03, 0.3]])
    rec_in = (rec - A[:3, 3]) @ np.linalg.inv(A[:3, :3]).T
    # an L, edges on half-lattice coordinates
    crop = tanks._crop_volume("z", -0.5, 0.5, [[-0.05, -0.05, 0], [2.05, -0.05, 0], [2.05, 1.05, 0], [1.05, 1.05, 0],
                                                [1.05, 2.55, 0], [-0.05, 2.55, 0]])
    return rec_in.astype(np.float32), gt, crop, tau


def test_whole_call_against_the_oracle():
    rng = np.random.default_rng(6)
    A = _similarity(rng, 1.3, [0.7, -0.4, 0.2])
    rec, gt, crop, tau = _lattice_scene(rng, A)
    n0 = mvs_b200.launch_count()
    got = mvs_b200.evaluate_tanks_and_temples(_g(rec), _g(gt), crop, A, tau, return_details=True)
    launches = mvs_b200.launch_count() - n0
    assert launches == 2 * 3 + 2 * 3                        # per cloud crop, keys, means; per direction grid keys, cells, search
    cap = tanks.search_cap(tau, 5, tanks.histogram_edges(tau))
    want = oracle.evaluate(rec, gt, tuple(crop), A, tau, cap=cap)
    assert want["margin_s"].min() >= 1e-4 and want["margin_t"].min() >= 1e-4
    assert np.array_equal(got["xyz_down"].cpu().numpy(), want["xyz_down"])
    assert np.array_equal(got["gt_down"].cpu().numpy(), want["gt_down"])
    for k in ("n", "n_cropped", "n_down", "m", "m_cropped", "m_down", "n_precision", "m_recall", "precision", "recall", "fscore"):
        assert got[k] == want[k], k
    for k in ("edges", "cum_precision", "cum_recall"):
        assert np.array_equal(got[k], want[k]), k
    assert 0 < got["n_precision"] < got["n_down"] < got["n"] and 0 < got["m_recall"] < got["m_down"] < got["m"]
    assert 0 < got["cum_precision"][-1] < 1 and got["cum_precision"][-1] > got["precision"]
    # determinism
    again = mvs_b200.evaluate_tanks_and_temples(_g(rec), _g(gt), crop, A, tau, return_details=True)
    for k in ("xyz_down", "gt_down", "d_s", "d_t"):
        assert torch.equal(got[k], again[k]), k
    for k in ("cum_precision", "cum_recall"):
        assert np.array_equal(got[k], again[k])
    assert got["fscore"] == again["fscore"]


def test_empty_crops_and_no_hits():
    rng = np.random.default_rng(7)
    gt, rec = _noisy_scene(rng, 5000, 3000)
    crop = _crop_volume("z", CONVEX)
    away = np.eye(4)
    away[2, 3] = 100.0                                     # the reconstruction leaves the crop volume
    for r in (mvs_b200.evaluate_tanks_and_temples(_g(rec), _g(gt), crop, away, 0.01),
              mvs_b200.evaluate_tanks_and_temples(torch.empty(0, 3, device=DEV), _g(gt), crop, None, 0.01)):
        assert r["n_cropped"] == 0 and r["m_down"] > 0
        assert (r["precision"], r["recall"], r["fscore"]) == (0.0, 0.0, 0.0)
        assert all(np.array_equal(r[k], [0]) for k in ("edges", "cum_precision", "cum_recall"))
    side = np.eye(4)
    side[2, 3] = 0.5                                       # inside the volume but farther than the cap: P = R = 0, F = 0
    r = mvs_b200.evaluate_tanks_and_temples(_g(rec * [1, 1, 0]), _g(gt * [1, 1, 0]), crop, side, 0.01)
    assert r["n_down"] > 0 and r["m_down"] > 0 and (r["precision"], r["recall"], r["fscore"]) == (0.0, 0.0, 0.0)
    assert r["cum_precision"][-1] == 0 and len(r["edges"]) == 500


def test_refusals():
    crop = _crop_volume("y", CONVEX)
    x = torch.rand(100, 3, device=DEV)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.evaluate_tanks_and_temples(x.cpu(), x, crop, None, 0.01)
    with pytest.raises(mvs_b200.MvsB200Error, match="finite"):
        mvs_b200.evaluate_tanks_and_temples(torch.where(x > 0.9, float("nan"), x), x, crop, None, 0.01)
    P = np.eye(4)
    P[3, 0] = 0.5
    with pytest.raises(mvs_b200.MvsB200Error, match="affine"):
        mvs_b200.evaluate_tanks_and_temples(x, x, crop, P, 0.01)
    with pytest.raises(mvs_b200.MvsB200Error, match="tau"):
        mvs_b200.evaluate_tanks_and_temples(x, x, crop, None, 0.0)
    far = torch.tensor([[0.0, 0.0, 0.0], [1000.0, 0.0, 0.0]], dtype=torch.float64, device=DEV)
    with pytest.raises(mvs_b200.MvsB200Error, match="too small"):
        mvs_b200.voxel_down_sample(far, 1e-7)
    with pytest.raises(mvs_b200.MvsB200Error, match="crop"):
        mvs_b200.crop_points(x, (crop.axis, crop.axis_min, crop.axis_max, crop.polygon))


def test_end_to_end_fused_disk_and_wrong_alignment():
    s = fusion_oracle.analytic_scene(6, 48, 64, normal="sweep", seed=0)
    depth = torch.from_numpy(s["depth"].astype(np.float32))[:, None].to(DEV)
    src = [[j for j in range(6) if j != i] for i in range(6)]
    xyz, _, _ = mvs_b200.fuse_depth_maps(depth, torch.ones_like(depth), torch.rand(6, 3, 48, 64, device=DEV), s["K"], s["R"], s["T"],
                                         src, conf_min=0.0, reproj_px=1e3, rel_depth=1.0, min_views=1)
    r, n0, centre = s["radius"], s["n0"], s["centre"]
    a0 = np.cross(n0, [0.0, 1.0, 0.0])
    a0 /= np.linalg.norm(a0)
    b0 = np.cross(n0, a0)
    A = _similarity(np.random.default_rng(8), 1.7, [3.0, -1.0, 2.0])
    # the ground truth: the disk (radius + 10 %) on a lattice of 0.01 r in its plane, mapped by A
    step = 0.01 * r
    k = np.arange(-int(1.1 * r / step) - 1, int(1.1 * r / step) + 2) * step
    u, v = (a.ravel() for a in np.meshgrid(k, k, indexing="ij"))
    on = u * u + v * v <= (1.1 * r) ** 2
    disk = centre + u[on, None] * a0 + v[on, None] * b0
    gt = oracle.transform(disk, A).astype(np.float32)
    lo, hi = gt.min(0) - 1, gt.max(0) + 1
    crop = tanks._crop_volume("y", lo[1], hi[1], [[lo[0], 0, lo[2]], [hi[0], 0, lo[2]], [hi[0], 0, hi[2]], [lo[0], 0, hi[2]]])
    tau = 0.05 * 1.7 * r / 4                               # 0.085: about 6 lattice steps of the GT, far above the fp32 noise
    out = mvs_b200.evaluate_tanks_and_temples(xyz, _g(gt), crop, A, tau)
    print({k: out[k] for k in ("precision", "recall", "fscore", "n", "n_down", "m", "m_down")})
    assert out["n_cropped"] == out["n"] > 1000 and out["m_cropped"] == out["m"]
    assert out["precision"] >= 0.99
    want = oracle.evaluate(xyz.cpu().numpy(), gt, tuple(crop), A, tau, cap=tanks.search_cap(tau, 5, tanks.histogram_edges(tau)))
    assert want["m_down"] == out["m_down"] and want["n_down"] == out["n_down"]
    unsure_t = int((want["margin_t"] < 1e-4).sum())
    unsure_s = int((want["margin_s"] < 1e-4).sum())
    assert abs(out["m_recall"] - want["m_recall"]) <= unsure_t and abs(out["n_precision"] - want["n_precision"]) <= unsure_s
    assert 0.2 < out["recall"] < 0.95                      # the ground truth reaches 10 % beyond the fused disk
    inv = np.eye(4)
    inv[:3, :3] = np.linalg.inv(A[:3, :3])
    inv[:3, 3] = -inv[:3, :3] @ A[:3, 3]
    wrong = mvs_b200.evaluate_tanks_and_temples(xyz, _g(gt), crop, inv, tau)
    assert wrong["precision"] < 0.1


def test_eval_tnt_tool_on_a_synthetic_directory(tmp_path):
    rng = np.random.default_rng(9)
    A = _similarity(rng, 1.3, [0.7, -0.4, 0.2])
    rec, gt, crop, tau = _lattice_scene(rng, A)
    d = tmp_path / "Synth"
    d.mkdir()
    mvs_b200.write_ply(str(d / "Synth.ply"), gt)
    with open(d / "Synth.json", "w") as f:
        json.dump({"class_name": "SelectionPolygonVolume", "orthogonal_axis": "z", "axis_min": crop.axis_min, "axis_max": crop.axis_max,
                   "bounding_polygon": crop.polygon.tolist(), "version_major": 1, "version_minor": 0}, f)
    np.savetxt(str(d / "Synth_trans.txt"), A, fmt="%.17g")
    ply = str(tmp_path / "rec.ply")
    mvs_b200.write_ply(ply, rec)
    out = str(tmp_path / "r.json")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "eval_tnt.py"), "--ply", ply, "--tnt", str(tmp_path), "--scene",
                        "Synth", "--tau", str(tau), "--out", out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = json.load(open(out))
    assert json.loads(r.stdout.strip().splitlines()[-1])["fscore"] == got["fscore"]
    want = mvs_b200.evaluate_tanks_and_temples(_g(rec), _g(gt), crop, A, tau)
    for k in ("precision", "recall", "fscore", "n_down", "m_down"):
        assert got[k] == want[k], k
    assert got["cum_recall"] == want["cum_recall"].tolist()
