"""The DTU point-cloud evaluation (K8, csrc/pointcloud.cu) on the GPU against the fp64 oracle (oracle/pointcloud_eval.py): exact
capped nearest distances, greedy thinning, the whole evaluation, an end-to-end run from fused depth maps, mutation checks and
determinism."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import fusion as fusion_oracle
import pointcloud_eval as oracle
import mvs_b200
from mvs_b200 import evaluation

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _g(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(DEV)


def _check_nearest(q, t, max_dist, **kw):
    got = mvs_b200.nearest_distance(_g(q), _g(t), max_dist, **kw).cpu().double().numpy()
    want, margin = oracle.capped(oracle.nearest(q, t), max_dist)
    sure = margin >= 1e-4
    assert np.array_equal(np.isfinite(got)[sure], np.isfinite(want)[sure])
    both = np.isfinite(got) & np.isfinite(want)
    if both.any():
        rel = np.abs(got[both] - want[both]) / np.maximum(want[both], 1e-30)
        assert rel.max() <= 1e-6 or np.abs(got[both] - want[both]).max() <= 1e-7
    return got, want


def _surface(rng, n):
    u, v = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, np.pi / 2, n)
    return np.stack([10 * np.cos(u) * np.sin(v), 10 * np.sin(u) * np.sin(v), 10 * np.cos(v)], 1)


@pytest.mark.parametrize("kind", ["uniform", "clustered", "surface"])
def test_nearest_against_the_oracle(kind):
    rng = np.random.default_rng(0)
    if kind == "uniform":
        t, q, md = rng.uniform(-5, 5, (6000, 3)), rng.uniform(-6, 6, (4000, 3)), 0.6
    elif kind == "clustered":
        c = rng.uniform(-20, 20, (12, 3))
        t = c[rng.integers(0, 12, 6000)] + rng.normal(0, 0.5, (6000, 3))
        q = c[rng.integers(0, 12, 4000)] + rng.normal(0, 2.0, (4000, 3))
        md = 3.0
    else:
        t = _surface(rng, 8000)
        q = _surface(rng, 3000) + rng.normal(0, 0.2, (3000, 3))
        q[:300] = rng.uniform(-15, 15, (300, 3))                       # outliers, some beyond max_dist
        md = 2.0
    got, want = _check_nearest(q.astype(np.float32), t.astype(np.float32), md)
    assert np.isfinite(want).mean() > 0.5 and (~np.isfinite(want)).any()


def test_nearest_far_queries_empty_and_single_target():
    rng = np.random.default_rng(1)
    t = rng.uniform(0, 1, (500, 3)).astype(np.float32)
    far = np.concatenate([rng.uniform(50, 60, (100, 3)), [[4.0, 0.5, 0.5], [-3.0, -3.0, -3.0]]]).astype(np.float32)
    got, want = _check_nearest(far, t, 5.0)
    assert not np.isfinite(got[:100]).any() and np.isfinite(got[100])
    e = mvs_b200.nearest_distance(_g(far), torch.empty(0, 3, device=DEV), 5.0)
    assert e.shape == (102,) and bool(torch.isinf(e).all())
    one = np.array([[0.25, -0.5, 1.0]], np.float32)
    _check_nearest(rng.uniform(-3, 3, (1000, 3)).astype(np.float32), one, 2.5)
    assert mvs_b200.nearest_distance(torch.empty(0, 3, device=DEV), _g(t), 1.0).shape == (0,)


def _anchored(pts):
    """Targets with anchors at (0, 0, 0) and (20, 20, 20): with cell = 1 the cell of x is floor(x), 3 blocks of 8 cells per axis."""
    return np.concatenate([[[0.0, 0.0, 0.0], [20.0, 20.0, 20.0]], pts]).astype(np.float32)


def test_ring_search_does_not_stop_at_the_first_hit():
    # ring 0 holds A at 1.1, ring 1 holds B at 0.25: the first point met is not the nearest
    t = _anchored([[5.95, 5.95, 5.95], [4.8, 5.5, 5.5]])
    q = np.array([[5.05, 5.5, 5.5]], np.float32)
    g = evaluation.build_grid(_g(t), cell=1.0)
    assert g.cell == 1.0 and g.nb == [3, 3, 3]
    got = float(mvs_b200.nearest_distance(_g(q), _g(t), 8.0, grid=g)[0])
    first_hit = float(np.linalg.norm(q[0] - t[2].astype(np.float64)))          # the mutation: stop at the first hit
    assert abs(got - 0.25) <= 1e-6 * 0.25 and first_hit > 4 * 0.25


def test_nearest_beyond_a_coarse_block_edge():
    # A in fine ring 2 (found by the fine shells) at 4.24; B in ring 3, across the block edge x = 8, at 2.6 (found by the blocks)
    t = _anchored([[3.05, 3.05, 3.05], [8.1, 5.5, 5.5]])
    q = np.array([[5.5, 5.5, 5.5]], np.float32)
    g = evaluation.build_grid(_g(t), cell=1.0)
    got = float(mvs_b200.nearest_distance(_g(q), _g(t), 8.0, grid=g)[0])
    assert abs(got - 2.6) <= 1e-6 * 2.6
    # and a whole field of queries around the block edges against a sparse target, on the same grid
    rng = np.random.default_rng(2)
    t2 = _anchored(rng.uniform(0, 20, (40, 3)))
    q2 = rng.uniform(-2, 22, (3000, 3)).astype(np.float32)
    _check_nearest(q2, t2, 9.0, grid=evaluation.build_grid(_g(t2), cell=1.0))
    _check_nearest(q2, t2, 9.0)


def test_nearest_large_against_fp64_cdist():
    g = torch.Generator(device=DEV).manual_seed(3)
    n = 200_000
    t = torch.rand(n, 3, device=DEV, generator=g) * torch.tensor([10.0, 10.0, 1.0], device=DEV)
    q = torch.rand(n, 3, device=DEV, generator=g) * torch.tensor([12.0, 12.0, 2.0], device=DEV) - 1
    md = 0.3
    got = mvs_b200.nearest_distance(q, t, md).double()
    t64 = t.double()
    want = torch.empty(n, dtype=torch.float64, device=DEV)
    for a in range(0, n, 2048):
        want[a:a + 2048] = torch.cdist(q[a:a + 2048].double(), t64).min(1).values
    sure = (want - md).abs() / md >= 1e-4
    fin = want < md
    assert torch.equal(torch.isfinite(got)[sure], fin[sure])
    both = torch.isfinite(got) & fin
    assert float(((got[both] - want[both]).abs() / want[both].clamp_min(1e-30)).max()) <= 1e-6
    assert 0.3 < float(fin.double().mean()) < 1.0


def _lattice(rng, n, kind):
    """fp32 points on a lattice of 0.01: with dst = 0.205 no pair distance sqrt(k) * 0.01 comes within 2.9e-4 of dst."""
    if kind == "uniform":
        k = rng.integers(0, 200, (n, 3))
    elif kind == "clustered":
        c = rng.integers(0, 300, (n // 50, 3))
        k = c[rng.integers(0, len(c), n)] + np.rint(rng.normal(0, 15, (n, 3))).astype(int)
    else:                                   # exact duplicates
        base = rng.integers(0, 100, (n // 4, 3))
        k = base[rng.integers(0, len(base), n)]
    return (k * 0.01).astype(np.float32)


@pytest.mark.parametrize("kind", ["uniform", "clustered", "duplicates"])
def test_thinning_is_the_sequential_greedy_set(kind):
    rng = np.random.default_rng(4)
    x = _lattice(rng, 6000, kind)
    dst = 0.205
    order = rng.permutation(len(x))
    nb, margin = oracle.neighbours(x, dst)
    assert margin >= 1e-4                                               # no pair near dst: the comparison is meaningful
    want = oracle.thin_sequential(x, dst, order, nb)
    want_r, rounds_r = oracle.thin_rounds(x, dst, order, nb)
    assert np.array_equal(want, want_r)
    kept, rounds = evaluation.thin(_g(x), dst, order=order)
    assert kept.dtype == torch.int64 and np.array_equal(kept.cpu().numpy(), want)
    assert rounds == rounds_r
    print(f"{kind}: {len(want)} of {len(x)} kept in {rounds} rounds")


def test_thinning_edge_cases_and_seed():
    # all points within dst of each other: the first in order is kept
    rng = np.random.default_rng(5)
    x = (rng.uniform(0, 0.05, (500, 3))).astype(np.float32)
    order = rng.permutation(500)
    assert mvs_b200.thin_points(_g(x), 0.2, order=order).tolist() == [int(order[0])]
    # exact duplicates only
    d = np.repeat(np.array([[1.0, 2.0, 3.0], [1.0, 2.0, 3.3]], np.float32), 50, 0)
    o = np.arange(100)[::-1].copy()
    assert mvs_b200.thin_points(_g(d), 0.2, order=o).tolist() == [49, 99]
    # |p - q| <= dst inclusive: a chain 0.25 apart with dst = 0.25 (exact in fp32 and fp64); "<" would keep all four
    c = np.array([[0.0, 0, 0], [0.25, 0, 0], [0.5, 0, 0], [0.75, 0, 0]], np.float32)
    assert mvs_b200.thin_points(_g(c), 0.25, order=[0, 1, 2, 3]).tolist() == [0, 2]
    assert len(oracle.thin_sequential(c, np.nextafter(0.25, 0), [0, 1, 2, 3])) == 4      # the "<" mutation
    # seed reproducibility, and the seed's order is the CPU generator's permutation
    y = _lattice(rng, 3000, "uniform")
    a = mvs_b200.thin_points(_g(y), 0.205, seed=7)
    b = mvs_b200.thin_points(_g(y), 0.205, seed=7)
    assert torch.equal(a, b)
    perm = torch.randperm(3000, generator=torch.Generator().manual_seed(7)).numpy()
    assert np.array_equal(a.cpu().numpy(), oracle.thin_sequential(y, 0.205, perm))
    assert not torch.equal(a, mvs_b200.thin_points(_g(y), 0.205, seed=8))


def _scene(seed=11):
    """A hemisphere of radius 10 (ground truth, lattice-rounded data with noise and outliers), a ground patch of stl far from any
    data, a mask of 0.4-voxels with BB[0] offset so that no data coordinate sits near a half voxel."""
    rng = np.random.default_rng(seed)
    stl = _surface(rng, 12000)
    ground = np.stack([rng.uniform(-30, -20, 1500), rng.uniform(-5, 5, 1500), np.zeros(1500)], 1)
    lid = np.stack([rng.uniform(-5, 5, 500), rng.uniform(-5, 5, 500), np.full(500, 20.0)], 1)   # above the plane, not covered
    stl = np.concatenate([stl, ground, lid]).astype(np.float32)
    data = _surface(rng, 9000) * (1 + rng.normal(0, 0.002, (9000, 1)))
    data = np.concatenate([data, rng.uniform(-12, 12, (300, 3)) * [1, 1, 0.5] + [0, 0, 25],      # outliers outside the block grid
                           rng.uniform(-3, 3, (100, 3)) + [0, 0, 2]])                          # and inside the mask, far from stl
    data = (np.rint(data / 0.01) * 0.01).astype(np.float32)
    bb = np.array([[-11.003, -11.003, -1.003], [11.0, 11.0, 12.0]])
    res = 0.4
    shape = tuple(int(v) for v in np.floor((bb[1] - bb[0]) / res) + 1)
    mask = np.zeros(shape, bool)
    mask[:, : shape[1] * 3 // 4, :] = True
    plane = np.array([0.05, -0.02, 1.0, -1.2345])
    return data, stl, mask, bb, res, plane


def test_whole_evaluation_against_the_oracle():
    data, stl, mask, bb, res, plane = _scene()
    kw = dict(dst=0.205, max_dist=2.0, block=6.0)
    order = np.random.default_rng(7).permutation(len(data))
    want = oracle.evaluate(data, stl, mask, bb, res, plane, order=order, **kw)
    assert want["margin_thin"] >= 1e-4
    sure_d, sure_s = want["margin_data"] >= 1e-4, want["margin_stl"] >= 1e-4
    n0 = mvs_b200.launch_count()
    got = mvs_b200.evaluate_point_cloud(_g(data), _g(stl), torch.from_numpy(mask), bb, res, plane, order=order, return_details=True, **kw)
    launches = mvs_b200.launch_count() - n0
    # grid keys + cells for the thinning grid, count, list, one launch per round; keys + cells + search per direction
    assert launches == 4 + got["thin_rounds"] + 2 * 3
    assert np.array_equal(got["kept"].cpu().numpy(), want["kept"])
    for k in ("DataInMask",):
        assert np.array_equal(got[k].cpu().numpy()[sure_d], want[k][sure_d])
    assert np.array_equal(got["StlAbovePlane"].cpu().numpy()[sure_s], want["StlAbovePlane"][sure_s])
    for k, sure in (("Ddata", sure_d), ("Dstl", sure_s)):
        g, w = got[k].cpu().double().numpy(), want[k]
        assert np.array_equal(np.isfinite(g)[sure], np.isfinite(w)[sure])
        both = np.isfinite(g) & np.isfinite(w) & sure
        assert np.max(np.abs(g[both] - w[both]) / np.maximum(w[both], 1e-6)) <= 1e-6
    print({k: want[k] for k in ("accuracy", "completeness", "n_reduced", "n_accuracy", "n_completeness")},
          f"margins: data {want['margin_data'].min():.2e}, stl {want['margin_stl'].min():.2e}, thin {want['margin_thin']:.2e}")
    assert sure_d.all() and sure_s.all()                    # every margin is clear: statistics comparable to 1e-6
    for k in ("n", "n_reduced", "n_in_mask", "n_accuracy", "m", "m_above_plane", "n_completeness"):
        assert got[k] == want[k], k
    for k in ("accuracy", "completeness", "overall", "median_accuracy", "median_completeness"):
        assert abs(got[k] - want[k]) <= 1e-6 * abs(want[k]), k
    # every part of the protocol is exercised
    assert 0 < want["n_accuracy"] < want["n_in_mask"] < want["n_reduced"] < want["n"]
    assert 0 < want["n_completeness"] < want["m_above_plane"] < want["m"]
    # determinism
    again = mvs_b200.evaluate_point_cloud(_g(data), _g(stl), torch.from_numpy(mask), bb, res, plane, order=order, return_details=True, **kw)
    for k in ("kept", "Ddata", "Dstl", "DataInMask", "StlAbovePlane"):
        assert torch.equal(got[k], again[k])
    assert all(got[k] == again[k] or (np.isnan(got[k]) and np.isnan(again[k])) for k in ("accuracy", "completeness", "overall"))


def test_voxel_rounding_and_coverage_mutations():
    # (q - BB0) / Res at -0.5 and +2.5 on x: half away from zero gives -1 (outside) and 3; half to even gives 0 (inside) and 2
    bb = np.array([[0.0, 0.0, 0.0], [2.0, 2.0, 2.0]])
    res = 0.5
    mask = np.zeros((4, 4, 4), bool)
    mask[:3] = True                                       # index 3 on x is outside the mask, 0..2 inside
    q = np.array([[-0.25, 0.5, 0.5], [1.25, 0.5, 0.5]], np.float32)
    got = evaluation.in_mask(_g(q), torch.from_numpy(mask).to(DEV), bb, res).cpu().numpy()
    assert got.tolist() == [False, False]
    even = oracle.in_mask(q, mask, bb, res, rounding=np.round)[0]
    assert even.tolist() == [True, True]
    # the whole evaluation on the same points: nothing of them is in the mask, so accuracy has no sample
    stl = np.array([[-0.25, 0.5, 0.6], [1.25, 0.5, 0.6], [0.5, 0.5, 0.5]], np.float32)
    r = mvs_b200.evaluate_point_cloud(_g(q), _g(stl), mask, bb, res, [0, 0, 1, 0], dst=0.1, max_dist=1.0, block=0.8)
    assert r["n_in_mask"] == 0 and np.isnan(r["accuracy"]) and np.isnan(r["overall"])
    # coverage: R = floor(2 / 0.8) = 2 -> covered on [0, 2.4); the stl point at x = 2.45 lies 0.15 from a data point but gets
    # `block` (0.8 >= max_dist 0.5); without the quirk it would count
    q2 = np.array([[2.3, 0.5, 0.5], [0.5, 0.5, 0.5]], np.float32)
    s2 = np.array([[2.45, 0.5, 0.5], [0.55, 0.5, 0.5]], np.float32)
    r2 = mvs_b200.evaluate_point_cloud(_g(q2), _g(s2), mask, bb, res, [0, 0, 1, 0], dst=0.01, max_dist=0.5, block=0.8,
                                       return_details=True)
    assert r2["Dstl"].tolist()[0] == pytest.approx(0.8) and r2["n_completeness"] == 1
    assert r2["completeness"] == pytest.approx(0.05, rel=1e-6)


def test_end_to_end_fused_disk_and_convention_swap():
    s = fusion_oracle.analytic_scene(6, 48, 64, normal="sweep", seed=0)
    depth = torch.from_numpy(s["depth"].astype(np.float32))[:, None].to(DEV)
    conf = torch.ones_like(depth)
    colours = torch.rand(6, 3, 48, 64, device=DEV)
    src = [[j for j in range(6) if j != i] for i in range(6)]
    loose = dict(conf_min=0.0, reproj_px=1e3, rel_depth=1.0, min_views=1)
    r = s["radius"]
    n0, centre = s["n0"], s["centre"]
    a0 = np.cross(n0, [0.0, 1.0, 0.0])
    a0 /= np.linalg.norm(a0)
    b0 = np.cross(n0, a0)
    # the ground truth: the disk on a square lattice of 2e-4 r (mean distance to it 0.38 x 2e-4 r from a point on the plane)
    step = 2e-4 * r
    k = torch.arange(-int(r / step) - 1, int(r / step) + 2, device=DEV, dtype=torch.float64) * step
    u, v = torch.meshgrid(k, k, indexing="ij")
    on = u * u + v * v <= (r + 2 * step) ** 2
    u, v = u[on], v[on]
    t = lambda a: torch.as_tensor(a, dtype=torch.float64, device=DEV)        # noqa: E731
    gt = (t(centre) + u[:, None] * t(a0) + v[:, None] * t(b0)).float()
    del u, v, on
    bb = np.stack([gt.min(0).values.cpu().double().numpy() - 1, gt.max(0).values.cpu().double().numpy() + 1])
    mask = np.ones((4, 4, 4), bool)
    res = float((bb[1] - bb[0]).max() / 3)
    accs = {}
    for normal in ("sweep", "optical_axis"):
        xyz, _, _ = mvs_b200.fuse_depth_maps(depth, conf, colours, s["K"], s["R"], s["T"], src, normal=normal, **loose)
        out = mvs_b200.evaluate_point_cloud(xyz, gt, mask, bb, res, [0, 0, 0, 1], dst=0.02, max_dist=0.1 * r, block=4 * r)
        accs[normal] = out["accuracy"]
        print(normal, {k: out[k] for k in ("accuracy", "completeness", "n", "n_reduced", "n_accuracy")})
        if normal == "sweep":
            assert out["n_accuracy"] > 1000 and out["n_accuracy"] == out["n_reduced"]
            assert out["accuracy"] <= 1e-4 * r
    assert accs["optical_axis"] >= 10 * accs["sweep"]


def test_eval_dtu_tool_on_a_synthetic_directory(tmp_path):
    sio = pytest.importorskip("scipy.io")
    data, stl, mask, bb, res, plane = _scene(13)
    os.makedirs(tmp_path / "Points" / "stl")
    os.makedirs(tmp_path / "ObsMask")
    mvs_b200.write_ply(str(tmp_path / "Points" / "stl" / "stl003_total.ply"), stl)
    sio.savemat(str(tmp_path / "ObsMask" / "ObsMask3_10.mat"), {"ObsMask": mask, "BB": bb, "Res": res})
    sio.savemat(str(tmp_path / "ObsMask" / "Plane3.mat"), {"P": plane.reshape(4, 1)})
    ply = str(tmp_path / "scan3.ply")
    mvs_b200.write_ply(ply, data)
    out = str(tmp_path / "r.json")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "eval_dtu.py"), "--ply", ply, "--dtu", str(tmp_path), "--scan", "3",
                        "--out", out, "--dst", "0.205", "--max-dist", "2.0", "--block", "6.0", "--seed", "11"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = json.load(open(out))
    assert "accuracy" in r.stdout and "completeness" in r.stdout and "overall" in r.stdout
    order = torch.randperm(len(data), generator=torch.Generator().manual_seed(11)).numpy()
    want = oracle.evaluate(data, stl, mask, bb, res, plane, dst=0.205, max_dist=2.0, block=6.0, order=order)
    assert (want["margin_data"] >= 1e-4).all() and (want["margin_stl"] >= 1e-4).all()
    for k in ("accuracy", "completeness", "overall"):
        assert abs(got[k] - want[k]) <= 1e-6 * abs(want[k]), k
