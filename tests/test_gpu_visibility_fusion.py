"""Visibility fusion (mvs_b200.visibility_fusion, the VIS form of csrc/fusion.cu's check) on the GPU: exact against the fp64 oracle
(oracle/fusion_visibility.py) on a scene where fp32 cannot move a decision, the subset-and-bits property against fuse_depth_maps
on generic scenes, determinism, edge cases, launch counts, and an end-to-end evaluation of the analytic disk."""
import os

import numpy as np
import pytest
import torch

import fusion as oracle
import fusion_visibility as vis
import mvs_b200
from mvs_b200 import dtu, harness
from test_gpu_fusion import _noisy_scene, _sources, _t

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MUTATIONS = ("ignore_marks", "mark_all", "floor_marks", "marks_at_start")


def _orders(N, seed):
    return [list(range(N)), list(range(N - 1, -1, -1)), np.random.default_rng(seed).permutation(N).tolist()]


def _bits(x):
    return x.contiguous().view(torch.int32)


@pytest.mark.parametrize("normal", ["sweep", "optical_axis"])
def test_exact_on_the_layered_scene(normal):
    s = vis.layered_scene(12, 32, seed=0)
    args = (s["depth"], s["conf"], s["colours"], s["K"], s["R"], s["T"], s["sources"], normal)
    d, c, col = _t(s["depth"]), _t(s["conf"]), _t(s["colours"], 3)
    for order in _orders(12, seed=1):
        xyz_o, rgb_o, mask_o, _, _, _, used_o, min_margin = vis.visibility_fuse(*args, order)
        assert min_margin >= 1e-4                                 # no decision and no mark within reach of fp32 rounding
        xyz, rgb, masks = mvs_b200.visibility_fusion(d, c, col, s["K"], s["R"], s["T"], s["sources"], order=order, normal=normal)
        got = masks[:, 0].cpu().numpy()
        assert np.array_equal(got, mask_o) and xyz.shape == (mask_o.sum(), 3) and rgb.shape == xyz.shape
        extent = np.abs(xyz_o).max()
        assert np.abs(xyz.cpu().double().numpy() - xyz_o).max() <= 1e-6 * extent
        assert np.array_equal(rgb.cpu().numpy(), rgb_o.astype(np.float32))
        changed = {m: int((vis.visibility_fuse(*args, order, **{m: True})[2] != mask_o).sum()) for m in MUTATIONS}
        print(f"{normal} order {order[:3]}...: {mask_o.sum()} points, {used_o.sum()} marks, min margin {min_margin:.2e}, "
              f"kept pixels changed by the mutations {changed}")
        for m, n in changed.items():
            assert n >= 0.01 * mask_o.sum(), m


def _subset_and_bits(args, kw, k7, orders):
    """visibility_fusion under each order against fuse_depth_maps' result k7 -> the masks per order."""
    k_xyz, k_rgb, k_masks = k7
    out = []
    for order in orders:
        xyz, rgb, masks = mvs_b200.visibility_fusion(*args, order=order, **kw)
        assert not bool((masks & ~k_masks).any())
        sel = masks.reshape(-1)[k_masks.reshape(-1)]              # K7's rows (view-major, row-major) of the pixels kept here
        assert torch.equal(_bits(xyz), _bits(k_xyz[sel])) and torch.equal(_bits(rgb), _bits(k_rgb[sel]))
        assert torch.equal(masks[order[0]], k_masks[order[0]])
        assert 0 < xyz.shape[0] < k_xyz.shape[0]
        out.append(masks)
    return out


def _agreement(masks, depth, conf, colours, K, R, T, src, normal, order, kw, what):
    want = vis.visibility_fuse(depth, conf, colours, K, R, T, src, normal, order, **kw)[2]
    got = masks[:, 0].cpu().numpy()
    agree = float((got == want).mean())
    print(f"{what} order {order[:3]}...: masks agree with the oracle at {agree:.4%} of the pixels "
          f"({int((got != want).sum())} differ; {int(want.sum())} kept by the oracle, {int(got.sum())} by the GPU)")
    assert agree >= 0.99


@pytest.mark.parametrize("S,thr", [(4, dict()), (10, dict()), (10, dict(conf_min=0.6, reproj_px=0.5, rel_depth=0.003, min_views=2))])
@pytest.mark.parametrize("normal", ["sweep", "optical_axis"])
def test_properties_on_noisy_scenes(S, thr, normal):
    s, depth, conf, colours = _noisy_scene(S, normal=normal)
    N = depth.shape[0]
    src = _sources(N, S, seed=S)
    args = (_t(depth), _t(conf), _t(colours, 3), s["K"], s["R"], s["T"], src)
    kw = dict(normal=normal, **thr)
    orders = _orders(N, seed=S)
    masks = _subset_and_bits(args, kw, mvs_b200.fuse_depth_maps(*args, **kw), orders)
    for m, order in zip(masks, orders):
        _agreement(m, depth, conf, colours, s["K"], s["R"], s["T"], src, normal, order, thr, f"S={S} {normal}")


def test_properties_on_the_dtu_cameras_through_infer_scene():
    cams = dtu.read_cameras(os.path.join(ROOT, "tests", "golden", "dtu"), [0, 1, 2, 3])
    H, W, D = 128, 160, 32
    K = np.stack(cams["K"]).copy()
    K[:, :2] /= 4.0
    R, T = np.stack(cams["R"]), np.stack(cams["T"])
    d_min = np.array([np.asarray(d).item() for d in cams["d"]])
    d_int = np.array([np.asarray(d).item() for d in cams["d_int"]])
    torch.manual_seed(0)
    fz = mvs_b200.FrozenMVSNet(harness.MVSNet(D, 2.5).to(DEV).eval())
    img = torch.rand(4, 3, H, W, generator=torch.Generator().manual_seed(2))
    depth, conf, colours = mvs_b200.infer_scene(fz, img, K, R, T, d_min, d_int, cams["pairs"], n_views=3, batch_size=2)
    src = [list(p) for p in cams["pairs"]]
    kw = dict(conf_min=0.0, reproj_px=50.0, rel_depth=0.5, min_views=1)
    args = (depth, conf, colours, K, R, T, src)
    orders = _orders(4, seed=3)
    masks = _subset_and_bits(args, kw, mvs_b200.fuse_depth_maps(*args, **kw), orders)
    dn, cn, coln = (t.cpu().numpy() for t in (depth[:, 0], conf[:, 0], colours))
    for m, order in zip(masks, orders):
        _agreement(m, dn, cn, coln, K, R, T, src, "sweep", order, kw, "DTU cameras")


def test_determinism_edge_cases_and_launches():
    s, depth, conf, colours = _noisy_scene(5)
    N = depth.shape[0]
    src = _sources(N, 10, seed=5)
    d, c, col = _t(depth), _t(conf), _t(colours, 3)
    cam = (s["K"], s["R"], s["T"])
    n0 = mvs_b200.launch_count()
    a = mvs_b200.visibility_fusion(d, c, col, *cam, src, order=[3, 1, 0, 2] + list(range(4, N)))
    assert mvs_b200.launch_count() - n0 == N + 1                  # N checks and one compaction
    b = mvs_b200.visibility_fusion(d, c, col, *cam, src, order=[3, 1, 0, 2] + list(range(4, N)))
    assert a[0].shape[0] > 0 and all(torch.equal(x.view(torch.uint8), y.view(torch.uint8)) for x, y in zip(a, b))
    xyz, rgb, masks = mvs_b200.visibility_fusion(d, torch.zeros_like(c), col, *cam, src)
    assert xyz.shape == (0, 3) and rgb.shape == (0, 3) and not masks.any()
    # one view: no source can be consistent, so min_views = 0 keeps every valid pixel, as K7 does
    one = (d[:1], c[:1], col[:1], s["K"][:1], s["R"][:1], s["T"][:1], [[-1]])
    for mv in (0, 1):
        want = mvs_b200.fuse_depth_maps(*one, min_views=mv)
        got = mvs_b200.visibility_fusion(*one, min_views=mv)
        assert all(torch.equal(x.view(torch.uint8), y.view(torch.uint8)) for x, y in zip(got, want))
    assert want[0].shape[0] == 0 and mvs_b200.fuse_depth_maps(*one, min_views=0)[0].shape[0] > 0
    with pytest.raises(mvs_b200.MvsB200Error, match="lists itself"):
        mvs_b200.visibility_fusion(d, c, col, *cam, [[0]] + src[1:])


def test_end_to_end_on_the_analytic_disk():
    s = oracle.analytic_scene(6, 48, 64, normal="sweep", seed=0)
    depth = torch.from_numpy(s["depth"].astype(np.float32))[:, None].to(DEV)
    conf = torch.ones_like(depth)
    colours = torch.rand(6, 3, 48, 64, device=DEV)
    src = [[j for j in range(6) if j != i] for i in range(6)]
    loose = dict(conf_min=0.0, reproj_px=1e3, rel_depth=1.0, min_views=2)
    r, n0, centre = s["radius"], s["n0"], s["centre"]
    a0 = np.cross(n0, [0.0, 1.0, 0.0])
    a0 /= np.linalg.norm(a0)
    b0 = np.cross(n0, a0)
    step = 2e-4 * r                                               # the disk on a square lattice, as in test_gpu_evaluation
    k = torch.arange(-int(r / step) - 1, int(r / step) + 2, device=DEV, dtype=torch.float64) * step
    u, v = torch.meshgrid(k, k, indexing="ij")
    on = u * u + v * v <= (r + 2 * step) ** 2
    u, v = u[on], v[on]
    t = lambda a: torch.as_tensor(a, dtype=torch.float64, device=DEV)        # noqa: E731
    gt = (t(centre) + u[:, None] * t(a0) + v[:, None] * t(b0)).float()
    del u, v, on
    bb = np.stack([gt.min(0).values.cpu().double().numpy() - 1, gt.max(0).values.cpu().double().numpy() + 1])
    res = float((bb[1] - bb[0]).max() / 3)
    out = {}
    for name, fn in (("fuse_depth_maps", mvs_b200.fuse_depth_maps), ("visibility_fusion", mvs_b200.visibility_fusion)):
        xyz, _, _ = fn(depth, conf, colours, s["K"], s["R"], s["T"], src, **loose)
        out[name] = mvs_b200.evaluate_point_cloud(xyz, gt, np.ones((4, 4, 4), bool), bb, res, [0, 0, 0, 1], dst=0.02,
                                                  max_dist=0.1 * r, block=4 * r)
        out[name]["points"] = xyz.shape[0]
        print(name, {q: out[name][q] for q in ("points", "accuracy", "completeness", "n_reduced")})
    o = out["visibility_fusion"]
    assert o["accuracy"] <= 1e-4 * r
    assert o["points"] < out["fuse_depth_maps"]["points"]
    assert o["completeness"] <= 0.1                               # one pixel's footprint at depth 10 (f = 100)
