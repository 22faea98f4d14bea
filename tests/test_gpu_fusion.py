"""Photometric confidence (K4), consistency filter and point-cloud fusion (K7) on the GPU against the fp64 oracle
(oracle/fusion.py), FrozenMVSNet(return_confidence=True), and infer_scene -> fuse_depth_maps -> write_ply end to end."""
import os

import numpy as np
import pytest
import torch

import fusion as oracle
import mvs_b200
from mvs_b200 import _lib, dtu, fusion, harness, ops
from mvs_b200.ops import _stream

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------------------------ confidence
def _conf_case(B, D, h, w, seed):
    """Logits whose depth lands on every plane, the first and last included, plus one all-NaN column per sample."""
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(B, 1, D, h, w, generator=g) * 3
    peak = torch.randint(0, D, (B, h, w), generator=g)
    logits.scatter_add_(2, peak[:, None, None], torch.full((B, 1, 1, h, w), 8.0))
    # depth exactly d_0: all mass on plane 0 (rank(0) = 0 is kept).  Depth exactly d_{D-1}: the kept planes are {rank(j) : j < 5}
    # (depthmap.py's positional mask), so plane D-1 is kept when plane 0 ranks last, and then carries all the mass
    logits[:, 0, 0, 0, :3] += 100.0
    logits[:, 0, D - 1, 0, 3:6] += 100.0
    logits[:, 0, 0, 0, 3:6] -= 100.0
    logits[:, :, :, 1, 1] = float("nan")
    d_batch = (425.0 + 2.5 * torch.arange(D, dtype=torch.float32)).repeat(B, 1).reshape(B, D, 1, 1) + 10.0 * torch.arange(B).reshape(B, 1, 1, 1)
    return logits.to(DEV), d_batch


@pytest.mark.parametrize("B,D,h,w", [(2, 48, 16, 20), (1, 1, 8, 9), (3, 5, 7, 33), (1, 192, 32, 40)])
def test_confidence_fused_and_standalone_against_the_oracle(B, D, h, w):
    logits, d_batch = _conf_case(B, D, h, w, seed=D)
    prob, ranks, depth, conf = ops.softmax_depth_confidence(logits, d_batch)
    # prob, ranks and depth are those of the plain entry and depth_from_ranks
    n_keep = min(5, D)
    p0 = torch.empty(B, D, h, w, device=DEV)
    r0 = torch.empty(B, n_keep, h, w, dtype=torch.int32, device=DEV)
    d0 = torch.empty(B, h, w, device=DEV)
    dv = d_batch.reshape(B, D).contiguous().to(DEV)
    _lib.call("mvsb200_softmax_depth_fwd", logits.contiguous().data_ptr(), 1, None, p0.data_ptr(), r0.data_ptr(), None, B, D, h, w, 5, _stream())
    _lib.call("mvsb200_depth_from_ranks", p0.data_ptr(), r0.data_ptr(), dv.data_ptr(), d0.data_ptr(), B, D, h, w, n_keep, _stream())
    assert torch.equal(prob.reshape(B, D, h, w).view(torch.int32), p0.view(torch.int32))
    assert torch.equal(ranks, r0)
    assert torch.equal(depth.reshape(B, h, w).view(torch.int32), d0.view(torch.int32))
    # standalone == fused, bit for bit (NaN included)
    conf2 = mvs_b200.depth_confidence(prob, depth, d_batch)
    assert torch.equal(conf.view(torch.int32), conf2.view(torch.int32))
    want = oracle.confidence(prob.reshape(B, D, h, w).cpu().numpy(), depth.reshape(B, h, w).cpu().numpy(), d_batch.reshape(B, D).numpy())
    got = conf.reshape(B, h, w).cpu().double().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.isnan(got[:, 1, 1]).all()
    ok = ~np.isnan(want)
    assert np.max(np.abs(got[ok] - want[ok]) / np.maximum(np.abs(want[ok]), 1e-30)) <= 1e-6
    if D == 1:
        assert (got[ok] == 1.0).all()
    else:   # the window met both ends of the sweep
        t = (depth.reshape(B, h, w).cpu().numpy() - d_batch[:, 0, 0, 0].numpy()[:, None, None]) / 2.5
        assert (np.floor(t[ok]) == 0).any() and (np.floor(t[ok]) == D - 1).any()


def test_frozen_model_confidence_leaves_the_depth_maps_bit_identical():
    B, V, H, W, D = 2, 3, 64, 80, 32
    torch.manual_seed(0)
    m = harness.MVSNet(D, 480.0 / D).to(DEV).eval()
    K, R, T = harness.synthetic_cameras(B, V, H // 4, W // 4, seed=0)
    img = torch.randn(B * V, 3, H, W, generator=torch.Generator().manual_seed(1)).to(DEV)
    d_min, d_int = torch.full((B, 1, 1, 1), 425.0), torch.ones(B, 1, 1, 1)
    fz = mvs_b200.FrozenMVSNet(m)
    i0, r0 = fz(img, K, R, T, d_min, d_int, B, V)
    i1, r1, conf = fz(img, K, R, T, d_min, d_int, B, V, return_confidence=True)
    assert torch.equal(i0, i1) and torch.equal(r0, r1) and conf.shape == i0.shape
    c = conf[torch.isfinite(conf)]
    assert c.numel() > 0 and bool(((c >= 0) & (c <= 1.0 + 1e-6)).all())


# ------------------------------------------------------------------------------------------------------------------ fusion
def _noisy_scene(seed, N=12, h=48, w=64, normal="sweep", noise=2e-3):
    s = oracle.analytic_scene(N, h, w, normal=normal, seed=seed)
    rng = np.random.default_rng(seed + 100)
    depth = s["depth"] * (1 + noise * rng.standard_normal(s["depth"].shape))
    conf = rng.uniform(0.5, 1.0, depth.shape)
    colours = rng.uniform(size=(N, 3, h, w))
    return s, depth.astype(np.float32), conf.astype(np.float32), colours.astype(np.float32)


def _sources(N, S, seed):
    rng = np.random.default_rng(seed)
    rows = []
    for i in range(N):
        k = int(rng.integers(1, S + 1))                          # 1 .. S real sources, padded with -1 to S
        r = rng.choice([j for j in range(N) if j != i], k, replace=False).tolist()
        rows.append(r + [-1] * (S - k))
    return rows


def _t(a, c=1):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).reshape(a.shape[0], c, *a.shape[-2:]).to(DEV)


@pytest.mark.parametrize("S,thr", [(1, dict(min_views=1)), (4, dict()), (10, dict()), (10, dict(conf_min=0.6, reproj_px=0.5, rel_depth=0.003, min_views=2))])
@pytest.mark.parametrize("normal", ["sweep", "optical_axis"])
def test_fusion_against_the_oracle(S, thr, normal):
    s, depth, conf, colours = _noisy_scene(S, normal=normal)
    N = depth.shape[0]
    src = _sources(N, S, seed=S)
    xyz, rgb, masks = mvs_b200.fuse_depth_maps(_t(depth), _t(conf), _t(colours, 3), s["K"], s["R"], s["T"], src, normal=normal, **thr)
    m_g, c_g, f_g = fusion.check_consistency(_t(depth), _t(conf), s["K"], s["R"], s["T"], src, normal=normal, **thr)
    oxyz, orgb, om, oc, of, margin = oracle.fuse(depth, conf, colours, s["K"], s["R"], s["T"], src, normal, **thr)
    sure = margin >= 1e-4
    print(f"S={S} {normal}: {1 - sure.mean():.4%} of the pixels within 1e-4 of a threshold, {om.mean():.3f} kept")
    assert 1 - sure.mean() < 0.01
    gm = m_g[:, 0].cpu().numpy()
    assert torch.equal(masks, m_g)
    assert np.array_equal(gm[sure], om[sure])
    valid = (conf >= thr.get("conf_min", 0.8)) & (depth > 0)
    assert np.array_equal(c_g[:, 0].cpu().numpy()[sure & valid], oc[sure & valid])
    fg = f_g[:, 0].cpu().double().numpy()
    both = sure & valid
    assert np.max(np.abs(fg[both] - of[both]) / of[both]) <= 1e-5
    assert om.sum() > 100
    # the points of the pixels both keep, in order: xyz where the oracle's margin is >= 1e-4 (elsewhere a source near a threshold
    # may count on one side only, which moves the fused depth), rgb everywhere
    assert xyz.shape == (gm.sum(), 3) and rgb.shape == xyz.shape
    both_k = (gm & om).reshape(-1)
    sel_g, sel_o = both_k[gm.reshape(-1)], both_k[om.reshape(-1)]
    sure_g, sure_o = sure.reshape(-1)[gm.reshape(-1)][sel_g], sure.reshape(-1)[om.reshape(-1)][sel_o]
    assert np.array_equal(sure_g, sure_o)
    gx = xyz.cpu().double().numpy()[sel_g]
    err = np.abs(gx - oxyz[sel_o]).max(1)
    extent = np.abs(oxyz).max()
    print(f"  xyz error / extent: {err[sure_g].max() / extent:.2e} at margin >= 1e-4, "
          f"{err[~sure_g].max(initial=0) / extent:.2e} at the {int((~sure_g).sum())} kept points below it")
    assert err[sure_g].max() <= 1e-5 * extent
    assert np.array_equal(rgb.cpu().numpy()[sel_g], orgb[sel_o].astype(np.float32))


def test_fusion_edge_cases_and_determinism():
    s, depth, conf, colours = _noisy_scene(3)
    N = depth.shape[0]
    src = _sources(N, 10, seed=3)
    args = (s["K"], s["R"], s["T"], src)
    xyz, rgb, masks = mvs_b200.fuse_depth_maps(_t(depth), _t(np.zeros_like(conf)), _t(colours, 3), *args)
    assert xyz.shape == (0, 3) and rgb.shape == (0, 3) and not masks.any()
    # the val_dmin0 pattern: NaN depth and confidence over whole regions give no point there
    d2, c2 = depth.copy(), conf.copy()
    d2[:, 5:20] = np.nan
    c2[:, 5:20] = np.nan
    xyz, rgb, masks = mvs_b200.fuse_depth_maps(_t(d2), _t(c2), _t(colours, 3), *args)
    assert xyz.shape[0] > 0 and not masks[:, :, 5:20].any() and bool(torch.isfinite(xyz).all())
    a = mvs_b200.fuse_depth_maps(_t(depth), _t(conf), _t(colours, 3), *args)
    b = mvs_b200.fuse_depth_maps(_t(depth), _t(conf), _t(colours, 3), *args)
    assert all(torch.equal(x.view(torch.uint8), y.view(torch.uint8)) for x, y in zip(a, b))


def _read_ply(path):
    with open(path, "rb") as f:
        raw = f.read()
    head, body = raw.split(b"end_header\n", 1)
    lines = head.decode().splitlines()
    assert lines[0] == "ply" and lines[1] == "format binary_little_endian 1.0"
    n = int([l for l in lines if l.startswith("element vertex")][0].split()[-1])
    props = [l.split() for l in lines if l.startswith("property")]
    dt = [(p[2], "<f4" if p[1] == "float" else "u1") for p in props]
    return np.frombuffer(body, dtype=dt, count=n)


def test_infer_scene_fuse_and_write_ply_end_to_end(tmp_path):
    base = os.path.join(ROOT, "tests", "golden", "dtu")
    cams = dtu.read_cameras(base, [0, 1, 2, 3])
    H, W, D = 128, 160, 32
    K = np.stack(cams["K"]).copy()
    K[:, :2] /= 4.0                                               # feature resolution
    R, T = np.stack(cams["R"]), np.stack(cams["T"])
    d_min = np.array([np.asarray(d).item() for d in cams["d"]])
    d_min[2] = 440.0                                              # a second depth range: views 2 and 0/1/3 run in separate batches
    d_int = np.array([np.asarray(d).item() for d in cams["d_int"]])
    torch.manual_seed(0)
    m = harness.MVSNet(D, 2.5).to(DEV).eval()
    fz = mvs_b200.FrozenMVSNet(m)
    img = torch.rand(4, 3, H, W, generator=torch.Generator().manual_seed(2))
    n0 = mvs_b200.launch_count()
    depth, conf, colours = mvs_b200.infer_scene(fz, img, K, R, T, d_min, d_int, cams["pairs"], n_views=3, batch_size=2)
    assert depth.shape == (4, 1, 32, 40) and conf.shape == depth.shape and colours.shape == (4, 3, 32, 40)
    assert mvs_b200.launch_count() > n0
    # each view equals a lone run of that view with its own sources and depth range
    for i in (0, 2):
        idx = [i] + [int(j) for j in cams["pairs"][i][:2]]
        kk, rr, tt = (torch.from_numpy(a[idx]).float() for a in (K, R, T))
        ini, ref, cf = fz(img[idx].to(DEV), kk, rr, tt, torch.full((1, 1, 1, 1), d_min[i]), torch.full((1, 1, 1, 1), d_int[i]), 1, 3,
                          return_confidence=True)
        assert torch.equal(ref, depth[i:i + 1]) and torch.equal(cf.view(torch.int32), conf[i:i + 1].view(torch.int32))
    d2, c2, col2 = mvs_b200.infer_scene(fz, img, K, R, T, d_min, d_int, cams["pairs"], n_views=3, batch_size=2)
    assert torch.equal(d2, depth) and torch.equal(c2.view(torch.int32), conf.view(torch.int32)) and torch.equal(col2, colours)
    src = [list(p) for p in cams["pairs"]]
    xyz, rgb, masks = mvs_b200.fuse_depth_maps(depth, conf, colours, K, R, T, src, conf_min=0.0, reproj_px=50.0, rel_depth=0.5,
                                               min_views=1)
    assert xyz.shape[0] == int(masks.sum()) and rgb.shape == xyz.shape
    xyz2, rgb2, _ = mvs_b200.fuse_depth_maps(depth, conf, colours, K, R, T, src, conf_min=0.0, reproj_px=50.0, rel_depth=0.5,
                                             min_views=1)
    assert torch.equal(xyz, xyz2) and torch.equal(rgb, rgb2)
    p = tmp_path / "scene.ply"
    mvs_b200.write_ply(str(p), xyz, rgb)
    rec = _read_ply(str(p))
    assert len(rec) == xyz.shape[0]
    assert np.array_equal(np.stack([rec["x"], rec["y"], rec["z"]], 1), xyz.cpu().numpy())
    assert np.array_equal(np.stack([rec["red"], rec["green"], rec["blue"]], 1),
                          np.clip(np.rint(rgb.cpu().double().numpy() * 255), 0, 255).astype(np.uint8))


def test_colours_are_the_refine_input_resize():
    img = torch.rand(3, 3, 37, 53, generator=torch.Generator().manual_seed(0)).to(DEV)
    got = fusion.resize_colours(img, 9, 13)
    want = torch.nn.functional.interpolate(img, (9, 13), mode="bilinear", align_corners=False)
    assert float((got - want).abs().max()) < 1e-6
