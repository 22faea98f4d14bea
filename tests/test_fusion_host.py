"""Geometry of the confidence / consistency-filter / fusion feature without a GPU: the sweep's planes pinned, the fp64 oracle on an
analytic scene, and the refusals that need no device."""
import numpy as np
import pytest
import torch

import fusion as oracle
import mvs_b200
from mvs_b200 import fusion


def _random_cameras(rng, n):
    Ks, Rs, Ts = [], [], []
    for _ in range(n):
        q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        q *= np.sign(np.linalg.det(q))
        Ks.append(np.array([[rng.uniform(80, 400), 0, rng.uniform(20, 80)], [0, rng.uniform(80, 400), rng.uniform(20, 60)], [0, 0, 1]]))
        Rs.append(q)
        Ts.append(rng.normal(scale=50.0, size=(3, 1)))
    return np.stack(Ks), np.stack(Rs), np.stack(Ts)


def test_sweep_unprojection_is_the_plane_sweep_homography():
    """Depth d_k under normal="sweep", unprojected in the reference and projected into view i, is H_i(d_k) p (DESIGN §1 a1-a3)."""
    rng = np.random.default_rng(0)
    K, R, T = _random_cameras(rng, 5)
    cams = fusion.camera_fields(K, R, T, "sweep")                 # the table the kernels read, before its fp32 rounding
    C = oracle.centres(R, T)
    n = R[0][:, 2]                                                # n = R_ref[:, 2], the third column
    x, y = rng.uniform(0, 160, 50), rng.uniform(0, 128, 50)
    p = np.stack([x, y, np.ones_like(x)])
    for d in (425.0, 611.5, 904.0):
        X = oracle.unproject(K[0], R[0], C[0], oracle.normals(R, "sweep")[0], x, y, np.full_like(x, d))
        r = cams[0, 12:21].reshape(3, 3) @ p                      # the table's own fields give the same point
        Xt = cams[0, 21:24][:, None] + d / (cams[0, 24:27] @ r) * r
        assert np.allclose(Xt.T, X, rtol=1e-12, atol=0)
        for i in range(1, 5):
            H = K[i] @ R[i] @ (np.eye(3) - np.outer(C[i] - C[0], n) / d) @ R[0].T @ np.linalg.inv(K[0])
            hp = H @ p
            u, v, _ = oracle.project(K[i], R[i], T[i], X)
            q = cams[i, 0:12].reshape(3, 4) @ np.vstack([X.T, np.ones_like(x)])
            for got in (np.stack([u, v]), q[:2] / q[2]):
                assert np.max(np.abs(got - hp[:2] / hp[2]) / np.abs(hp[:2] / hp[2])) < 1e-9


def _visible_count(s, i, sources):
    """Per pixel of view i: the sources in which the surface point lands inside the image with four on-surface depth taps."""
    K, R, T, depth = s["K"], s["R"], s["T"], s["depth"]
    h, w = depth.shape[1:]
    nv = oracle.normals(R, s["normal"])
    C = oracle.centres(R, T)
    y, x = np.meshgrid(np.arange(h, dtype=float), np.arange(w, dtype=float), indexing="ij")
    X = oracle.unproject(K[i], R[i], C[i], nv[i], x, y, np.where(depth[i] > 0, depth[i], 10.0))
    seen = np.zeros((h, w), int)
    for j in sources:
        u, v, z = oracle.project(K[j], R[j], T[j], X)
        inside = (z > 0) & (u >= 0) & (u <= w - 1) & (v >= 0) & (v <= h - 1)
        x0, y0 = np.floor(np.clip(u, 0, w - 1)).astype(int), np.floor(np.clip(v, 0, h - 1)).astype(int)
        x1, y1 = np.minimum(x0 + 1, w - 1), np.minimum(y0 + 1, h - 1)
        dj = depth[j] > 0
        seen += inside & dj[y0, x0] & dj[y0, x1] & dj[y1, x0] & dj[y1, x1]
    return np.where(depth[i] > 0, seen, 0)


@pytest.mark.parametrize("normal", ["sweep", "optical_axis"])
def test_oracle_on_an_analytic_scene(normal):
    s = oracle.analytic_scene(6, normal=normal, seed=1)
    s["normal"] = normal
    N = 6
    src = [[j for j in range(N) if j != i] for i in range(N)]
    conf = np.ones_like(s["depth"])
    colours = np.random.default_rng(0).uniform(size=(N, 3) + s["depth"].shape[1:])
    xyz, rgb, mask, count, fused, margin = oracle.fuse(s["depth"], conf, colours, s["K"], s["R"], s["T"], src, normal)
    for i in range(N):
        want = _visible_count(s, i, src[i]) >= 3
        assert np.array_equal(mask[i], want), f"view {i}: {np.sum(mask[i] != want)} pixels differ"
    assert mask.mean() > 0.5
    dist = xyz @ s["n0"]                                          # on the plane n0^T X = 0 ...
    assert np.abs(dist).max() < 1e-9 * 10
    assert np.linalg.norm(xyz - s["centre"], axis=1).max() <= s["radius"] + 1e-9       # ... inside the disk
    assert rgb.shape == xyz.shape
    # a corrupted patch in view 0 (depth 5 % too far) is rejected there
    bad = s["depth"].copy()
    bad[0, 10:30, 20:40] *= 1.05
    m2, _, _, _ = oracle.check(bad, conf, s["K"], s["R"], s["T"], src, normal)
    assert mask[0, 10:30, 20:40].mean() > 0.5 and not m2[0, 10:30, 20:40].any()
    # mutation: the other normal convention reads the same depth maps as other surfaces
    other = "optical_axis" if normal == "sweep" else "sweep"
    m3, _, _, _ = oracle.check(s["depth"], conf, s["K"], s["R"], s["T"], src, other)
    assert m3.mean() * 10 <= mask.mean()


def test_oracle_confidence_window():
    prob = np.array([0.1, 0.2, 0.3, 0.25, 0.15]).reshape(1, 5, 1, 1) * np.ones((1, 5, 1, 4))
    depths = np.array([[10.0, 12.0, 14.0, 16.0, 18.0]])
    depth = np.array([[[10.5, 13.0, 18.0, np.nan]]])                 # k0 = 0, 1, 4 (D-1), non-finite
    c = oracle.confidence(prob, depth, depths)[0, 0]
    assert np.allclose(c[:3], [0.1 + 0.2 + 0.3, 0.1 + 0.2 + 0.3 + 0.25, 0.25 + 0.15]) and np.isnan(c[3])
    assert oracle.confidence(prob[:, :1], depth, depths[:, :1])[0, 0, 0] == 1.0


def test_refusals_without_a_gpu():
    N, h, w = 3, 8, 10
    K = torch.eye(3).repeat(N, 1, 1)
    R = torch.eye(3).repeat(N, 1, 1)
    T = torch.zeros(N, 3, 1)
    d, c, col = torch.ones(N, 1, h, w), torch.ones(N, 1, h, w), torch.zeros(N, 3, h, w)
    src = [[1, 2], [0, 2], [0, 1]]
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        mvs_b200.fuse_depth_maps(d, c, col, K, R, T, src)
    with pytest.raises(mvs_b200.MvsB200Error, match="normal"):
        fusion.camera_fields(K, R, T, normal="z")
    with pytest.raises(mvs_b200.MvsB200Error, match="at most 16"):
        fusion.source_table([list(range(17))] * 20, 20)
    with pytest.raises(mvs_b200.MvsB200Error, match="source ids"):
        fusion.source_table([[1], [3], [0]], 3)
    with pytest.raises(mvs_b200.MvsB200Error, match="one source list"):
        fusion.source_table([[1], [0]], 3)
    with pytest.raises(mvs_b200.MvsB200Error, match="values"):
        fusion.camera_fields(torch.eye(3), R, T)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA"):
        fusion.resize_colours(col, 4, 5)


def test_write_ply_header_and_colour_rule(tmp_path):
    xyz = np.array([[0.0, 1.0, 2.0], [3.0, 4.0, 5.0]], np.float32)
    rgb = np.array([[0.0, 0.5, 1.0], [-0.2, 1.3, 0.5 / 255.0]])
    p = tmp_path / "t.ply"
    mvs_b200.write_ply(str(p), xyz, rgb)
    raw = p.read_bytes()
    head, body = raw.split(b"end_header\n")
    assert b"format binary_little_endian 1.0" in head and b"element vertex 2" in head
    rec = np.frombuffer(body, dtype=[("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("r", "u1"), ("g", "u1"), ("b", "u1")])
    assert np.array_equal(np.stack([rec["x"], rec["y"], rec["z"]], 1), xyz)
    assert rec["r"].tolist() == [0, 0] and rec["g"].tolist() == [128, 255] and rec["b"].tolist() == [255, 0]
