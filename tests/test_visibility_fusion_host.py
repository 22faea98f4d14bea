"""Visibility fusion without a GPU: the fp64 oracle (oracle/fusion_visibility.py) against a literal pixel-by-pixel loop of its
definition, its marks-ignored mutation against oracle.fuse, and the refusals of mvs_b200.visibility_fusion that need no device."""
import math

import numpy as np
import pytest
import torch

import fusion as oracle
import fusion_visibility as vis
import mvs_b200


def _literal(depth, conf, K, R, T, sources, normal, order, conf_min, reproj_px, rel_depth, min_views):
    """The definition, one pixel and one source at a time -> (mask, fused, used)."""
    N, h, w = depth.shape
    T = T.reshape(N, 3)
    C, n = oracle.centres(R, T), oracle.normals(R, normal)

    def unproject(i, x, y, d):
        r = R[i].T @ np.linalg.inv(K[i]) @ np.array([x, y, 1.0])
        return C[i] + d / (n[i] @ r) * r

    def project(j, X):
        q = K[j] @ (R[j] @ X + T[j])
        return q[0] / q[2], q[1] / q[2], q[2]

    def usable(v):
        return math.isfinite(v) and v > 0

    used = np.zeros((N, h, w), bool)
    mask = np.zeros((N, h, w), bool)
    fused = np.full((N, h, w), np.nan)
    for r in order:
        for y in range(h):
            for x in range(w):
                d = float(depth[r, y, x])
                if used[r, y, x] or not (conf[r, y, x] >= conf_min and usable(d)):
                    continue
                X = unproject(r, x, y, d)
                count, total, marks = 0, d, []
                for j in sources[r]:
                    if j < 0:
                        continue
                    u, v, z = project(j, X)
                    if not (z > 0 and 0 <= u <= w - 1 and 0 <= v <= h - 1):
                        continue
                    x0, y0 = math.floor(u), math.floor(v)
                    x1, y1 = min(x0 + 1, w - 1), min(y0 + 1, h - 1)
                    taps = [float(depth[j, a, b]) for a, b in ((y0, x0), (y0, x1), (y1, x0), (y1, x1))]
                    if not all(usable(t) for t in taps):
                        continue
                    ax, ay = u - x0, v - y0
                    ds = (1 - ay) * ((1 - ax) * taps[0] + ax * taps[1]) + ay * ((1 - ax) * taps[2] + ax * taps[3])
                    Xs = unproject(j, u, v, ds)
                    ur, vr, _ = project(r, Xs)
                    dr = n[r] @ (Xs - C[r])
                    if math.hypot(ur - x, vr - y) < reproj_px and abs(dr - d) / d < rel_depth:
                        count += 1
                        total += dr
                        marks.append((j, math.floor(v + 0.5), math.floor(u + 0.5)))
                if count >= min_views:
                    mask[r, y, x] = True
                    fused[r, y, x] = total / (1 + count)
                    for j, a, b in marks:
                        used[j, a, b] = True
    return mask, fused, used


def _tiny(seed, normal):
    s = oracle.analytic_scene(5, 12, 16, normal=normal, seed=seed, focal=20.0)
    rng = np.random.default_rng(seed)
    depth = s["depth"] * (1 + 2e-3 * rng.standard_normal(s["depth"].shape))
    depth[1, 2:4, 3:6] = np.nan
    conf = rng.uniform(0.5, 1.0, depth.shape)
    colours = rng.uniform(size=(5, 3, 12, 16))
    sources = [[j for j in rng.permutation(5).tolist() if j != i][:int(rng.integers(2, 5))] for i in range(5)]
    sources = [r + [-1] * (4 - len(r)) for r in sources]
    return s, depth, conf, colours, sources


@pytest.mark.parametrize("normal", ["sweep", "optical_axis"])
@pytest.mark.parametrize("order", [[0, 1, 2, 3, 4], [4, 2, 0, 3, 1]])
def test_oracle_is_the_literal_loop(normal, order):
    s, depth, conf, colours, sources = _tiny(3, normal)
    thr = dict(conf_min=0.6, reproj_px=1.0, rel_depth=0.01, min_views=2)
    xyz, rgb, mask, count, fused, margin, used, min_margin = vis.visibility_fuse(depth, conf, colours, s["K"], s["R"], s["T"],
                                                                                 sources, normal, order, **thr)
    lm, lf, lu = _literal(depth, conf, s["K"], s["R"], s["T"], sources, normal, order, **thr)
    assert min_margin > 1e-9                       # both are fp64: the summation orders differ only in the last bits
    assert mask.sum() > 50 and used.sum() > 50 and (~mask & (depth > 0)).sum() > 50
    assert np.array_equal(mask, lm) and np.array_equal(used, lu)
    assert np.allclose(fused[mask], lf[mask], rtol=1e-12, atol=0)
    assert xyz.shape == (mask.sum(), 3) and np.array_equal(rgb, np.concatenate([colours[i][:, mask[i]].T for i in range(5)]))


@pytest.mark.parametrize("normal", ["sweep", "optical_axis"])
def test_oracle_with_marks_ignored_is_fuse(normal):
    s, depth, conf, colours, sources = _tiny(4, normal)
    args = (depth, conf, colours, s["K"], s["R"], s["T"], sources, normal)
    want = oracle.fuse(*args, min_views=2)
    for order in ([0, 1, 2, 3, 4], [3, 1, 4, 0, 2]):
        got = vis.visibility_fuse(*args, order, ignore_marks=True, min_views=2)
        for g, w in zip(got[:6], want):
            assert np.array_equal(g, w, equal_nan=True)
        assert got[6].any()                                 # the marks are written, only not read
        assert vis.visibility_fuse(*args, order, min_views=2)[2].sum() < want[2].sum()


def test_refusals_without_a_device():
    depth, conf, colours = torch.ones(3, 1, 4, 5), torch.ones(3, 1, 4, 5), torch.ones(3, 3, 4, 5)
    K = np.repeat(np.array([[[10.0, 0, 2], [0, 10, 2], [0, 0, 1]]]), 3, 0)
    R, T = np.repeat(np.eye(3)[None], 3, 0), np.zeros((3, 3, 1))
    ok = [[1, 2], [0, 2], [0, 1]]
    with pytest.raises(mvs_b200.MvsB200Error, match="view 1 lists itself"):
        mvs_b200.visibility_fusion(depth, conf, colours, K, R, T, [[1, 2], [0, 1], [0, -1]])
    for bad in ([0, 1], [0, 1, 1], [0, 1, 3], [2, 1, 0, 0], [0.0, 1.0, 2.0], [[0, 1, 2]]):
        with pytest.raises(mvs_b200.MvsB200Error, match="permutation of range"):
            mvs_b200.visibility_fusion(depth, conf, colours, K, R, T, ok, order=bad)
    with pytest.raises(mvs_b200.MvsB200Error, match="CUDA tensor"):
        mvs_b200.visibility_fusion(depth, conf, colours, K, R, T, ok, order=torch.tensor([2, 0, 1]))
    with pytest.raises(mvs_b200.MvsB200Error, match="at most 16 sources"):
        mvs_b200.visibility_fusion(depth, conf, colours, K, R, T, [list(range(17))] * 3)
