"""fp64 numpy restatement of visibility fusion (mvs_b200.visibility_fusion, DESIGN §4 "K7 confidence and fusion"): the consistency
test of oracle/fusion.py run view after view in a given order, with a state `used` that suppresses references already absorbed by
an earlier view's point.  Written from the definition, not from the kernel.  Test infrastructure only.

For reference view r, in order: a pixel with used[r] set is not a reference (mask false); every other pixel runs fusion.check's
test; a kept pixel sets used[j, floor(v + 1/2), floor(u + 1/2)] for every consistent source j, (u, v) its projection into j.  The
points are fusion.fuse's points of the kept pixels, view-major in index order, row-major."""
from __future__ import annotations

import numpy as np

from fusion import centres, normals, project, unproject


def _check_view(i, depth, conf, K, R, T, C, nv, sources_i, conf_min, reproj_px, rel_depth):
    """fusion.check for reference view i alone -> (valid, count, fused, margin, per source (j, inside, good, u, v)).  The formulas
    and the margin are those of fusion.check, line for line."""
    N, h, w = depth.shape
    y, x = np.meshgrid(np.arange(h, dtype=np.float64), np.arange(w, dtype=np.float64), indexing="ij")
    usable = np.isfinite(depth) & (depth > 0)
    rel = lambda a, thr: np.abs(a - thr) / abs(thr)          # noqa: E731
    d = depth[i]
    with np.errstate(invalid="ignore"):
        valid = (conf[i] >= conf_min) & usable[i]
        margin = np.where(usable[i] & np.isfinite(conf[i]), rel(conf[i], conf_min), np.inf)
    X = unproject(K[i], R[i], C[i], nv[i], x, y, np.where(valid, d, 1.0))
    total = np.where(valid, d, 0.0)
    cnt = np.zeros((h, w), np.int64)
    per_source = []
    for j in np.asarray(sources_i).reshape(-1):
        j = int(j)
        if j < 0:
            continue
        with np.errstate(invalid="ignore", divide="ignore"):
            u, v, z = project(K[j], R[j], T[j], X)
            inside = valid & (z > 0) & (u >= 0) & (u <= w - 1) & (v >= 0) & (v <= h - 1)
        m_b = np.minimum.reduce([np.abs(u) / w, np.abs(u - (w - 1)) / w, np.abs(v) / h, np.abs(v - (h - 1)) / h])
        uc, vc = np.clip(np.nan_to_num(u), 0, w - 1), np.clip(np.nan_to_num(v), 0, h - 1)
        x0, y0 = np.floor(uc).astype(np.int64), np.floor(vc).astype(np.int64)
        x1, y1 = np.minimum(x0 + 1, w - 1), np.minimum(y0 + 1, h - 1)
        dj, uj = depth[j], usable[j]
        taps_ok = uj[y0, x0] & uj[y0, x1] & uj[y1, x0] & uj[y1, x1]
        xm, ym = np.clip(x0 - 1, 0, w - 1), np.clip(y0 - 1, 0, h - 1)
        xp, yp = np.clip(x0 + 2, 0, w - 1), np.clip(y0 + 2, 0, h - 1)
        near_bad = ~(uj[ym, xm] & uj[ym, xp] & uj[yp, xm] & uj[yp, xp] & uj[ym, x0] & uj[ym, x1] & uj[yp, x0] & uj[yp, x1]
                     & uj[y0, xm] & uj[y1, xm] & uj[y0, xp] & uj[y1, xp] & taps_ok)
        fu, fv = uc - x0, vc - y0
        m_t = np.where(near_bad, np.minimum.reduce([fu, 1 - fu, fv, 1 - fv]), np.inf)
        ok = inside & taps_ok
        ds = (1 - fv) * ((1 - fu) * dj[y0, x0] + fu * dj[y0, x1]) + fv * ((1 - fu) * dj[y1, x0] + fu * dj[y1, x1])
        Xs = unproject(K[j], R[j], C[j], nv[j], uc, vc, np.where(ok, ds, 1.0))
        with np.errstate(invalid="ignore", divide="ignore"):
            ur, vr, _ = project(K[i], R[i], T[i], Xs)
            dr = (Xs - C[i]) @ nv[i]
            dist = np.hypot(ur - x, vr - y)
            reld = np.abs(dr - d) / d
            good = ok & (dist < reproj_px) & (reld < rel_depth)
        m_src = np.where(valid & (z > 0), m_b, np.inf)
        m_src = np.minimum(m_src, np.where(inside, m_t, np.inf))
        m_src = np.minimum(m_src, np.where(ok, np.minimum(rel(dist, reproj_px), rel(reld, rel_depth)), np.inf))
        margin = np.minimum(margin, np.nan_to_num(m_src, nan=0.0))
        cnt += good
        total = total + np.where(good, dr, 0.0)
        per_source.append((j, inside, good, uc, vc))
    fused = np.where(valid, total / (1 + cnt), d)
    return valid, cnt, fused, margin, per_source


def visibility_fuse(depth, conf, colours, K, R, T, sources, normal="sweep", order=None, *, ignore_marks=False, mark_all=False,
                    floor_marks=False, marks_at_start=False, conf_min=0.8, reproj_px=1.0, rel_depth=0.01, min_views=3):
    """depth, conf [N, h, w]; colours [N, 3, h, w]; K, R [N, 3, 3]; T [N, 3(, 1)]; sources [N, S] (-1 pads); order a permutation of
    range(N) (default index order) -> (xyz [M, 3], rgb [M, 3], mask, count, fused, margin, used, min_margin).

    mask, count, fused, margin [N, h, w] as fusion.fuse (margin inf at pixels that were no reference); used bool [N, h, w], the
    final state.  min_margin: the smallest of every decision's margin (fusion.check's, at the pixels that were references) and of
    the rounding margin min(|frac(u) - 1/2|, |frac(v) - 1/2|) (pixels) of every mark written.

    Mutations (each a plausible mistake the tests must be able to see): ignore_marks (no view reads the marks: fusion.fuse's
    result), mark_all (every source the point projects inside is marked, consistent or not), floor_marks (floor(u) in place of
    floor(u + 1/2)), marks_at_start (every view reads the marks as they were before the first view ran: a one-launch shortcut)."""
    depth = np.asarray(depth, np.float64)
    conf = np.asarray(conf, np.float64)
    K, R = np.asarray(K, np.float64), np.asarray(R, np.float64)
    T = np.asarray(T, np.float64).reshape(-1, 3)
    N, h, w = depth.shape
    C, nv = centres(R, T), normals(R, normal)
    order = list(range(N)) if order is None else [int(i) for i in order]
    assert sorted(order) == list(range(N)), order
    used = np.zeros((N, h, w), bool)
    start = used.copy()
    mask = np.zeros((N, h, w), bool)
    count = np.zeros((N, h, w), np.int64)
    fused = depth.copy()
    margin = np.full((N, h, w), np.inf)
    min_margin = np.inf
    for i in order:
        seen = start if marks_at_start else used
        reference = np.ones((h, w), bool) if ignore_marks else ~seen[i]
        valid, cnt, fu, mg, per_source = _check_view(i, depth, conf, K, R, T, C, nv, np.asarray(sources[i]), conf_min, reproj_px,
                                                     rel_depth)
        keep = reference & valid & (cnt >= min_views)
        mask[i] = keep
        count[i] = np.where(reference & valid, cnt, 0)
        fused[i] = np.where(reference, fu, depth[i])
        margin[i] = np.where(reference, mg, np.inf)
        for j, inside, good, u, v in per_source:
            sel = keep & (inside if mark_all else good)
            if floor_marks:
                xm, ym = np.floor(u), np.floor(v)
            else:
                xm, ym = np.floor(u + 0.5), np.floor(v + 0.5)
                if sel.any():
                    rm = np.minimum(np.abs(u - np.floor(u) - 0.5), np.abs(v - np.floor(v) - 0.5))
                    min_margin = min(min_margin, float(rm[sel].min()))
            used[j, ym[sel].astype(np.int64), xm[sel].astype(np.int64)] = True
    min_margin = min(min_margin, float(margin.min()))
    xyz, rgb = [], []
    for i in range(N):
        yy, xx = np.nonzero(mask[i])
        xyz.append(unproject(K[i], R[i], C[i], nv[i], xx.astype(np.float64), yy.astype(np.float64), fused[i][yy, xx]))
        rgb.append(np.asarray(colours[i], np.float64)[:, yy, xx].T)
    return np.concatenate(xyz).reshape(-1, 3), np.concatenate(rgb).reshape(-1, 3), mask, count, fused, margin, used, min_margin


def layered_scene(n_views=12, size=32, seed=0):
    """A scene on which fp32 reproduces the fp64 decisions exactly: an occluding square (|x|, |y| <= 1) at depth 8 over a background
    plane at depth 16, seen by n_views <= 16 cameras on the plane z = 0, each rotated by a multiple of 90 degrees about its optical
    axis (+z, so both depth normals are +z), with f = 64 and the principal point on a pixel (size // 2) of a square image.

    Each camera centre coordinate is (k + m / 16) / 16 with m distinct across views, so a disparity f dC / Z between two views is
    a multiple of 1/32 pixel that is never integer nor 1/2 (by at least 1/32 at depth 8 and 1/64 at depth 16).  With depth
    ratio 2 a disparity cannot be 1/4 or 3/4 on both layers.  Every quantity on a same-layer round trip is a dyadic rational, so
    fp32 computes it exactly.  Three views carry a corrupted 4 x 4 patch (depth 12), one view a NaN band (depth and confidence),
    confidences are drawn from {0.5, 0.95}, and each view has 3 to 10 sources padded with -1 to 10.
    -> dict K, R, T [N, 3, 1], depth, conf [N, h, w] float32, colours [N, 3, h, w] float32, sources [N, 10]."""
    assert n_views <= 16
    rng = np.random.default_rng(seed)
    c = size // 2
    K = np.array([[64.0, 0, c], [0, 64.0, c], [0, 0, 1]])
    mx, my = rng.permutation(16)[:n_views], rng.permutation(16)[:n_views]
    kx, ky = rng.integers(-6, 7, n_views), rng.integers(-6, 7, n_views)
    Cs = np.stack([(kx + mx / 16) / 16, (ky + my / 16) / 16, np.zeros(n_views)], 1)
    rot = {0: [[1, 0], [0, 1]], 1: [[0, -1], [1, 0]], 2: [[-1, 0], [0, -1]], 3: [[0, 1], [-1, 0]]}
    Rs = []
    for q in rng.integers(0, 4, n_views):
        Rm = np.eye(3)
        Rm[:2, :2] = rot[int(q)]
        Rs.append(Rm)
    R = np.stack(Rs)
    T = -R @ Cs[:, :, None]
    Ks = np.repeat(K[None], n_views, 0)
    y, x = np.meshgrid(np.arange(size, dtype=np.float64), np.arange(size, dtype=np.float64), indexing="ij")
    depth = np.empty((n_views, size, size))
    for i in range(n_views):
        X = unproject(K, R[i], Cs[i], np.array([0.0, 0.0, 1.0]), x, y, np.full_like(x, 8.0))
        depth[i] = np.where((np.abs(X[..., 0]) <= 1) & (np.abs(X[..., 1]) <= 1), 8.0, 16.0)
    conf = rng.choice([0.5, 0.95], size=depth.shape, p=[0.15, 0.85])
    for i in range(3):
        py, px = rng.integers(0, size - 4, 2)
        depth[i, py:py + 4, px:px + 4] = 12.0
    depth[3, 5:8] = np.nan
    conf[3, 5:8] = np.nan
    sources = []
    for i in range(n_views):
        k = int(rng.integers(3, 11))
        r = rng.choice([j for j in range(n_views) if j != i], k, replace=False).tolist()
        sources.append(r + [-1] * (10 - k))
    colours = rng.uniform(size=(n_views, 3, size, size))
    return {"K": Ks, "R": R, "T": T, "depth": depth.astype(np.float32), "conf": conf.astype(np.float32),
            "colours": colours.astype(np.float32), "sources": np.array(sources)}
