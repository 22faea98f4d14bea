"""fp64 numpy restatement of the photometric confidence and of MVSNet's consistency filter and fusion (§4.2), written from the
definitions (DESIGN §4 "K7 confidence and fusion"), not from the kernels.  Test infrastructure only.

Geometry: depth d at pixel p = (x, y, 1) of view i is X = C_i + d / (n_i^T r) r, r = R_i^T K_i^-1 p; the depth of X in view j is
n_j^T (X - C_j); n = R[:, 2] ("sweep") or R[2, :] ("optical_axis")."""
from __future__ import annotations

import numpy as np


def normals(R, normal):
    R = np.asarray(R, np.float64)
    if normal == "sweep":
        return R[:, :, 2].copy()
    if normal == "optical_axis":
        return R[:, 2, :].copy()
    raise ValueError(normal)


def centres(R, T):
    R, T = np.asarray(R, np.float64), np.asarray(T, np.float64).reshape(-1, 3, 1)
    return (-np.transpose(R, (0, 2, 1)) @ T)[:, :, 0]


def unproject(K, R, C, n, x, y, d):
    """Pixels (x, y) with depths d (arrays of one shape) of one view -> points [..., 3]."""
    p = np.stack([x, y, np.ones_like(x)], -1).astype(np.float64)
    r = p @ (R.T @ np.linalg.inv(K)).T
    return C + (d / (r @ n))[..., None] * r


def project(K, R, T, X):
    """Points [..., 3] -> (u, v, z) of K (R X + T)."""
    q = (X @ R.T + T.reshape(3)) @ K.T
    return q[..., 0] / q[..., 2], q[..., 1] / q[..., 2], q[..., 2]


def confidence(prob, depth, depths):
    """prob [B, D, h, w], depth [B, h, w], depths [B, D] -> fp64 [B, h, w].  The plane index t = (depth - d_0) / (d_1 - d_0) is
    formed in fp32 as the definition states (so that floor(t) is the one of the fp32 inputs); the sum is exact in fp64."""
    prob = np.asarray(prob, np.float64)
    B, D, h, w = prob.shape
    depth = np.asarray(depth, np.float32)
    out = np.empty((B, h, w))
    for b in range(B):
        dv = np.asarray(depths[b], np.float32)
        if D == 1:
            out[b] = 1.0
        else:
            with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
                t = (depth[b] - dv[0]) / np.float32(dv[1] - dv[0])
            k0 = np.floor(t.astype(np.float64))
            s = np.zeros((h, w))
            for o in (-1, 0, 1, 2):
                with np.errstate(invalid="ignore"):
                    k = k0 + o
                    ok = np.isfinite(k) & (k >= 0) & (k <= D - 1)
                ki = np.where(ok, k, 0).astype(np.int64)
                pk = np.take_along_axis(prob[b], ki[None], 0)[0]
                s += np.where(ok, pk, 0.0)
            out[b] = np.where(np.isfinite(t) & np.isfinite(s), s, np.nan)
        out[b][~np.isfinite(depth[b])] = np.nan
    return out


def check(depth, conf, K, R, T, sources, normal="sweep", conf_min=0.8, reproj_px=1.0, rel_depth=0.01, min_views=3):
    """depth, conf [N, h, w]; K, R [N, 3, 3]; T [N, 3(, 1)]; sources [N, S] (-1 pads) ->
    (mask bool, count int, fused fp64, margin fp64), each [N, h, w].  margin: the smallest relative distance of any quantity the
    decision of that pixel depends on to its threshold (conf / conf_min, the bounds of the image, the integer steps of the tap
    position where they change which taps are read and one of the candidates is unusable, |p' - p| / reproj_px, the relative depth
    difference / rel_depth); inf where nothing is near."""
    depth = np.asarray(depth, np.float64)
    conf = np.asarray(conf, np.float64)
    K, R = np.asarray(K, np.float64), np.asarray(R, np.float64)
    T = np.asarray(T, np.float64).reshape(-1, 3)
    N, h, w = depth.shape
    C, nv = centres(R, T), normals(R, normal)
    y, x = np.meshgrid(np.arange(h, dtype=np.float64), np.arange(w, dtype=np.float64), indexing="ij")
    usable = np.isfinite(depth) & (depth > 0)
    mask = np.zeros((N, h, w), bool)
    count = np.zeros((N, h, w), np.int64)
    fused = depth.copy()
    margin = np.full((N, h, w), np.inf)
    rel = lambda a, thr: np.abs(a - thr) / abs(thr)          # noqa: E731
    for i in range(N):
        d = depth[i]
        with np.errstate(invalid="ignore"):
            valid = (conf[i] >= conf_min) & usable[i]
            margin[i] = np.where(usable[i] & np.isfinite(conf[i]), rel(conf[i], conf_min), np.inf)
        dd = np.where(valid, d, 1.0)
        X = unproject(K[i], R[i], C[i], nv[i], x, y, dd)
        total = np.where(valid, d, 0.0)
        cnt = np.zeros((h, w), np.int64)
        for j in np.asarray(sources[i]).reshape(-1):
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
            # where u or v sits near an integer the tap set may differ in fp32; that matters only if an unusable depth is near
            xm, ym = np.clip(x0 - 1, 0, w - 1), np.clip(y0 - 1, 0, h - 1)
            xp, yp = np.clip(x0 + 2, 0, w - 1), np.clip(y0 + 2, 0, h - 1)
            near_bad = ~(uj[ym, xm] & uj[ym, xp] & uj[yp, xm] & uj[yp, xp] & uj[ym, x0] & uj[ym, x1] & uj[yp, x0] & uj[yp, x1]
                         & uj[y0, xm] & uj[y1, xm] & uj[y0, xp] & uj[y1, xp] & taps_ok)
            fu, fv = uc - x0, vc - y0
            m_t = np.where(near_bad, np.minimum.reduce([fu, 1 - fu, fv, 1 - fv]), np.inf)
            ok = inside & taps_ok
            ax, ay = uc - x0, vc - y0
            ds = (1 - ay) * ((1 - ax) * dj[y0, x0] + ax * dj[y0, x1]) + ay * ((1 - ax) * dj[y1, x0] + ax * dj[y1, x1])
            ds = np.where(ok, ds, 1.0)
            Xs = unproject(K[j], R[j], C[j], nv[j], uc, vc, ds)
            with np.errstate(invalid="ignore", divide="ignore"):
                ur, vr, _ = project(K[i], R[i], T[i], Xs)
                dr = (Xs - C[i]) @ nv[i]
                dist = np.hypot(ur - x, vr - y)
                reld = np.abs(dr - d) / d
                good = ok & (dist < reproj_px) & (reld < rel_depth)
            m_src = np.where(valid & (z > 0), m_b, np.inf)
            m_src = np.minimum(m_src, np.where(valid & inside, m_t, np.inf))
            m_src = np.minimum(m_src, np.where(ok, np.minimum(rel(dist, reproj_px), rel(reld, rel_depth)), np.inf))
            margin[i] = np.minimum(margin[i], np.nan_to_num(m_src, nan=0.0))
            cnt += good
            total = total + np.where(good, dr, 0.0)
        count[i] = cnt
        mask[i] = valid & (cnt >= min_views)
        fused[i] = np.where(valid, total / (1 + cnt), d)
    return mask, count, fused, margin


def fuse(depth, conf, colours, K, R, T, sources, normal="sweep", **thresholds):
    """-> (xyz [M, 3], rgb [M, 3], mask, count, fused, margin); points view-major, row-major."""
    mask, count, fused, margin = check(depth, conf, K, R, T, sources, normal, **thresholds)
    R = np.asarray(R, np.float64)
    T = np.asarray(T, np.float64).reshape(-1, 3)
    C, nv = centres(R, T), normals(R, normal)
    N, h, w = mask.shape
    xyz, rgb = [], []
    for i in range(N):
        yy, xx = np.nonzero(mask[i])
        xyz.append(unproject(np.asarray(K[i], np.float64), R[i], C[i], nv[i], xx.astype(np.float64), yy.astype(np.float64),
                             fused[i][yy, xx]))
        rgb.append(np.asarray(colours[i], np.float64)[:, yy, xx].T)
    return np.concatenate(xyz).reshape(-1, 3), np.concatenate(rgb).reshape(-1, 3), mask, count, fused, margin


def analytic_scene(n_cams=6, h=48, w=64, normal="sweep", seed=0, radius=4.0, focal=100.0):
    """A disk of radius `radius` on the plane n0^T X = 0 seen by n_cams cameras, each 10 units in front of it, rotated about n0
    and shifted along the plane, with K at (h, w) and focal length `focal` pixels.  Every camera's depth normal (R[:, 2] for "sweep", R[2, :] for "optical_axis")
    is n0, so each depth map is exactly 10 on the disk (bilinear sampling is then exact) and 0 elsewhere.
    -> dict K, R, T [N, 3, 1], depth [N, h, w], n0, centre, radius."""
    rng = np.random.default_rng(seed)
    n0 = np.array([0.6, -0.3, 1.0])
    n0 /= np.linalg.norm(n0)
    a0 = np.cross(n0, [0.0, 1.0, 0.0])
    a0 /= np.linalg.norm(a0)
    b0 = np.cross(n0, a0)
    K = np.array([[focal, 0, (w - 1) / 2], [0, focal, (h - 1) / 2], [0, 0, 1]])
    centre = 0.5 * a0 - 0.3 * b0
    Ks, Rs, Ts = [], [], []
    for th in np.linspace(-0.8, 0.8, n_cams) + rng.uniform(-0.05, 0.05, n_cams):
        a, b = np.cos(th) * a0 + np.sin(th) * b0, -np.sin(th) * a0 + np.cos(th) * b0
        Rc = np.stack([a, b, n0], 1)                       # columns a, b, n0: R[:, 2] = n0, det = +1
        R = Rc if normal == "sweep" else Rc.T
        axis = R[2]                                        # the optical axis, aimed at the disk's centre (+ a jitter)
        hit = -10.0 * n0 + 10.0 / (axis @ n0) * axis
        C = -10.0 * n0 - hit + centre + rng.uniform(-0.8, 0.8) * a0 + rng.uniform(-0.8, 0.8) * b0
        Ks.append(K.copy()); Rs.append(R); Ts.append((-R @ C).reshape(3, 1))
    K, R, T = np.stack(Ks), np.stack(Rs), np.stack(Ts)
    C = centres(R, T)
    nv = normals(R, normal)
    y, x = np.meshgrid(np.arange(h, dtype=np.float64), np.arange(w, dtype=np.float64), indexing="ij")
    depth = np.zeros((n_cams, h, w))
    for i in range(n_cams):
        X = unproject(K[i], R[i], C[i], nv[i], x, y, np.full((h, w), 10.0))
        on = np.linalg.norm(X - centre, axis=-1) <= radius
        depth[i] = np.where(on, 10.0, 0.0)
    return {"K": K, "R": R, "T": T, "depth": depth, "n0": n0, "centre": centre, "radius": radius}
