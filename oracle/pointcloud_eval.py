"""fp64 numpy restatement of the DTU point-cloud evaluation (BaseEvalMain_web.m, reducePts_haa.m, MaxDistCP.m, ComputeStat_web.m),
written from the protocol (DESIGN §4 "K8 point-cloud evaluation"), not from the kernels.  numpy only (no scipy).  Test
infrastructure only.

Every decision comes with a relative margin to its threshold (as oracle/fusion.py does): |d - dst| / dst per thinning pair,
|d - max_dist| / max_dist per distance, the distance of (q - BB[0]) / Res to the nearest half-integer per voxel index, the
distance to the block grid's faces over `block` per coverage test, and |P.x + P3| / (|P0 x| + |P1 y| + |P2 z| + |P3|) per plane
test (whose threshold is zero)."""
from __future__ import annotations

import numpy as np


def _f64(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64) if np.asarray(a).dtype == np.float32 else np.asarray(a, np.float64)


def nearest(query, target, chunk=2048):
    """Brute force: the distance from every query point to its nearest target point, fp64 -> [n] (inf for an empty target)."""
    q, t = _f64(query).reshape(-1, 3), _f64(target).reshape(-1, 3)
    out = np.full(q.shape[0], np.inf)
    if t.shape[0] == 0:
        return out
    for a in range(0, q.shape[0], chunk):
        qa = q[a:a + chunk]
        best = np.full(qa.shape[0], np.inf)
        for b in range(0, t.shape[0], 8192):
            tb = t[b:b + 8192]
            d2 = ((qa[:, None, :] - tb[None, :, :]) ** 2).sum(-1)
            best = np.minimum(best, d2.min(1))
        out[a:a + chunk] = np.sqrt(best)
    return out


def capped(d, max_dist):
    """-> (distance with +inf where it is not < max_dist, relative margin |d - max_dist| / max_dist)."""
    d = np.asarray(d, np.float64)
    return np.where(d < max_dist, d, np.inf), np.abs(d - max_dist) / max_dist


def neighbours(xyz, dst, chunk=2048):
    """All pairs within dst (inclusive, fp64) -> (list of neighbour index arrays, smallest relative margin |d - dst| / dst over
    all pairs)."""
    x = _f64(xyz).reshape(-1, 3)
    n = x.shape[0]
    nb, margin = [], np.inf
    for a in range(0, n, chunk):
        d = np.sqrt(((x[a:a + chunk, None, :] - x[None, :, :]) ** 2).sum(-1))
        margin = min(margin, float(np.min(np.abs(d - dst) / dst)) if d.size else np.inf)
        close = d <= dst
        for k in range(close.shape[0]):
            row = np.nonzero(close[k])[0]
            nb.append(row[row != a + k])
    return nb, margin


def thin_sequential(xyz, dst, order, nbrs=None):
    """reducePts_haa in the given visiting order: a visited point still present is kept and removes its neighbours within dst
    -> kept indices ascending."""
    n = len(order)
    nbrs = neighbours(xyz, dst)[0] if nbrs is None else nbrs
    present = np.ones(n, bool)
    keep = np.zeros(n, bool)
    for i in np.asarray(order):
        if present[i]:
            keep[i] = True
            present[nbrs[i]] = False
            present[i] = False
    return np.nonzero(keep)[0]


def thin_rounds(xyz, dst, order, nbrs=None):
    """The parallel greedy rounds: an undecided point becomes kept when every lower-ranked neighbour is removed, removed when one
    is kept; every round reads the previous states -> (kept indices ascending, rounds)."""
    n = len(order)
    nbrs = neighbours(xyz, dst)[0] if nbrs is None else nbrs
    rank = np.empty(n, np.int64)
    rank[np.asarray(order)] = np.arange(n)
    lower = [nb[rank[nb] < rank[i]] for i, nb in enumerate(nbrs)]
    state = np.zeros(n, np.int8)                                     # 0 undecided, 1 kept, 2 removed
    rounds = 0
    while (state == 0).any():
        new = state.copy()
        for i in np.nonzero(state == 0)[0]:
            s = state[lower[i]]
            if (s == 1).any():
                new[i] = 2
            elif (s == 2).all():
                new[i] = 1
        state = new
        rounds += 1
        if rounds > n:
            raise RuntimeError("no progress")
    return np.nonzero(state == 1)[0], rounds


def covered(q, bb, block):
    """MaxDistCP's block grid -> (covered bool [n], margin: distance to the nearest grid face on any axis over block)."""
    q, bb = _f64(q).reshape(-1, 3), np.asarray(bb, np.float64).reshape(2, 3)
    R = np.floor((bb[1] - bb[0]) / block)
    hi = bb[0] + (R + 1) * block
    cov = ((q >= bb[0]) & (q < hi)).all(1)
    margin = np.minimum(np.abs(q - bb[0]), np.abs(q - hi)).min(1) / block
    return cov, margin


def covered_literal(q, bb, block):
    """A literal transcription of MaxDistCP's triple loop over blocks: the points some block visits."""
    q, bb = _f64(q).reshape(-1, 3), np.asarray(bb, np.float64).reshape(2, 3)
    R = np.floor((bb[1] - bb[0]) / block).astype(int)
    look = np.zeros(q.shape[0], int)
    for x in range(R[0] + 1):
        for y in range(R[1] + 1):
            for z in range(R[2] + 1):
                low = bb[0] + np.array([x, y, z]) * block
                high = low + block
                idx = np.nonzero((q[:, 0] >= low[0]) & (q[:, 1] >= low[1]) & (q[:, 2] >= low[2])
                                 & (q[:, 0] < high[0]) & (q[:, 1] < high[1]) & (q[:, 2] < high[2]))[0]
                look[idx] += 1
    return look > 0


def round_half_away(x):
    x = np.asarray(x, np.float64)
    return np.sign(x) * np.floor(np.abs(x) + 0.5)


def in_mask(q, obs_mask, bb, res, rounding=round_half_away):
    """DataInMask -> (bool [n], margin: the distance of (q - BB[0]) / Res to the nearest half-integer, smallest over the axes)."""
    q, bb = _f64(q).reshape(-1, 3), np.asarray(bb, np.float64).reshape(2, 3)
    obs_mask = np.asarray(obs_mask, bool)
    x = (q - bb[0]) / res
    i = rounding(x)
    inside = ((i >= 0) & (i < np.array(obs_mask.shape))).all(1)
    ii = np.where(inside[:, None], i, 0).astype(np.int64)
    m = inside & obs_mask[ii[:, 0], ii[:, 1], ii[:, 2]]
    margin = np.abs(np.abs(x - np.floor(x)) - 0.5).min(1)
    return m, margin


def above_plane(s, plane):
    """StlAbovePlane -> (bool [m], margin |s| / (sum of the magnitudes of its terms))."""
    s, P = _f64(s).reshape(-1, 3), np.asarray(plane, np.float64).reshape(4)
    v = s @ P[:3] + P[3]
    scale = np.abs(s * P[:3]).sum(1) + abs(P[3])
    return v > 0, np.abs(v) / np.maximum(scale, 1e-300)


def mean_median(v):
    v = np.asarray(v, np.float64)
    if v.size == 0:
        return float("nan"), float("nan")
    return float(v.mean()), float(np.median(v))


def evaluate(xyz, stl, obs_mask, bb, res, plane, dst=0.2, max_dist=20.0, block=60.0, order=None):
    """The whole protocol -> dict of the statistics, counts, per-point arrays and margins (keys as evaluate_point_cloud's, plus
    margin_thin, margin_data [n_reduced] and margin_stl [m])."""
    x = _f64(xyz).reshape(-1, 3)
    s = _f64(stl).reshape(-1, 3)
    nbrs, m_thin = neighbours(x, dst)
    kept = thin_sequential(x, dst, order, nbrs)
    q = x[kept]
    dd, m_dd = capped(nearest(q, s), max_dist)
    ds, m_ds = capped(nearest(s, q), max_dist)
    cq, m_cq = covered(q, bb, block)
    cs, m_cs = covered(s, bb, block)
    dd = np.where(cq, dd, block)
    ds = np.where(cs, ds, block)
    din, m_in = in_mask(q, obs_mask, bb, res)
    sab, m_pl = above_plane(s, plane)
    sel_a = din & (dd < max_dist)
    sel_c = sab & (ds < max_dist)
    acc, med_a = mean_median(dd[sel_a])
    comp, med_c = mean_median(ds[sel_c])
    return {"accuracy": acc, "completeness": comp, "overall": (acc + comp) / 2, "median_accuracy": med_a,
            "median_completeness": med_c, "n": x.shape[0], "n_reduced": q.shape[0], "n_in_mask": int(din.sum()),
            "n_accuracy": int(sel_a.sum()), "m": s.shape[0], "m_above_plane": int(sab.sum()), "n_completeness": int(sel_c.sum()),
            "kept": kept, "Ddata": dd, "Dstl": ds, "DataInMask": din, "StlAbovePlane": sab, "margin_thin": m_thin,
            "margin_data": np.minimum.reduce([m_dd, m_cq, m_in]), "margin_stl": np.minimum.reduce([m_ds, m_cs, m_pl])}
