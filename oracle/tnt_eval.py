"""fp64 numpy restatement of the Tanks and Temples evaluation (the toolbox's EvaluateHisto and get_f1_score_histo2 with the Open3D
functions they call), written from the contract in DESIGN §4 "K9 Tanks and Temples evaluation", not from the kernels.  numpy, and
scipy.spatial.cKDTree for the nearest distances.  Test infrastructure only.

Steps 1-3 use numpy's elementwise fp64 ufuncs, one rounding per operation in the contract's order, so that their bits are the
contract's.  Every decision comes with a relative margin (as oracle/pointcloud_eval.py does): the axis bounds and the polygon's
vertex v-levels and crossing nodes over the polygon's extent, and the distances to tau, to the histogram edges and to the search cap
over tau.  Mutation switches reproduce plausible mistakes; the tests show that each one changes a result."""
from __future__ import annotations

import numpy as np

AXES = {"x": (1, 2, 0), "y": (0, 2, 1), "z": (0, 1, 2)}
INT_MAX = 2 ** 31 - 1


def _f64(a):
    return np.asarray(a, dtype=np.float64).reshape(-1, 3)


def transform(p, A):
    """p' = A [p; 1]: component i = ((A[i,0] x + A[i,1] y) + A[i,2] z) + A[i,3]."""
    p, A = _f64(p), np.asarray(A, np.float64)
    return np.stack([((A[i, 0] * p[:, 0] + A[i, 1] * p[:, 1]) + A[i, 2] * p[:, 2]) + A[i, 3] for i in range(3)], 1)


def crop(p, axis, axis_min, axis_max, polygon, closed_both=False, exclusive_bounds=False):
    """Open3D's CropInPolygon -> (inside bool [n], margin [n]).  closed_both: <= at both ends of an edge's v-range (mutation);
    exclusive_bounds: p_w on axis_min / axis_max is outside (mutation).  margin: the smallest of |p_w - axis bound|, |p_v - b_i,v|
    over the vertices and |node - p_u| over the crossing nodes, over the polygon's largest extent."""
    p = _f64(p)
    u, v, w = AXES[axis.lower()]
    b = np.asarray(polygon, np.float64).reshape(-1, 3)
    k = b.shape[0]
    pu, pv, pw = p[:, u], p[:, v], p[:, w]
    if exclusive_bounds:
        out_w = (pw <= axis_min) | (pw >= axis_max)
    else:
        out_w = (pw < axis_min) | (pw > axis_max)
    below = np.zeros(p.shape[0], np.int64)
    m_node = np.full(p.shape[0], np.inf)
    for i in range(k):
        j = (i + 1) % k
        biu, biv, bju, bjv = b[i, u], b[i, v], b[j, u], b[j, v]
        if closed_both:
            cross = ((biv <= pv) & (bjv >= pv)) | ((bjv <= pv) & (biv >= pv))
        else:
            cross = ((biv < pv) & (bjv >= pv)) | ((bjv < pv) & (biv >= pv))
        with np.errstate(divide="ignore", invalid="ignore"):
            node = biu + (pv - biv) / (bjv - biv) * (bju - biu)
        below += cross & (node < pu)
        m_node = np.where(cross, np.minimum(m_node, np.abs(node - pu)), m_node)
    inside = ~out_w & (below % 2 == 1)
    scale = max(float(np.ptp(b[:, u])), float(np.ptp(b[:, v])), abs(axis_max - axis_min), 1e-300)
    m_w = np.minimum(np.abs(pw - axis_min), np.abs(pw - axis_max))
    m_v = np.abs(pv[:, None] - b[None, :, v]).min(1)
    return inside, np.minimum.reduce([m_w, m_v, m_node]) / scale


def inside_winding(p, axis, axis_min, axis_max, polygon):
    """An independent point-in-polygon test: the winding number of the polygon around (p_u, p_v) (sum of signed angles), for
    points away from the edges."""
    p = _f64(p)
    u, v, w = AXES[axis.lower()]
    b = np.asarray(polygon, np.float64).reshape(-1, 3)
    du, dv = b[None, :, u] - p[:, u, None], b[None, :, v] - p[:, v, None]
    a = np.arctan2(dv, du)
    d = np.diff(np.concatenate([a, a[:, :1]], 1), axis=1)
    d = (d + np.pi) % (2 * np.pi) - np.pi
    wind = np.rint(d.sum(1) / (2 * np.pi)).astype(int)
    return (wind != 0) & (p[:, w] >= axis_min) & (p[:, w] <= axis_max)


def _sequential_sums(x, starts, counts):
    """Per segment, the sum of its rows added one after another from 0 (vectorised over the position in the segment)."""
    s = np.zeros((len(starts), x.shape[1]))
    for pos in range(int(counts.max()) if len(counts) else 0):
        live = counts > pos
        s[live] = s[live] + x[starts[live] + pos]
    return s


def _pairwise(x):
    n = len(x)
    return x[0] if n == 1 else _pairwise(x[:n // 2]) + _pairwise(x[n // 2:])


def voxel_down_sample(p, voxel, summation="sequential", divide=True, half_offset=True):
    """Open3D's VoxelDownSample -> (mean fp64 [v, 3] in ascending key order, counts [v], keys [v]).  Mutations: summation
    "pairwise" (a balanced tree per voxel), divide=False (multiply by the reciprocal of voxel), half_offset=False (vmin = min)."""
    p = _f64(p)
    lo, hi = p.min(0), p.max(0)
    vmin = lo - voxel * 0.5 if half_offset else lo
    vmax = hi + voxel * 0.5
    if voxel * INT_MAX < (vmax - vmin).max():
        raise ValueError("voxel_size is too small")
    rel = p - vmin
    idx = np.floor(rel / voxel if divide else rel * (1.0 / voxel)).astype(np.int64)
    nb = np.floor((hi - vmin) / voxel).astype(np.int64) + 1
    keys = (idx[:, 2] * nb[1] + idx[:, 1]) * nb[0] + idx[:, 0]
    order = np.argsort(keys, kind="stable")
    sk = keys[order]
    first = np.concatenate([[True], sk[1:] != sk[:-1]])
    starts = np.nonzero(first)[0]
    counts = np.diff(np.concatenate([starts, [len(sk)]]))
    ps = p[order]
    if summation == "pairwise":
        sums = np.stack([_pairwise(ps[a:a + c]) for a, c in zip(starts, counts)])
    else:
        sums = _sequential_sums(ps, starts, counts)
    return sums / counts[:, None].astype(np.float64), counts, sk[starts]


def voxel_down_sample_dict(p, voxel):
    """A literal restatement of VoxelDownSample with a dict of voxel -> running sum, in input order -> {voxel index: mean}."""
    p = _f64(p)
    vmin = p.min(0) - voxel * 0.5
    acc = {}
    for q in p:
        key = tuple(int(np.floor(c)) for c in (q - vmin) / voxel)
        s, c = acc.get(key, (np.zeros(3), 0))
        acc[key] = (s + q, c + 1)
    return {k: s / c for k, (s, c) in acc.items()}


def nearest(query, target, cap):
    """cKDTree distances from every query point to its nearest target point, +inf where that is not < cap."""
    from scipy.spatial import cKDTree
    q, t = _f64(query), _f64(target)
    if len(t) == 0:
        return np.full(len(q), np.inf)
    d, _ = cKDTree(t).query(q, k=1, distance_upper_bound=cap, workers=-1)
    return np.where(d < cap, d, np.inf)


def histogram_edges(tau, stretch=5):
    return np.arange(0, tau * stretch, tau / 100)


def f1_histo(tau, stretch, d_s, d_t):
    """get_f1_score_histo2 -> (precision, recall, fscore, edges, cum_precision, cum_recall); fscore = 0 when precision + recall = 0
    (the toolbox raises ZeroDivisionError)."""
    if len(d_s) and len(d_t):
        recall = float(np.sum(d_t < tau)) / float(len(d_t))
        precision = float(np.sum(d_s < tau)) / float(len(d_s))
        fscore = 2 * recall * precision / (recall + precision) if recall + precision > 0 else 0.0
        edges = histogram_edges(tau, stretch)
        cum_s = np.cumsum(np.histogram(d_s, edges)[0]).astype(float) / len(d_s)
        cum_t = np.cumsum(np.histogram(d_t, edges)[0]).astype(float) / len(d_t)
        return precision, recall, fscore, edges, cum_s, cum_t
    z = np.array([0])
    return 0.0, 0.0, 0.0, z, z, z


def distance_margin(d, tau, stretch, cap):
    """Relative margins of each distance decision over tau: to tau, to the nearest histogram edge, to the search cap."""
    d = np.asarray(d, np.float64)
    e = histogram_edges(tau, stretch)
    fin = np.isfinite(d)
    m_e = np.full(len(d), np.inf)
    if fin.any():
        i = np.clip(np.searchsorted(e, d[fin]), 1, len(e) - 1)
        m_e[fin] = np.minimum(np.abs(d[fin] - e[i - 1]), np.abs(d[fin] - e[i]))
    return np.minimum.reduce([np.abs(d - tau), m_e, np.abs(d - cap)]) / tau


def evaluate(xyz, gt, crop_volume, A, tau, stretch=5, cap=None, round_fp32=True, crop_before_transform=False):
    """The whole evaluation -> dict with the keys of evaluate_tanks_and_temples plus keep_s / keep_t, the down-sampled clouds, d_s,
    d_t and the margins.  crop_volume: (axis, axis_min, axis_max, polygon); A: 4 x 4 or None; cap: the searches' max_dist (default
    stretch * tau); round_fp32=False searches the fp64 down-sampled points; crop_before_transform is a mutation."""
    axis, amin, amax, poly = crop_volume
    x, g = _f64(xyz), _f64(gt)
    cap = stretch * tau if cap is None else cap
    if crop_before_transform:
        ks, ms = crop(x, axis, amin, amax, poly)
        xs = x[ks] if A is None else transform(x[ks], A)
    else:
        xt = x if A is None else transform(x, A)
        ks, ms = crop(xt, axis, amin, amax, poly)
        xs = xt[ks]
    kt, mt = crop(g, axis, amin, amax, poly)
    gs = g[kt]
    s = voxel_down_sample(xs, tau / 2)[0] if len(xs) else np.zeros((0, 3))
    t = voxel_down_sample(gs, tau / 2)[0] if len(gs) else np.zeros((0, 3))
    sq, tq = (s.astype(np.float32), t.astype(np.float32)) if round_fp32 else (s, t)
    if len(s) and len(t):
        d_s, d_t = nearest(sq, tq, cap), nearest(tq, sq, cap)
    else:
        d_s, d_t = np.full(len(s), np.inf), np.full(len(t), np.inf)
    precision, recall, fscore, edges, cum_s, cum_t = f1_histo(tau, stretch, d_s, d_t)
    return {"precision": precision, "recall": recall, "fscore": fscore, "tau": tau, "n": len(x), "n_cropped": len(xs), "n_down": len(s),
            "m": len(g), "m_cropped": len(gs), "m_down": len(t), "n_precision": int(np.sum(d_s < tau)), "m_recall": int(np.sum(d_t < tau)),
            "edges": edges, "cum_precision": cum_s, "cum_recall": cum_t, "keep_s": ks, "keep_t": kt, "xyz_down": s, "gt_down": t,
            "d_s": d_s, "d_t": d_t, "margin_crop_s": ms, "margin_crop_t": mt,
            "margin_s": distance_margin(d_s, tau, stretch, cap), "margin_t": distance_margin(d_t, tau, stretch, cap)}
