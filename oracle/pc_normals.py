"""numpy + cKDTree restatement of K10 (DESIGN §4 "K10 normals"): exact k-nearest neighbourhoods under the order (d^2, row), the
centred fp64 covariance, np.linalg.eigh, and both sign rules, with the margins that say where a GPU result must agree exactly.

Mutation switches (each must change a planted case; tests/test_normals_host.py):
    exclude_self      the query point is not its own neighbour
    ties_larger       ties of d^2 go to the larger row
    cumulant          the covariance as fp32 raw cumulants E[p p^T] - mu mu^T (Open3D's form) instead of centred fp64
    flip_le           the viewpoint flip on n . (v - p) <= 0 instead of < 0
    canon_smallest    the canonical sign taken on the component of smallest magnitude"""
import numpy as np
from scipy.spatial import cKDTree


def d2_fp32(q, p):
    """(dx^2 + dy^2) + dz^2 in fp32 of fp32 points q [.., 3] and p [.., 3]."""
    d = np.asarray(p, np.float32) - np.asarray(q, np.float32)
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def knn(query, target, k, max_dist=np.inf, *, exclude_self=False, ties_larger=False):
    """-> (index int64 [n, k] (-1 padded), d fp64 [n, k] (+inf padded), margin fp64 [n]): the k target rows first in (d^2, row)
    among d < max_dist, d = sqrt of the fp32 d^2; margin = the relative gap between the last listed distance and the first
    distance left out (by the order or the cap), and the relative distance of either to a finite cap (1.0 when nothing is cut)."""
    q = np.asarray(query, np.float32)
    t = np.asarray(target, np.float32)
    n, m = len(q), len(t)
    idx = np.full((n, k), -1, np.int64)
    dist = np.full((n, k), np.inf)
    margin = np.ones(n)
    if n == 0 or m == 0:
        return idx, dist, margin
    tree = cKDTree(t.astype(np.float64))
    kk = min(m, 2 * k + 32)
    while True:
        _, cand = tree.query(q.astype(np.float64), kk)
        cand = np.asarray(cand).reshape(n, -1)
        d2 = d2_fp32(q[:, None, :], t[cand]).astype(np.float64)
        # the candidates are enough when the farthest exceeds the (k + 1)-th in fp32 (no tie group is cut) or all were taken
        srt = np.sort(d2, 1)
        if kk == m or (srt[:, -1] > srt[:, min(k, kk - 1)]).all():
            break
        kk = min(m, 2 * kk)
    for i in range(n):
        c, dd = cand[i], d2[i]
        if exclude_self:
            keep = c != i
            c, dd = c[keep], dd[keep]
        order = np.lexsort((-c if ties_larger else c, dd))
        c, dd = c[order], np.sqrt(dd[order])
        inside = dd < max_dist
        cin, din = c[inside][:k], dd[inside][:k]
        idx[i, :len(cin)], dist[i, :len(din)] = cin, din
        nxt = dd[len(cin)] if len(cin) < len(dd) else np.inf
        last = din[-1] if len(din) else 0.0
        g = [(nxt - last) / nxt if np.isfinite(nxt) and nxt > 0 else 1.0]
        if np.isfinite(max_dist):
            g += [abs(max_dist - last) / max_dist]
            if np.isfinite(nxt):
                g += [abs(nxt - max_dist) / max_dist]
        margin[i] = min(g)
    return idx, dist, margin


def covariance(pts, *, cumulant=False):
    """The covariance of the points [c, 3] (fp32 values) in list order: centred fp64 two-pass, or the fp32 raw cumulants."""
    if cumulant:
        p = np.asarray(pts, np.float32)
        mu = p.mean(0, dtype=np.float32)
        return (p.T @ p / np.float32(len(p)) - np.outer(mu, mu)).astype(np.float64)
    p = np.asarray(pts, np.float32).astype(np.float64)
    mu = p.sum(0) / len(p)
    d = p - mu
    return d.T @ d / len(p)


def normals(xyz, k=30, max_dist=np.inf, viewpoints=None, *, exclude_self=False, ties_larger=False, cumulant=False, flip_le=False,
            canon_smallest=False):
    """-> dict normal fp64 [n, 3] (zero where c < 3 or trace 0), count [n], and the margins nbr (knn's), eigengap
    (lambda1 - lambda0) / lambda2, canon (|largest| - |second largest| component, or smallest for canon_smallest), orient
    |n . (v - p)| / |v - p| (inf without viewpoints)."""
    p = np.asarray(xyz, np.float32)
    n = len(p)
    idx, _, nbr = knn(p, p, k, max_dist, exclude_self=exclude_self, ties_larger=ties_larger)
    out = np.zeros((n, 3))
    gap, canon, orient = np.full(n, np.inf), np.full(n, np.inf), np.full(n, np.inf)
    count = (idx >= 0).sum(1)
    v = None if viewpoints is None else np.broadcast_to(np.asarray(viewpoints, np.float64).reshape(-1, 3), (n, 3))
    for i in range(n):
        c = count[i]
        if c < 3:
            continue
        C = covariance(p[idx[i, :c]], cumulant=cumulant)
        if not np.trace(C) > 0:
            continue
        w, V = np.linalg.eigh(C)
        nv = V[:, 0]
        gap[i] = (w[1] - w[0]) / w[2] if w[2] > 0 else 0.0
        a = np.abs(nv)
        srt = np.sort(a)
        if canon_smallest:
            ax = int(np.argmin(a))
            canon[i] = srt[1] - srt[0]
        else:
            ax = int(np.argmax(a))                     # the first axis on a tie
            canon[i] = srt[2] - srt[1]
        if nv[ax] < 0:
            nv = -nv
        if v is not None:
            r = v[i] - p[i].astype(np.float64)
            dot = float(nv @ r)
            if dot < 0 or (flip_le and dot <= 0):
                nv = -nv
            nr = np.linalg.norm(r)
            orient[i] = abs(dot) / nr if nr > 0 else 0.0
        out[i] = nv
    return {"normal": out, "count": count, "nbr": nbr, "eigengap": gap, "canon": canon, "orient": orient}


def surface(kind, n, rng, scale=1.0, offset=(0.0, 0.0, 0.0), noise=0.0):
    """n points of a plane z = 0 patch, a sphere of radius scale or a cylinder x^2 + y^2 = scale^2 (axis z), plus Gaussian noise of
    `noise` scale per axis, moved by offset -> (fp32 points [n, 3], fp64 analytic unit normals [n, 3] at the noise-free points)."""
    if kind == "plane":
        x = rng.uniform(-scale, scale, (n, 2))
        p = np.c_[x, np.zeros(n)]
        nrm = np.tile([0.0, 0.0, 1.0], (n, 1))
    elif kind == "sphere":
        nrm = rng.standard_normal((n, 3))
        nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
        p = scale * nrm
    elif kind == "cylinder":
        th = rng.uniform(0, 2 * np.pi, n)
        nrm = np.c_[np.cos(th), np.sin(th), np.zeros(n)]
        p = np.c_[scale * nrm[:, :2], rng.uniform(-scale, scale, n)]
    else:
        raise ValueError(kind)
    p = p + noise * scale * rng.standard_normal((n, 3)) + np.asarray(offset)
    return p.astype(np.float32), nrm


def angle(a, b):
    """The unsigned angle between the lines of a and b [n, 3] (radians, fp64), robust near 0."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    a = a / np.linalg.norm(a, axis=1, keepdims=True)
    b = b / np.linalg.norm(b, axis=1, keepdims=True)
    s = np.linalg.norm(np.cross(a, b), axis=1)
    return np.arctan2(s, np.abs((a * b).sum(1)))
