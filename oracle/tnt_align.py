"""fp64 numpy restatement of the Tanks and Temples trajectory alignment (the toolbox's registration.py::trajectory_alignment with
Open3D 0.10's RegistrationRANSACBasedOnCorrespondence), written from the contract in DESIGN §4 "K9 trajectory alignment", not from
the kernels.  The Umeyama solve is oracle/tnt_register.py's (numpy's LAPACK SVD), one hypothesis at a time; the scoring is
vectorised over hypotheses.  Test infrastructure only.

Every hypothesis comes with two margins: the smallest |d^2 - d_max^2| / d_max^2 over its correspondences (how far its inlier count
is from flipping) and the conditioning sigma_2 / sigma_1 of its 3 x 3 cross-covariance (how well its transform is determined).
Mutation switches reproduce plausible mistakes; the tests show that each one changes a result:
    mapping_base=0          the mapping's frame numbers read as 0-based
    apply_gt_trans=False    the reference centres left in T&T's COLMAP frame
    tie="last"              the last of exactly tied hypotheses instead of the first
    select="fitness"        the best hypothesis by inlier count alone, ignoring the rmse
    swap=True               the reference registered onto the trajectory instead of the other way round"""
from __future__ import annotations

import numpy as np

import tnt_eval
import tnt_register

GOLDEN = np.uint64(0x9E3779B97F4A7C15)


def splitmix64(x):
    """The SplitMix64 finaliser of uint64 states x (numpy arrays wrap mod 2^64)."""
    z = np.asarray(x, np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def draws(seed, n_hyp, ransac_n, n, first=0):
    """The indices of hypotheses first .. first + n_hyp - 1 -> int64 [n_hyp, ransac_n]: draw j of hypothesis h is
    splitmix64(seed + (h ransac_n + j + 1) GOLDEN mod 2^64) mod n."""
    k = (np.arange(first, first + n_hyp, dtype=np.uint64)[:, None] * np.uint64(ransac_n)
         + np.arange(ransac_n, dtype=np.uint64)[None] + np.uint64(1))
    with np.errstate(over="ignore"):
        return (splitmix64(np.uint64(seed) + k * GOLDEN) % np.uint64(n)).astype(np.int64)


def points(poses, reference_poses, gt_trans, mapping=None, mapping_base=1, apply_gt_trans=True):
    """-> (source centres [k, 3], reference centres [k, 3]) as the toolbox pairs them; mapping: rows [k, 2] (frame numbers in the
    second column), used when there are more than 1600 poses."""
    P = np.asarray(poses, np.float64)
    if len(P) > 1600:
        P = P[np.asarray(mapping)[:, 1].astype(np.int64) - mapping_base]
    c = np.asarray(reference_poses, np.float64)[:, :3, 3]
    ref = tnt_eval.transform(c, np.asarray(gt_trans, np.float64)) if apply_gt_trans else c
    assert len(P) >= len(ref), "fewer points to register than reference points"
    return P[:len(ref), :3, 3].copy(), ref


def hypotheses(src, tgt, idx, with_scaling=True):
    """Per hypothesis (rows of idx) tnt_register.umeyama on its pairs -> (T fp64 [H, 4, 4], NaN for fewer than 3 distinct indices;
    conditioning sigma_2 / sigma_1 [H], 0 for those)."""
    T = np.full((len(idx), 4, 4), np.nan)
    cond = np.zeros(len(idx))
    for h, k in enumerate(idx):
        if len(np.unique(k)) < 3:
            continue
        s, t = src[k], tgt[k]
        T[h] = tnt_register.umeyama(s, t, with_scaling)
        sv = np.linalg.svd((t - t.mean(0)).T @ (s - s.mean(0)) / len(k), compute_uv=False)
        cond[h] = sv[1] / sv[0] if sv[0] > 0 else 0.0
    return T, cond


def score(src, tgt, T, d_max, chunk=1024):
    """Vectorised scoring of transforms T [H, 4, 4] -> (good int64 [H], error2 [H] added in correspondence order, margin [H] the
    smallest |d^2 - d_max^2| / d_max^2, inf for a NaN transform).  d^2 = ((dx dx + dy dy) + dz dz), dx from K9 step 1's order."""
    thr = d_max * d_max
    H = len(T)
    good, error2, margin = np.zeros(H, np.int64), np.zeros(H), np.full(H, np.inf)
    for a in range(0, H, chunk):
        M = T[a:a + chunk]
        q = [((M[:, r, 0, None] * src[None, :, 0] + M[:, r, 1, None] * src[None, :, 1]) + M[:, r, 2, None] * src[None, :, 2])
             + M[:, r, 3, None] for r in range(3)]
        d = [q[r] - tgt[None, :, r] for r in range(3)]
        d2 = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]
        with np.errstate(invalid="ignore"):
            inl = d2 < thr
        good[a:a + chunk] = inl.sum(1)
        error2[a:a + chunk] = np.cumsum(np.where(inl, d2, 0.0), axis=1)[:, -1] if src.shape[0] else 0.0
        m = np.abs(d2 - thr) / thr
        margin[a:a + chunk] = np.where(np.isnan(m).any(1), np.inf, np.nanmin(np.where(np.isnan(m), np.inf, m), axis=1))
    return good, error2, margin


def rmse(good, error2):
    """sqrt(error2 / good), 0 where good = 0."""
    g = np.asarray(good, np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(g > 0, np.sqrt(np.asarray(error2) / g), 0.0)


def select(good, error2, tie="first", select="lexicographic"):
    """Open3D's running best from the identity (fitness 0, rmse 0), replaced on a larger fitness or an equal one with a strictly
    smaller rmse -> the winning h, -1 when no hypothesis has an inlier.  tie="last" / select="fitness" are mutations."""
    good = np.asarray(good)
    if not (good > 0).any():
        return -1
    cand = good == good.max()
    if select == "lexicographic":
        r = rmse(good, error2)
        cand &= r == r[cand].min()
    h = np.flatnonzero(cand)
    return int(h[0] if tie == "first" else h[-1])


def align(poses, reference_poses, gt_trans, mapping=None, d_max=0.2, ransac_n=6, n_hyp=100000, with_scaling=True, seed=0,
          mapping_base=1, apply_gt_trans=True, tie="first", select_by="lexicographic", swap=False):
    """The whole alignment -> dict with transformation, hypothesis, fitness, inlier_rmse, inliers, sample, and per hypothesis good,
    error2, transforms, cond, margin; `gap`: the relative rmse gap between the best and the runner-up among the hypotheses with
    the best's inlier count whose rmse differs from the best's (inf when there is none)."""
    src, tgt = points(poses, reference_poses, gt_trans, mapping, mapping_base, apply_gt_trans)
    if swap:
        src, tgt = tgt, src
    idx = draws(seed, n_hyp, ransac_n, len(src))
    T, cond = hypotheses(src, tgt, idx, with_scaling)
    good, error2, margin = score(src, tgt, T, d_max)
    h = select(good, error2, tie, select_by)
    out = {"hypothesis": h, "good": good, "error2": error2, "transforms": T, "cond": cond, "margin": margin, "draws": idx,
           "n_correspondences": len(src), "gap": np.inf}
    if h < 0:
        out.update(transformation=np.eye(4), fitness=0.0, inlier_rmse=0.0, inliers=0, sample=[])
        return out
    r = rmse(good, error2)
    out.update(transformation=T[h], fitness=good[h] / len(src), inlier_rmse=float(r[h]), inliers=int(good[h]), sample=idx[h].tolist())
    others = r[(good == good[h]) & (r != r[h])]
    if len(others):
        out["gap"] = float((others.min() - r[h]) / r[h]) if r[h] > 0 else np.inf
    return out


# ---- seeded test scenes ---------------------------------------------------------------------------------------------------------

def _rotations(rng, n):
    q = rng.standard_normal((n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.stack([np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)], -1),
                     np.stack([2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)], -1),
                     np.stack([2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], -1)], 1)


def poses_at(centres, rng):
    """Camera-to-world poses with random rotations and the given centres -> [n, 4, 4]."""
    P = np.zeros((len(centres), 4, 4))
    P[:, :3, :3] = _rotations(rng, len(centres))
    P[:, :3, 3] = centres
    P[:, 3, 3] = 1.0
    return P


def orbit_centres(n, rng, radius=15.0):
    """A T&T-like capture path in the ground truth's frame: 1.3 turns around the scene on a wobbling ellipse, the camera height
    varying by about 2 units -> [n, 3], tens of units across."""
    th = np.linspace(0, 2.6 * np.pi, n) + 0.01 * rng.standard_normal(n)
    r = radius * (1 + 0.15 * np.sin(3 * th))
    return np.stack([1.2 * r * np.cos(th), r * np.sin(th), 1.6 + 1.0 * np.sin(2 * th) + 0.5 * np.cos(5 * th)], 1)


def orbit_scene(n=400, seed=0, noise=0.01, outliers=0.15, S=None, G=None):
    """-> dict: poses (the user's trajectory in its own frame), reference (T&T's COLMAP trajectory), gt_trans (COLMAP -> GT),
    S_true (the user's frame -> GT: the transform to recover) and outlier (bool [n]).  The user's centres are the GT-frame centres
    with Gaussian noise of `noise` per axis and a fraction `outliers` displaced by 1-3 units, mapped by S_true^-1."""
    rng = np.random.default_rng(seed)
    c = orbit_centres(n, rng)
    S_true = S if S is not None else tnt_register.similarity(tnt_register.rotation([0.3, -0.8, 0.5], 130.0), 0.37, [250.0, -40.0, 12.0])
    G = G if G is not None else tnt_register.similarity(tnt_register.rotation([1.0, 0.2, -0.1], 25.0), 2.3, [1.5, -0.5, 0.2])
    out = np.zeros(n, bool)
    out[rng.choice(n, int(round(outliers * n)), replace=False)] = True
    u = c + noise * rng.standard_normal(c.shape)
    v = rng.standard_normal((int(out.sum()), 3))
    u[out] += v / np.linalg.norm(v, axis=1, keepdims=True) * rng.uniform(1.0, 3.0, (len(v), 1))
    return {"poses": poses_at(tnt_eval.transform(u, np.linalg.inv(S_true)), rng),
            "reference": poses_at(tnt_eval.transform(c, np.linalg.inv(G)), rng), "gt_trans": G, "S_true": S_true, "outlier": out}
