"""fp64 numpy restatement of the Tanks and Temples registration (the toolbox's registration_vol_ds / registration_unif stages of
run.py, with Open3D 0.10's point-to-point ICP with scaling), written from the contract in DESIGN §4 "K9 registration", not from the
kernels.  numpy, and scipy.spatial.cKDTree for the correspondences; the transform, crop and voxel down-sampling are
oracle/tnt_eval.py's.  Test infrastructure only.

Every correspondence decision of every iteration comes with a relative margin: |d - d_max| / d_max, and for a point with a
correspondence the gap between its first and second nearest target points over the second.  Mutation switches reproduce plausible
mistakes; the tests show that each one changes a result:
    with_scaling=False                                   no scale in the Umeyama update
    compose="init_first"                                 a stage's result T_init @ T_icp instead of T_icp @ T_init
    transform_gt=True                                    the stage's transform applied to the ground truth instead of the reconstruction
    relative_fitness / relative_rmse / max_iteration     the criteria (max_iteration=20, relative_rmse=1e-6: the other reading)
    rounding="half_up" / "floor" / "ceil"                the uniform rate's rounding instead of Python's half-to-even round"""
from __future__ import annotations

import math

import numpy as np

import tnt_eval

MAX_POINT_NUMBER = 4_000_000


def _f64(a):
    return np.asarray(a, dtype=np.float64).reshape(-1, 3)


def umeyama(src, dst, with_scaling=True):
    """Eigen's umeyama(src^T, dst^T, with_scaling) for corresponding rows src [c, 3], dst [c, 3] -> 4 x 4 (the identity for c = 0,
    and, with scaling, for a zero source variance)."""
    s, t = _f64(src), _f64(dst)
    c = len(s)
    if c == 0:
        return np.eye(4)
    mu_s, mu_t = s.mean(0), t.mean(0)
    a, b = s - mu_s, t - mu_t
    sigma = b.T @ a / c
    var = float((a * a).sum()) / c
    if with_scaling and var == 0:
        return np.eye(4)
    U, D, Vt = np.linalg.svd(sigma)
    S = np.ones(3)
    if np.linalg.det(U) * np.linalg.det(Vt) < 0:
        S[2] = -1.0
    R = (U * S) @ Vt
    scale = float(D @ S) / var if with_scaling else 1.0
    out = np.eye(4)
    out[:3, 3] = mu_t - scale * (R @ mu_s)
    out[:3, :3] = scale * R
    return out


def correspondences(p, tree, target_len, d_max, round_fp32=True):
    """Per source point the nearest target point if its distance is < d_max -> (index int64 [n], -1 for none; the distance; the
    decision margin [n]).  round_fp32: search the fp32 rounding of the points (the tree is built on the target's)."""
    q = p.astype(np.float32).astype(np.float64) if round_fp32 else p
    if target_len == 0 or len(q) == 0:
        return np.full(len(q), -1), np.full(len(q), np.inf), np.full(len(q), np.inf)
    k = min(2, target_len)
    d, i = tree.query(q, k=k, workers=-1)
    d, i = d.reshape(len(q), k), i.reshape(len(q), k)
    has = d[:, 0] < d_max
    idx = np.where(has, i[:, 0], -1)
    margin = np.abs(d[:, 0] - d_max) / d_max
    if k == 2:
        with np.errstate(divide="ignore", invalid="ignore"):
            gap = np.where(d[:, 1] > 0, (d[:, 1] - d[:, 0]) / d[:, 1], 0.0)
        margin = np.where(has, np.minimum(margin, gap), margin)
    return idx, np.where(has, d[:, 0], np.inf), margin


def icp(source, target, d_max, with_scaling=True, relative_fitness=1e-6, relative_rmse=20.0, max_iteration=30, round_fp32=True):
    """Open3D 0.10's RegistrationICP (point to point) from the identity -> dict with transformation, fitness, inlier_rmse,
    correspondences, iterations, history (per search: correspondences, fitness, inlier_rmse) and min_margin over every decision."""
    from scipy.spatial import cKDTree
    p, t = _f64(source).copy(), _f64(target)
    n = len(p)
    tree = cKDTree(t.astype(np.float32).astype(np.float64) if round_fp32 else t) if len(t) else None
    state = {"margin": np.inf}

    def result(p):
        idx, _, margin = correspondences(p, tree, len(t), d_max, round_fp32)
        if len(margin):
            state["margin"] = min(state["margin"], float(margin.min()))
        sel = idx >= 0
        c = int(sel.sum())
        d2 = ((p[sel] - t[idx[sel]]) ** 2).sum(1)
        return idx, c, (c / n if n else 0.0), (math.sqrt(float(d2.sum()) / c) if c else 0.0)

    T = np.eye(4)
    idx, c, fit, rmse = result(p)
    history = [{"correspondences": c, "fitness": fit, "inlier_rmse": rmse}]
    iterations = 0
    for i in range(max_iteration):
        sel = idx >= 0
        U = umeyama(p[sel], t[idx[sel]], with_scaling)
        T = U @ T
        p = tnt_eval.transform(p, U)
        prev_fit, prev_rmse = fit, rmse
        idx, c, fit, rmse = result(p)
        history.append({"correspondences": c, "fitness": fit, "inlier_rmse": rmse})
        iterations = i + 1
        if abs(prev_fit - fit) < relative_fitness and abs(prev_rmse - rmse) < relative_rmse:
            break
    return {"transformation": T, "fitness": fit, "inlier_rmse": rmse, "correspondences": c, "iterations": iterations,
            "history": history, "min_margin": state["margin"], "points": p}


def uniform_rate(n, max_points=MAX_POINT_NUMBER, rounding="half_even"):
    """The toolbox's rate: int(round(n / max_points)) when n > max_points, else 1; `rounding` other than half_even is a mutation."""
    if n <= max_points:
        return 1
    r = n / float(max_points)
    return {"half_even": lambda: int(round(r)), "half_up": lambda: int(math.floor(r + 0.5)), "floor": lambda: int(math.floor(r)),
            "ceil": lambda: int(math.ceil(r))}[rounding]()


def crop_and_downsample(p, crop_volume, method, voxel, A, max_points=MAX_POINT_NUMBER, rounding="half_even"):
    """The toolbox's crop_and_downsample: transform by A (None: none), crop, then voxel down-sample or uniformly down-sample."""
    axis, amin, amax, poly = crop_volume
    x = _f64(p) if A is None else tnt_eval.transform(p, A)
    keep, _ = tnt_eval.crop(x, axis, amin, amax, poly)
    x = x[keep]
    if method == "voxel":
        return (tnt_eval.voxel_down_sample(x, voxel)[0] if len(x) else np.zeros((0, 3))), None
    k = uniform_rate(len(x), max_points, rounding)
    return x[::k], k


def register(xyz, gt, crop_volume, init, tau, max_points=MAX_POINT_NUMBER, with_scaling=True, relative_fitness=1e-6,
             relative_rmse=20.0, max_iteration=30, compose="icp_first", transform_gt=False, rounding="half_even", round_fp32=True):
    """The three stages -> dict with transformation, stages (per stage: method, n_down, m_down, rates, iterations, fitness,
    inlier_rmse, correspondences, history, transformation) and min_margin over every stage."""
    T = np.asarray(init, np.float64)
    stages, margin = [], np.inf
    for method, voxel, d_max in (("voxel", tau, 80 * tau), ("voxel", tau / 2, 20 * tau), ("uniform", None, 2 * tau)):
        s, ks = crop_and_downsample(xyz, crop_volume, method, voxel, None if transform_gt else T, max_points, rounding)
        t, kt = crop_and_downsample(gt, crop_volume, method, voxel, T if transform_gt else None, max_points, rounding)
        r = icp(s, t, d_max, with_scaling, relative_fitness, relative_rmse, max_iteration, round_fp32)
        T = r["transformation"] @ T if compose == "icp_first" else T @ r["transformation"]
        margin = min(margin, r["min_margin"])
        stages.append({"method": method, "voxel": voxel, "rate_source": ks, "rate_target": kt, "max_correspondence_distance": d_max,
                       "n_down": len(s), "m_down": len(t), "iterations": r["iterations"], "fitness": r["fitness"],
                       "inlier_rmse": r["inlier_rmse"], "correspondences": r["correspondences"], "history": r["history"],
                       "transformation": T})
    return {"transformation": T, "stages": stages, "min_margin": margin}


def similarity_error(T, T_true):
    """The error E = T T_true^-1 of an estimated similarity -> (its rotation angle in rad, |scale - 1|, |translation|)."""
    E = T @ np.linalg.inv(T_true)
    s = float(np.cbrt(np.linalg.det(E[:3, :3])))
    R = E[:3, :3] / s
    ang = float(np.arccos(np.clip((np.trace(R) - 1) / 2, -1.0, 1.0)))
    return ang, abs(s - 1.0), float(np.linalg.norm(E[:3, 3]))


# ---- seeded test scenes ---------------------------------------------------------------------------------------------------------

def rotation(axis, deg):
    """The rotation by `deg` degrees about `axis` (Rodrigues)."""
    a = np.asarray(axis, np.float64)
    a = a / np.linalg.norm(a)
    t = np.radians(deg)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * K @ K


def similarity(R, s, t):
    A = np.eye(4)
    A[:3, :3] = s * np.asarray(R)
    A[:3, 3] = t
    return A


def _walls(rng, n, x_max=4.0):
    k = rng.multinomial(n, [0.45, 0.2, 0.2, 0.15])
    x, y = rng.uniform(0, x_max, k[0]), rng.uniform(0, 3, k[0])
    ground = np.stack([x, y, 0.1 * np.sin(1.7 * x) * np.cos(1.1 * y) + 0.03 * x], 1)
    y, z = rng.uniform(0, 3, k[1]), rng.uniform(0, 1.5, k[1])
    wall_x = np.stack([0.05 * np.sin(2 * y), y, z], 1)
    x, z = rng.uniform(0, x_max, k[2]), rng.uniform(0, 1.2, k[2])
    wall_y = np.stack([x, 0.1 * z * z, z], 1)
    u = rng.standard_normal((k[3], 3))
    u[:, 2] = np.abs(u[:, 2])
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    blob = np.array([2.6, 1.9, 0.0]) + u * np.array([0.7, 0.45, 0.6])
    return np.concatenate([ground, wall_x, wall_y, blob])


def walls_scene(seed=0, n_gt=40000, n_rec=25000, tau=0.03, noise=0.002, deg=3.0, scale=1.02, shift=3.0):
    """A non-symmetric curved scene (a wavy ground, two walls, a half ellipsoid; metres) -> (reconstruction fp32 [~n_rec, 3] in its
    own frame, ground truth fp32 [n_gt, 3], crop volume, T_true mapping the reconstruction onto the ground truth, T0 = P T_true with
    P the planted perturbation: `deg` degrees, `scale`, `shift` tau), and tau.  The reconstruction covers x < 3.7 with Gaussian noise."""
    rng = np.random.default_rng(seed)
    gt = _walls(rng, n_gt).astype(np.float32)
    rec = _walls(rng, n_rec, 3.7)
    rec = rec + noise * rng.standard_normal(rec.shape)
    T_true = similarity(rotation([0.2, -0.3, 1.0], 25.0), 1.3, [0.5, -0.2, 0.1])
    rec_in = tnt_eval.transform(rec, np.linalg.inv(T_true)).astype(np.float32)
    P = similarity(rotation([1.0, 0.5, 0.3], deg), scale, np.array([1.0, -0.67, 0.5]) * shift * tau)
    crop = ("Z", -0.5, 1.4, np.array([[-0.3, -0.3, 0.0], [3.9, -0.2, 0.0], [4.2, 3.2, 0.0], [2.0, 2.6, 0.0], [-0.2, 3.1, 0.0]]))
    return rec_in, gt, crop, T_true, P @ T_true, tau


def lattice_icp_scene(seed=6, k=10, jitter=0.08, noise=0.03, deg=4.0, scale=1.01, shift=0.15):
    """ICP inputs with wide decision margins: the target a jittered unit lattice k^3; the source 60 % of it with noise, moved by a
    small similarity about its centre, plus 20 outliers above the lattice -> (source fp64, target fp64)."""
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(*[np.arange(k)] * 3, indexing="ij"), -1).reshape(-1, 3).astype(np.float64)
    tgt = g + jitter * rng.uniform(-1, 1, g.shape)
    sel = rng.random(len(tgt)) < 0.6
    src = tgt[sel] + noise * rng.standard_normal((int(sel.sum()), 3))
    c = src.mean(0)
    P = similarity(rotation(rng.standard_normal(3), deg), scale, shift * rng.standard_normal(3))
    src = (src - c) @ P[:3, :3].T + c + P[:3, 3]
    out = rng.uniform(-3, k + 2, (20, 3))
    out[:, 2] = k + 3 + rng.uniform(0, 2, 20)
    return np.concatenate([src, out]), tgt
