"""Registration of a reconstruction to the Tanks and Temples ground truth: the official toolbox's (python_toolbox/evaluation: run.py,
registration.py) RANSAC trajectory alignment over camera centres (trajectory_alignment, with Open3D 0.10's
RegistrationRANSACBasedOnCorrespondence) and the three ICP stages it runs before it scores a cloud (registration_vol_ds /
registration_unif, with Open3D 0.10's point-to-point ICP with scaling, RegistrationICP, TransformationEstimationPointToPoint).
DESIGN §4 "K9 trajectory alignment" and "K9 registration" state the contracts and where they differ.

    gt, crop, trans = load_tnt_eval("/data/tnt", "Barn")
    ref, mapping = load_tnt_trajectory("/data/tnt", "Barn")
    _, poses = read_trajectory("Barn.log")                      # the cameras of the reconstruction, in its own frame
    init = align_trajectory(poses, ref, trans, mapping=mapping)["transformation"]
    reg = register_tanks_and_temples(xyz.cuda(), gt.cuda(), crop, init, tau=0.01)
    out = evaluate_tanks_and_temples(xyz.cuda(), gt.cuda(), crop, reg["transformation"], tau=0.01)

For a reconstruction already in T&T's COLMAP frame, `trans` itself is the init.  The hot path is kernels of this library: for the
alignment, one thread per RANSAC hypothesis (draws, Umeyama with an fp64 Jacobi SVD, scoring) and a deterministic selection; per ICP
iteration the capped nearest search with indices, the Umeyama sums in two deterministic fp64 passes and the fp64 update of the
source; K9's transform, crop and voxel down-sampling per stage.  The host reads camera centres, solves ICP's 3 x 3 SVD and composes
the 4 x 4 matrices in fp64 numpy.  There is no CPU path."""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _lib
from .evaluation import _cloud, _positive, build_grid, nearest_index_into
from .ops import _stream, _timed
from .tanks import CropVolume, _crop_volume, crop_points, voxel_down_sample

MAX_POINT_NUMBER = 4_000_000                     # the toolbox's MAX_POINT_NUMBER: stage 3's uniform down-sampling target
MAX_DENSE_POSES = 1600                           # a trajectory with more poses is every video frame: it is sampled by the mapping
RELATIVE_FITNESS, RELATIVE_RMSE, MAX_ITERATION = 1e-6, 20.0, 30     # ICPConvergenceCriteria(1e-6, 20) as the toolbox writes it


def _fail(msg):
    raise _lib.MvsB200Error("registration: " + msg)


def _points64(x, what):
    if not isinstance(x, torch.Tensor) or not x.is_cuda:
        _fail(f"{what} must be a CUDA tensor; mvs_b200 has no CPU path")
    if x.dtype != torch.float64 or x.dim() != 2 or x.shape[1] != 3:
        _fail(f"{what}: fp64 points [n, 3] expected, got {x.dtype} {tuple(x.shape)}")
    if x.shape[0] >= 2 ** 31 - 1:
        _fail(f"{what}: at most 2^31 - 1 points, got {x.shape[0]}")
    x = x.detach().contiguous()
    if x.numel() and not bool(torch.isfinite(x).all()):
        _fail(f"{what}: coordinates must be finite")
    return x


def _matrix(a, what):
    try:
        m = np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a, dtype=np.float64)
    except (TypeError, ValueError):
        _fail(f"{what} must be numeric")
    if m.shape != (4, 4):
        _fail(f"{what}: a 4 x 4 matrix expected, got shape {m.shape}")
    if not np.isfinite(m).all():
        _fail(f"{what} must be finite")
    if not np.array_equal(m[3], [0.0, 0.0, 0.0, 1.0]):
        _fail(f"{what}: an affine matrix (last row exactly 0, 0, 0, 1) expected, got last row {m[3].tolist()}")
    return m.copy()


def uniform_rate(n, max_points=MAX_POINT_NUMBER):
    """The toolbox's uniform rate: int(round(n / max_points)) when n > max_points (Python's round: halves to even), else 1."""
    return int(round(n / float(max_points))) if n > max_points else 1


def uniform_down_sample(xyz64, k):
    """Open3D's UniformDownSample: the points 0, k, 2k, ... of the CUDA cloud xyz64 [n, 3] fp64, k >= 1 -> fp64 [ceil(n / k), 3]."""
    x = _points64(xyz64, "xyz64")
    if isinstance(k, bool) or int(k) != k or int(k) < 1:
        _fail(f"k must be an integer >= 1, got {k!r}")
    return x[::int(k)].contiguous()


def umeyama(sums, with_scaling=True):
    """Eigen's umeyama from the correspondence sums of pc_icp_sums (host fp64 [18]) -> the 4 x 4 update [cR | t; 0 0 0 1]:
    Sigma = (1/c) sum (t - mu_t)(s - mu_s)^T, src_var = (1/c) sum |s - mu_s|^2, Sigma = U D V^T, S = diag(1, 1, -1) when
    det U det V < 0, R = U S V^T, scale = tr(D S) / src_var (1 without scaling), t = mu_t - scale R mu_s.  The identity when there is
    no correspondence, or when src_var = 0 (every matched source point the same; Eigen's scale would be 0 / 0)."""
    h = np.asarray(sums, dtype=np.float64)
    c = h[0]
    if c == 0:
        return np.eye(4)
    mu_s, mu_t = h[2:5] / c, h[5:8] / c
    sigma = h[8:17].reshape(3, 3) / c
    var = h[17] / c
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


def icp_point_to_point(source64, target64, max_correspondence_distance, *, with_scaling=True, relative_fitness=RELATIVE_FITNESS,
                       relative_rmse=RELATIVE_RMSE, max_iteration=MAX_ITERATION, return_history=False, target_grid=None):
    """Open3D 0.10's RegistrationICP with TransformationEstimationPointToPoint(with_scaling), from the identity, of the CUDA fp64
    clouds source64 [n, 3] onto target64 [m, 3]:

        result = correspondences(P)                  # per source point: the nearest target point if closer than d_max, else none
        for i in range(max_iteration):
            U = umeyama(P[corr], target[idx])        # identity with no correspondence
            T = U @ T;  P = U(P)                     # fp64, in place
            prev, result = result, correspondences(P)
            if |prev.fitness - result.fitness| < relative_fitness and |prev.rmse - result.rmse| < relative_rmse: break

    fitness = #corr / n, inlier_rmse = sqrt(sum d^2 / #corr) (both 0 with no correspondence).  The search runs on the fp32 rounding of
    the points (ties: the smaller target row); d^2 and every Umeyama sum are fp64 on the pair's fp64 coordinates.  The defaults are
    the toolbox's ICPConvergenceCriteria(1e-6, 20) read as (relative_fitness, relative_rmse) with max_iteration left at 30.
    target_grid: a build_grid of target64's fp32 rounding to reuse.

    -> dict with transformation (fp64 4 x 4 numpy), fitness, inlier_rmse, correspondences, iterations; with return_history also
    history: per correspondence search (the initial one first) a dict of correspondences, fitness, inlier_rmse."""
    src = _points64(source64, "source64").clone()
    tgt = _points64(target64, "target64")
    d_max = _positive(max_correspondence_distance, "max_correspondence_distance")
    max_iteration = int(max_iteration)
    if max_iteration < 0:
        _fail(f"max_iteration must be >= 0, got {max_iteration}")
    relative_fitness, relative_rmse = float(relative_fitness), float(relative_rmse)
    n, m = src.shape[0], tgt.shape[0]
    dev = src.device
    src32 = src.float()
    if n and m:
        grid = target_grid if target_grid is not None else build_grid(tgt.float())
        dist = torch.empty(n, dtype=torch.float32, device=dev)
        index = torch.empty(n, dtype=torch.int32, device=dev)
        partial = torch.empty(_lib.PC_ICP_BLOCKS * 10, dtype=torch.float64, device=dev)
        ticket = torch.zeros(2, dtype=torch.int32, device=dev)
        sums = torch.empty(_lib.PC_ICP_SUMS, dtype=torch.float64, device=dev)

    def correspond():
        if not (n and m):
            return np.zeros(_lib.PC_ICP_SUMS), 0.0, 0.0
        nearest_index_into(src32, grid, d_max, dist, index)
        with _timed("pc_icp_sums"):
            _lib.call("mvsb200_pc_icp_sums", src.data_ptr(), index.data_ptr(), n, tgt.data_ptr(), partial.data_ptr(), ticket.data_ptr(),
                      sums.data_ptr(), _stream())
        h = sums.cpu().numpy()                                                # the one read-back of the iteration
        c = h[0]
        return h, c / n, (math.sqrt(h[1] / c) if c else 0.0)

    T = np.eye(4)
    h, fitness, rmse = correspond()
    history = [{"correspondences": int(h[0]), "fitness": fitness, "inlier_rmse": rmse}]
    iterations = 0
    for i in range(max_iteration):
        U = umeyama(h, with_scaling)
        T = U @ T
        if n:
            with _timed("pc_transform64"):
                _lib.call("mvsb200_pc_transform64", src.data_ptr(), n, np.ascontiguousarray(U[:3].reshape(12)).ctypes.data_as(_lib._c.c_void_p),
                          src32.data_ptr(), _stream())
        prev_fitness, prev_rmse = fitness, rmse
        h, fitness, rmse = correspond()
        history.append({"correspondences": int(h[0]), "fitness": fitness, "inlier_rmse": rmse})
        iterations = i + 1
        if abs(prev_fitness - fitness) < relative_fitness and abs(prev_rmse - rmse) < relative_rmse:
            break
    out = {"transformation": T, "fitness": fitness, "inlier_rmse": rmse, "correspondences": int(h[0]), "iterations": iterations}
    if return_history:
        out["history"] = history
    return out


def register_tanks_and_temples(xyz, gt, crop, init, tau, *, max_points=MAX_POINT_NUMBER, with_scaling=True,
                               relative_fitness=RELATIVE_FITNESS, relative_rmse=RELATIVE_RMSE, max_iteration=MAX_ITERATION):
    """The toolbox's refinement of the alignment of a reconstruction xyz [n, 3] to the ground truth gt [m, 3] (CUDA tensors, fp32
    values), from the 4 x 4 affine `init` (T&T's _trans.txt for a reconstruction in its COLMAP frame), at threshold tau > 0:

        stage  down-sampling of both clouds        d_max     from
        1      voxel, voxel = tau                  80 tau    init
        2      voxel, voxel = tau / 2              20 tau    stage 1
        3      uniform, rate uniform_rate(size)    2 tau     stage 2

    Each stage transforms the reconstruction (only) by its initial transform T_init and crops both clouds (K9 steps 1-2), down-samples
    both, runs icp_point_to_point from the identity with the criteria given here, and ends with T_init advanced to T_icp @ T_init
    (fp64).  An empty cloud after the crop or the down-sampling gives fitness 0 and leaves T_init as it is.

    -> dict with transformation (fp64 4 x 4, for evaluate_tanks_and_temples), init, tau, and stages: per stage its method, voxel or
    rate_source / rate_target, max_correspondence_distance, n_down, m_down, iterations, fitness, inlier_rmse, correspondences and
    transformation (the stage's result)."""
    x = _cloud(xyz, "xyz")
    g = _cloud(gt, "gt")
    tau = _positive(tau, "tau")
    if not isinstance(crop, CropVolume):
        _fail(f"crop must be a CropVolume (read_crop_volume), got {type(crop).__name__}")
    crop = _crop_volume(*crop)
    T0 = _matrix(init, "init")
    max_points = int(max_points)
    if max_points < 1:
        _fail(f"max_points must be >= 1, got {max_points}")
    criteria = {"with_scaling": with_scaling, "relative_fitness": relative_fitness, "relative_rmse": relative_rmse,
                "max_iteration": max_iteration}
    gs, _ = crop_points(g, crop, None)                      # the ground truth's crop does not depend on the stage
    empty = torch.empty((0, 3), dtype=torch.float64, device=x.device)
    T = T0
    stages = []
    for method, param, d_max in (("voxel", tau, 80 * tau), ("voxel", tau / 2, 20 * tau), ("uniform", None, 2 * tau)):
        xs, _ = crop_points(x, crop, T)
        rec = {"method": method}
        if method == "voxel":
            s64 = voxel_down_sample(xs, param)[0] if xs.shape[0] else empty
            t64, t32 = voxel_down_sample(gs, param)[:2] if gs.shape[0] else (empty, None)
            rec["voxel"] = param
        else:
            ks, kt = uniform_rate(xs.shape[0], max_points), uniform_rate(gs.shape[0], max_points)
            s64, t64 = xs[::ks].contiguous(), gs[::kt].contiguous()
            t32 = t64.float()
            rec.update(rate_source=ks, rate_target=kt)
        grid = build_grid(t32) if s64.shape[0] and t64.shape[0] else None
        r = icp_point_to_point(s64, t64, d_max, target_grid=grid, **criteria)
        T = r["transformation"] @ T
        rec.update(max_correspondence_distance=d_max, n_down=s64.shape[0], m_down=t64.shape[0], iterations=r["iterations"],
                   fitness=r["fitness"], inlier_rmse=r["inlier_rmse"], correspondences=r["correspondences"], transformation=T)
        stages.append(rec)
    return {"transformation": T, "init": T0, "tau": tau, "stages": stages}


def _poses(p, what):
    a = p.detach().cpu().numpy() if isinstance(p, torch.Tensor) else p
    try:
        a = np.asarray(a, dtype=np.float64)
    except (TypeError, ValueError):
        _fail(f"{what} must be numeric")
    if a.ndim != 3 or a.shape[1:] != (4, 4):
        _fail(f"{what}: poses [n, 4, 4] expected, got shape {a.shape}")
    if not np.isfinite(a).all():
        _fail(f"{what} must be finite")
    return a


def trajectory_points(poses, reference_poses, gt_trans, mapping=None):
    """The point sets of the toolbox's trajectory_alignment -> (source fp64 [k, 3], reference fp64 [k, 3]), paired row by row:
    reference = the centres pose[:3, 3] of reference_poses mapped by gt_trans in K9 step 1's operation order; source = the centres
    of `poses`, or, when there are more than MAX_DENSE_POSES of them, of poses[m[1] - 1] for each row m of the mapping (a
    tanks.Mapping or rows [k, 2]), cut to the reference's length.  Refused: a trajectory over MAX_DENSE_POSES poses without a
    mapping, a mapping row outside 1..len(poses), and fewer source points than reference points."""
    P = _poses(poses, "poses")
    ref = _poses(reference_poses, "reference_poses")
    A = _matrix(gt_trans, "gt_trans")
    if len(P) > MAX_DENSE_POSES:
        if mapping is None:
            _fail(f"a trajectory of {len(P)} > {MAX_DENSE_POSES} poses is every video frame: the scene's mapping is needed")
        rows = np.asarray(getattr(mapping, "rows", mapping))
        if rows.ndim != 2 or rows.shape[1] != 2 or not np.array_equal(rows, rows.astype(np.int64)):
            _fail(f"mapping: integer rows [k, 2] expected, got shape {rows.shape}")
        frames = rows[:, 1].astype(np.int64)
        if len(frames) and (frames.min() < 1 or frames.max() > len(P)):
            _fail(f"mapping: frame numbers must lie in 1..{len(P)} (1-based), got {frames.min()}..{frames.max()}")
        P = P[frames - 1]
    c = ref[:, :3, 3]
    target = np.stack([((A[r, 0] * c[:, 0] + A[r, 1] * c[:, 1]) + A[r, 2] * c[:, 2]) + A[r, 3] for r in range(3)], 1)
    if len(P) < len(target):
        _fail(f"{len(P)} camera centres to register but {len(target)} reference centres: every reference centre needs its pair")
    return np.ascontiguousarray(P[:len(target), :3, 3]), target


def align_trajectory(poses, reference_poses, gt_trans, *, mapping=None, max_correspondence_distance=0.2, ransac_n=6,
                     max_iteration=100000, with_scaling=True, seed=0, return_details=False):
    """The toolbox's trajectory_alignment: RANSAC (Open3D 0.10's RegistrationRANSACBasedOnCorrespondence) over the camera centres
    of trajectory_points, pair i <-> i.  Hypothesis h < max_iteration draws ransac_n pairs with replacement (counter-based
    SplitMix64 from `seed`, DESIGN §4), solves Eigen's Umeyama on them and counts the pairs with |T s_i - r_i|^2 <
    max_correspondence_distance^2: good, and error2 their sum; fitness = good / n, inlier_rmse = sqrt(error2 / good).  Fewer than 3
    distinct indices in a draw: good = 0.  The result is the hypothesis with the most inliers, then the smallest rmse, then the
    smallest h; the identity when none has an inlier.  Its ransac_n-point transform is returned as solved, without a refit.

    -> dict with transformation (fp64 4 x 4, maps the reconstruction's frame into the ground truth's: the init of
    register_tanks_and_temples), fitness, inlier_rmse, inliers, hypothesis (-1: none), sample (its draws), n_correspondences; with
    return_details also, as CUDA tensors, good int32 [max_iteration], error2 fp64 [max_iteration], transforms fp64
    [max_iteration, 3, 4] (NaN where no transform was solved) and samples int32 [max_iteration, ransac_n]."""
    src, tgt = trajectory_points(poses, reference_poses, gt_trans, mapping)
    d_max = _positive(max_correspondence_distance, "max_correspondence_distance")
    if isinstance(ransac_n, bool) or int(ransac_n) != ransac_n or not 3 <= int(ransac_n) <= _lib.PC_RANSAC_MAX_SAMPLE:
        _fail(f"ransac_n must be an integer in 3..{_lib.PC_RANSAC_MAX_SAMPLE}, got {ransac_n!r}")
    if isinstance(max_iteration, bool) or int(max_iteration) != max_iteration or not 0 <= int(max_iteration) < 2 ** 31:
        _fail(f"max_iteration must be an integer in 0..2^31 - 1, got {max_iteration!r}")
    if isinstance(seed, bool) or int(seed) != seed or not 0 <= int(seed) < 2 ** 64:
        _fail(f"seed must be an integer in 0..2^64 - 1, got {seed!r}")
    rn, n_hyp, n = int(ransac_n), int(max_iteration), len(src)
    out = {"transformation": np.eye(4), "fitness": 0.0, "inlier_rmse": 0.0, "inliers": 0, "hypothesis": -1, "sample": [],
           "n_correspondences": n}
    dev = torch.device("cuda", torch.cuda.current_device())
    good = torch.empty(n_hyp, dtype=torch.int32, device=dev)
    error2 = torch.empty(n_hyp, dtype=torch.float64, device=dev)
    trans = torch.empty((n_hyp, 3, 4), dtype=torch.float64, device=dev)
    samples = torch.empty((n_hyp, rn), dtype=torch.int32, device=dev) if return_details else None
    if n == 0:                                                                # no pair: no hypothesis can be drawn
        good.zero_(), error2.zero_(), trans.fill_(float("nan"))
        if samples is not None:
            samples.fill_(-1)
    elif n_hyp:
        s, t = torch.from_numpy(src).to(dev), torch.from_numpy(tgt).to(dev)
        record = torch.empty(_lib.PC_RANSAC_RECORD, dtype=torch.float64, device=dev)
        with _timed("pc_ransac_align"):
            _lib.call("mvsb200_pc_ransac_align", s.data_ptr(), t.data_ptr(), n, n_hyp, rn, d_max * d_max, int(bool(with_scaling)),
                      int(seed), good.data_ptr(), error2.data_ptr(), trans.data_ptr(), samples.data_ptr() if return_details else None,
                      record.data_ptr(), _stream())
        r = record.cpu().numpy()                                              # the one read-back
        h = int(r[0])
        if h >= 0:
            T = np.eye(4)
            T[:3] = r[4:16].reshape(3, 4)
            out.update(transformation=T, fitness=float(r[1]) / n, inlier_rmse=float(r[3]), inliers=int(r[1]), hypothesis=h,
                       sample=[int(v) for v in r[16:16 + rn]])
    if return_details:
        out.update(good=good, error2=error2, transforms=trans, samples=samples)
    return out
