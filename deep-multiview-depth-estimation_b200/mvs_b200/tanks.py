"""The Tanks and Temples evaluation (Knapitsch et al. 2017) on the library's kernels: precision, recall and F-score of a
reconstruction at a distance threshold tau, the metric of MVSNet's Table 3 (Yao et al. 2018).  Restated from the evaluation stage
of the official toolbox (python_toolbox/evaluation: run.py, evaluation.py::EvaluateHisto, get_f1_score_histo2) and the Open3D
functions it calls (TransformPoints, SelectionPolygonVolume::CropInPolygon, PointCloud::VoxelDownSample,
ComputePointCloudDistance); DESIGN §4 K9 states the contract and where it differs.

    gt, crop, trans = load_tnt_eval("/data/tnt", "Barn")
    out = evaluate_tanks_and_temples(xyz.cuda(), gt.cuda(), crop, trans, tau=0.01)

`transform` is used as given.  The toolbox first refines `_trans.txt` with three ICP stages; that is
mvs_b200.register_tanks_and_temples (mvs_b200/registration.py), whose `transformation` this takes unchanged:

    reg = register_tanks_and_temples(xyz.cuda(), gt.cuda(), crop, trans, tau=0.01)
    out = evaluate_tanks_and_temples(xyz.cuda(), gt.cuda(), crop, reg["transformation"], tau=0.01)

A reconstruction made with the user's own cameras is first brought near the ground truth by the toolbox's RANSAC over camera
centres, mvs_b200.align_trajectory, from the user's `.log` trajectory and T&T's COLMAP one (read_trajectory, load_tnt_trajectory):

    poses = camera_poses(R, T)                       # the cameras the reconstruction was made with; write_trajectory(path, poses)
    ref, mapping = load_tnt_trajectory("/data/tnt", "Barn")
    init = align_trajectory(poses, ref, trans, mapping=mapping)["transformation"]
    reg = register_tanks_and_temples(xyz.cuda(), gt.cuda(), crop, init, tau=0.01)

The hot paths are kernels of this library: the fp64 transform and polygon crop, the voxel keys and sequential fp64 voxel means,
and K8's grid and exact capped nearest search.  Torch does the plumbing only: compaction, the stable sort, segment bounds, the
`< tau` counts and the histograms.  There is no CPU path."""
from __future__ import annotations

import json
import math
import os
from typing import NamedTuple

import numpy as np
import torch

from . import _lib
from .evaluation import _cloud, _positive, nearest_distance
from .ops import _stream, _timed

STRETCH = 5                                      # the toolbox's plot_stretch: the histograms span [0, stretch * tau)
_AXES = {"x": 0, "y": 1, "z": 2}
_MAX_POLYGON = 1024
_INT_MAX = 2 ** 31 - 1


def _fail(msg):
    raise _lib.MvsB200Error("tanks: " + msg)


class CropVolume(NamedTuple):
    """Open3D's SelectionPolygonVolume: the prism of `polygon` [k, 3] fp64 (only its two columns across `axis` are read) between
    axis_min and axis_max along `axis` ("X", "Y" or "Z")."""
    axis: str
    axis_min: float
    axis_max: float
    polygon: np.ndarray


def _finite(v, what):
    try:
        a = np.asarray(v, dtype=np.float64)
    except (TypeError, ValueError):
        _fail(f"{what} must be numeric")
    if not np.isfinite(a).all():
        _fail(f"{what} must be finite")
    return a


def _crop_volume(axis, axis_min, axis_max, polygon):
    if not isinstance(axis, str) or axis.lower() not in _AXES:
        _fail(f"orthogonal_axis must be x, y or z (either case), got {axis!r}")
    p = _finite(polygon, "bounding_polygon")
    if p.ndim != 2 or p.shape[1] != 3 or not 3 <= p.shape[0] <= _MAX_POLYGON:
        _fail(f"bounding_polygon: [k, 3] with 3 <= k <= {_MAX_POLYGON} expected, got shape {p.shape}")
    return CropVolume(axis.upper(), float(_finite(axis_min, "axis_min")), float(_finite(axis_max, "axis_max")), p.copy())


def read_crop_volume(path):
    """The crop file {scene}.json (Open3D's SelectionPolygonVolume JSON: class_name, orthogonal_axis, axis_min, axis_max,
    bounding_polygon) -> CropVolume.  Refused with MvsB200Error: another class_name, a missing field, an axis letter other than
    x, y, z, a polygon that is not [k, 3] with 3 <= k <= 1024, and non-finite values."""
    with open(path) as f:
        try:
            d = json.load(f)
        except json.JSONDecodeError as e:
            _fail(f"{path}: not JSON ({e})")
    if not isinstance(d, dict) or d.get("class_name") != "SelectionPolygonVolume":
        _fail(f"{path}: class_name SelectionPolygonVolume expected, got {d.get('class_name') if isinstance(d, dict) else d!r}")
    for k in ("orthogonal_axis", "axis_min", "axis_max", "bounding_polygon"):
        if k not in d:
            _fail(f"{path}: no {k}")
    return _crop_volume(d["orthogonal_axis"], d["axis_min"], d["axis_max"], d["bounding_polygon"])


def _affine(transform):
    """A 4 x 4 alignment -> its first three rows as 12 fp64 values, or None for no transform (None or the identity)."""
    if transform is None:
        return None
    a = np.asarray(transform.detach().cpu() if isinstance(transform, torch.Tensor) else transform, dtype=np.float64)
    if a.shape != (4, 4):
        _fail(f"transform: a 4 x 4 matrix expected, got shape {a.shape}")
    if not np.isfinite(a).all():
        _fail("transform must be finite")
    if not np.array_equal(a[3], [0.0, 0.0, 0.0, 1.0]):
        _fail(f"transform: an affine matrix (last row exactly 0, 0, 0, 1) expected, got last row {a[3].tolist()}")
    if np.array_equal(a, np.eye(4)):
        return None
    return np.ascontiguousarray(a[:3].reshape(12))


def crop_points(xyz, crop, transform=None):
    """Transform (when given) and crop the CUDA cloud xyz [n, 3] (fp32 values; DESIGN §4 K9 steps 1-2) -> (the kept points fp64
    [k, 3] after the transform, their int64 indices [k] ascending).  crop: a CropVolume; transform: a 4 x 4 affine matrix or None."""
    x = _cloud(xyz, "xyz")
    if not isinstance(crop, CropVolume):
        _fail(f"crop must be a CropVolume (read_crop_volume), got {type(crop).__name__}")
    crop = _crop_volume(*crop)
    a = _affine(transform)
    dev = x.device
    n = x.shape[0]
    if n == 0:
        return torch.empty((0, 3), dtype=torch.float64, device=dev), torch.empty(0, dtype=torch.int64, device=dev)
    poly = torch.from_numpy(crop.polygon).to(dev)
    out = torch.empty((n, 3), dtype=torch.float64, device=dev)
    keep = torch.empty(n, dtype=torch.uint8, device=dev)
    a_host = a.ctypes.data_as(_lib._c.c_void_p) if a is not None else None
    with _timed("pc_transform_crop"):
        _lib.call("mvsb200_pc_transform_crop", x.data_ptr(), n, a_host, poly.data_ptr(), poly.shape[0], _AXES[crop.axis.lower()],
                  crop.axis_min, crop.axis_max, out.data_ptr(), keep.data_ptr(), _stream())
    kept = torch.nonzero(keep).reshape(-1)
    return out[kept], kept


def voxel_keys(xyz64, voxel):
    """Open3D's voxel indices of the CUDA fp64 cloud xyz64 [n, 3], n >= 1: vmin = min - voxel * 0.5 per axis, i = floor((p - vmin)
    / voxel) -> int64 keys (iz ny + iy) nx + ix [n].  Refused as Open3D refuses it: voxel * INT_MAX < the largest extent of the
    padded box; and nx ny nz >= 2^62."""
    n = xyz64.shape[0]
    lo, hi = (v.cpu().numpy() for v in torch.aminmax(xyz64, dim=0))
    vmin, vmax = lo - voxel * 0.5, hi + voxel * 0.5
    if voxel * _INT_MAX < float((vmax - vmin).max()):
        _fail(f"voxel {voxel} is too small for an extent of {float((vmax - vmin).max())} (voxel * INT_MAX < extent)")
    nb = [int(np.floor((h - o) / voxel)) + 1 for h, o in zip(hi, vmin)]
    if math.prod(nb) >= 1 << 62:
        _fail(f"{nb} voxels: the int64 keys need nx ny nz < 2^62")
    keys = torch.empty(n, dtype=torch.int64, device=xyz64.device)
    with _timed("pc_voxel_keys"):
        _lib.call("mvsb200_pc_voxel_keys", xyz64.data_ptr(), n, *[float(o) for o in vmin], float(voxel), *nb, keys.data_ptr(), _stream())
    return keys


def voxel_means(xyz64, keys):
    """The voxel means of xyz64 [n, 3] for its keys [n]: a stable sort, the segments of equal keys, then one thread per voxel
    -> (mean fp64 [v, 3], mean fp32 [v, 3], counts int64 [v]) in ascending key order."""
    skeys, perm = torch.sort(keys, stable=True)
    counts = torch.unique_consecutive(skeys, return_counts=True)[1]
    v = counts.shape[0]
    dev = xyz64.device
    offsets = torch.zeros(v + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=offsets[1:])
    mean = torch.empty((v, 3), dtype=torch.float64, device=dev)
    mean32 = torch.empty((v, 3), dtype=torch.float32, device=dev)
    with _timed("pc_voxel_mean"):
        _lib.call("mvsb200_pc_voxel_mean", xyz64.data_ptr(), perm.data_ptr(), offsets.data_ptr(), v, mean.data_ptr(), mean32.data_ptr(),
                  _stream())
    return mean, mean32, counts


def voxel_down_sample(xyz64, voxel):
    """Open3D's VoxelDownSample of the CUDA cloud xyz64 [n, 3] fp64 (DESIGN §4 K9 step 3): one point per occupied voxel, the sum of
    its points in ascending input order added one after another from 0 in fp64, divided by their count -> (mean fp64 [v, 3],
    mean fp32 [v, 3], counts int64 [v]), in ascending voxel key order (Open3D's is hash-map order)."""
    if not isinstance(xyz64, torch.Tensor) or not xyz64.is_cuda:
        _fail("xyz64 must be a CUDA tensor; mvs_b200 has no CPU path")
    if xyz64.dtype != torch.float64 or xyz64.dim() != 2 or xyz64.shape[1] != 3:
        _fail(f"xyz64: fp64 points [n, 3] expected, got {xyz64.dtype} {tuple(xyz64.shape)}")
    if xyz64.shape[0] >= _INT_MAX:
        _fail(f"xyz64: at most 2^31 - 1 points, got {xyz64.shape[0]}")
    voxel = _positive(voxel, "voxel")
    x = xyz64.detach().contiguous()
    dev = x.device
    if x.shape[0] == 0:
        return (torch.empty((0, 3), dtype=torch.float64, device=dev), torch.empty((0, 3), dtype=torch.float32, device=dev),
                torch.empty(0, dtype=torch.int64, device=dev))
    if not bool(torch.isfinite(x).all()):
        _fail("xyz64: coordinates must be finite")
    return voxel_means(x, voxel_keys(x, voxel))


def histogram_edges(tau, stretch=STRETCH):
    """The toolbox's bins: np.arange(0, tau * stretch, tau / 100)."""
    return np.arange(0, tau * stretch, tau / 100)


def _histogram(d, edges):
    """np.histogram(d, edges) on the device: bins [e_k, e_k+1), the last one closed, values outside [e_0, e_K] dropped."""
    d64 = d.double()
    k = edges.numel() - 1
    idx = (torch.searchsorted(edges, d64, right=True) - 1).clamp_(max=k - 1)
    valid = (d64 >= edges[0]) & (d64 <= edges[-1])
    return torch.bincount(idx[valid], minlength=k)


def statistics(d_s, d_t, tau, edges):
    """-> host int64 [2 + 2K]: #(d_s < tau), #(d_t < tau), then the K-bin histograms of d_s and d_t over `edges` (one read-back)."""
    e = torch.from_numpy(edges).to(d_s.device)
    return torch.cat([(d_s.double() < tau).sum().view(1), (d_t.double() < tau).sum().view(1), _histogram(d_s, e),
                      _histogram(d_t, e)]).cpu().numpy()


def search_cap(tau, stretch, edges):
    """The max_dist of both searches: stretch * tau rounded to fp32, raised by one fp32 step when that rounding is not above
    stretch * tau and the last edge, so that every distance the counts or the histograms can see is below it."""
    cap = np.float32(stretch * tau)
    if float(cap) <= max(stretch * tau, float(edges[-1]), tau):
        cap = np.nextafter(cap, np.float32(np.inf))
    return float(cap)


def evaluate_tanks_and_temples(xyz, gt, crop, transform, tau, *, stretch=STRETCH, return_details=False):
    """The Tanks and Temples evaluation of a reconstruction xyz [n, 3] against the ground truth gt [m, 3] (CUDA tensors, fp32
    values) at threshold tau > 0 (DESIGN §4 K9).

    1. The reconstruction is transformed by `transform` (4 x 4 affine, last row exactly 0 0 0 1; None: identity) in fp64.
    2. Both clouds are cropped to `crop` (a CropVolume, read_crop_volume).
    3. Both are voxel down-sampled at tau / 2 (fp64 means).
    4. d_s: from each down-sampled reconstruction point to the nearest down-sampled GT point; d_t the other way; both exact fp32
       distances on the down-sampled points rounded to fp32, +inf at or above a cap just above stretch * tau.
    5. precision = #(d_s < tau) / len(d_s), recall = #(d_t < tau) / len(d_t), fscore = 2 recall precision / (recall + precision),
       and the cumulative histograms cum = cumsum(np.histogram(d, edges)) / len(d) with edges = np.arange(0, tau stretch, tau / 100).
       Either cloud empty after down-sampling: all zeros and edges = cum = [0], as the toolbox.  precision + recall = 0: fscore = 0
       (the toolbox raises ZeroDivisionError there).

    -> dict with precision, recall, fscore, tau, n, n_cropped, n_down, m, m_cropped, m_down, n_precision, m_recall, edges,
    cum_precision, cum_recall (numpy fp64); with return_details also xyz_down, gt_down (fp64 [v, 3]) and d_s, d_t (fp32), on the
    device of xyz."""
    x = _cloud(xyz, "xyz")
    g = _cloud(gt, "gt")
    tau = _positive(tau, "tau")
    stretch = _positive(stretch, "stretch")
    edges = histogram_edges(tau, stretch)
    if len(edges) < 2:
        _fail(f"stretch {stretch} gives no histogram bin: stretch > 0.01 expected")
    xs, _ = crop_points(x, crop, transform)
    gs, _ = crop_points(g, crop, None)
    empty64 = torch.empty((0, 3), dtype=torch.float64, device=x.device)
    empty32 = torch.empty((0, 3), dtype=torch.float32, device=x.device)
    s64, s32, _ = voxel_down_sample(xs, tau / 2) if xs.shape[0] else (empty64, empty32, None)
    t64, t32, _ = voxel_down_sample(gs, tau / 2) if gs.shape[0] else (empty64, empty32, None)
    n_down, m_down = s64.shape[0], t64.shape[0]
    out = {"tau": tau, "n": x.shape[0], "n_cropped": xs.shape[0], "n_down": n_down, "m": g.shape[0], "m_cropped": gs.shape[0],
           "m_down": m_down}
    if n_down == 0 or m_down == 0:
        d_s = torch.full((n_down,), float("inf"), dtype=torch.float32, device=x.device)
        d_t = torch.full((m_down,), float("inf"), dtype=torch.float32, device=x.device)
        zero = np.array([0])
        out.update(precision=0.0, recall=0.0, fscore=0.0, n_precision=0, m_recall=0, edges=zero, cum_precision=zero, cum_recall=zero)
    else:
        cap = search_cap(tau, stretch, edges)
        d_s = nearest_distance(s32, t32, cap)
        d_t = nearest_distance(t32, s32, cap)
        k = len(edges) - 1
        counts = statistics(d_s, d_t, tau, edges)
        n_prec, m_rec = int(counts[0]), int(counts[1])
        precision, recall = float(n_prec) / float(n_down), float(m_rec) / float(m_down)
        fscore = 2 * recall * precision / (recall + precision) if recall + precision > 0 else 0.0
        out.update(precision=precision, recall=recall, fscore=fscore, n_precision=n_prec, m_recall=m_rec, edges=edges,
                   cum_precision=np.cumsum(counts[2:2 + k]).astype(float) / n_down,
                   cum_recall=np.cumsum(counts[2 + k:]).astype(float) / m_down)
    if return_details:
        out.update(xyz_down=s64, gt_down=t64, d_s=d_s, d_t=d_t)
    return out


# matplotlib's "hot" segment data (x, value) per channel, as read from matplotlib's _cm.py, not diffed (matplotlib is not a
# dependency); LinearSegmentedColormap interpolates them at N = 256 evenly spaced points, and "hot_r" is that table reversed
_HOT = {"red": ((0.0, 0.0416), (0.365079, 1.0), (1.0, 1.0)),
        "green": ((0.0, 0.0), (0.365079, 0.0), (0.746032, 1.0), (1.0, 1.0)),
        "blue": ((0.0, 0.0), (0.746032, 0.0), (1.0, 1.0))}
COLOUR_CLIP = 3                                  # the toolbox colours distances up to 3 tau (as read here, not diffed)
NORMALS_KNN = 20                                 # the toolbox's KDTreeSearchParamKNN(knn=20) (as read here, not diffed)


def hot_r_table(N=256):
    """matplotlib's hot_r lookup table -> fp64 [N, 3] (RGB): row 0 is (1, 1, 1), row N - 1 is (0.0416, 0, 0)."""
    idx = np.arange(N, dtype=np.float64)
    lut = np.stack([np.interp(idx, [x * (N - 1) for x, _ in _HOT[c]], [v for _, v in _HOT[c]]) for c in ("red", "green", "blue")], 1)
    return np.clip(lut, 0.0, 1.0)[::-1].copy()


def hot_r(x, N=256):
    """A matplotlib colormap call on values x in [0, 1]: row int(x N) of hot_r_table, with x = 1 mapped to the last row -> fp64 [.., 3]."""
    i = np.floor(np.asarray(x, dtype=np.float64) * N)
    i = np.clip(np.where(i == N, N - 1, i), 0, N - 1).astype(np.int64)
    return hot_r_table(N)[i]


def distance_colours(d, tau, clip=COLOUR_CLIP):
    """The toolbox's colours of distances d (any shape, +inf allowed): hot_r(min(d, clip tau) / (clip tau)), fp64 [.., 3]."""
    top = clip * tau
    return hot_r(np.minimum(np.asarray(d, dtype=np.float64), top) / top)


def write_evaluation_files(directory, scene, result, *, knn=NORMALS_KNN, stretch=STRETCH):
    """The per-scene files of the toolbox's EvaluateHisto from evaluate_tanks_and_temples(..., return_details=True) -> their paths:
        {scene}.precision.ply        xyz_down (rounded to fp32), estimate_normals(k=knn) with the canonical sign, distance_colours(d_s)
        {scene}.recall.ply           the same for gt_down and d_t
        {scene}.precision.txt        np.savetxt of cum_precision
        {scene}.recall.txt           np.savetxt of cum_recall
        {scene}.prf_tau_plotstr.txt  np.savetxt of [precision, recall, fscore, tau, stretch]
    The names, contents and PLY property order are the toolbox's and Open3D's as read here, not diffed.  Refused with MvsB200Error:
    a result without the details."""
    from .fusion import write_ply
    from .normals import estimate_normals
    missing = [k for k in ("xyz_down", "gt_down", "d_s", "d_t") if k not in result]
    if missing:
        _fail(f"write_evaluation_files: the result has no {', '.join(missing)}: evaluate with return_details=True")
    os.makedirs(directory, exist_ok=True)
    base = os.path.join(directory, scene)
    tau = float(result["tau"])
    paths = []
    for name, pts, d in (("precision", result["xyz_down"], result["d_s"]), ("recall", result["gt_down"], result["d_t"])):
        p32 = pts.float().contiguous()
        path = f"{base}.{name}.ply"
        write_ply(path, p32, distance_colours(d.double().cpu().numpy(), tau), normals=estimate_normals(p32, knn))
        paths.append(path)
    return paths + write_curves(directory, scene, result, stretch=stretch)


def write_curves(directory, scene, result, *, stretch=STRETCH):
    """The three text files of write_evaluation_files ({scene}.precision.txt, .recall.txt, .prf_tau_plotstr.txt) -> their paths."""
    base = os.path.join(directory, scene)
    paths = []
    for name, key in (("precision", "cum_precision"), ("recall", "cum_recall")):
        paths.append(f"{base}.{name}.txt")
        np.savetxt(paths[-1], np.asarray(result[key], dtype=np.float64))
    paths.append(f"{base}.prf_tau_plotstr.txt")
    np.savetxt(paths[-1], np.array([result["precision"], result["recall"], result["fscore"], float(result["tau"]), float(stretch)]))
    return paths


def load_tnt_eval(root, scene):
    """Tanks and Temples' evaluation files of one scene -> (gt fp32 [m, 3] CPU tensor, CropVolume, transform fp64 [4, 4]), read from
        {root}/{scene}/{scene}.ply          the ground-truth points
        {root}/{scene}/{scene}.json         the crop volume
        {root}/{scene}/{scene}_trans.txt    the alignment of T&T's COLMAP frame to the ground truth's"""
    from .fusion import read_ply
    d = os.path.join(root, scene)
    paths = [os.path.join(d, f"{scene}.ply"), os.path.join(d, f"{scene}.json"), os.path.join(d, f"{scene}_trans.txt")]
    for p in paths:
        if not os.path.exists(p):
            _fail(f"load_tnt_eval: {p} not found")
    gt, _ = read_ply(paths[0])
    crop = read_crop_volume(paths[1])
    try:
        trans = np.loadtxt(paths[2], dtype=np.float64)
    except ValueError as e:
        _fail(f"load_tnt_eval: {paths[2]}: {e}")
    if trans.shape != (4, 4):
        _fail(f"load_tnt_eval: {paths[2]}: a 4 x 4 matrix expected, got shape {trans.shape}")
    return gt, crop, trans


# ---- trajectories (the toolbox's trajectory_io.py and registration.py::read_mapping; DESIGN §4 "K9 trajectory alignment") ----------

class Mapping(NamedTuple):
    """T&T's {scene}_mapping_reference.txt: rows [n_sampled, 2] int64, where the sparse trajectory takes traj[rows[k, 1] - 1] (the
    second column is 1-based), and n_total, the frame count the file states (not used by the alignment)."""
    n_total: int
    rows: np.ndarray


def _lines(path):
    """The non-blank lines of a text file, each split into its fields, with their 1-based line numbers."""
    with open(path) as f:
        return [(k + 1, ln.split()) for k, ln in enumerate(f) if ln.strip()]


def _ints(fields, path, line, count):
    try:
        v = [int(x) for x in fields]
    except ValueError:
        _fail(f"{path}:{line}: integers expected, got {' '.join(fields)!r}")
    if len(v) != count:
        _fail(f"{path}:{line}: {count} integers expected, got {len(v)}")
    return v


def read_trajectory(path):
    """A trajectory file (.log): per camera one line of three integers (metadata, not interpreted) and four lines of its 4 x 4
    camera-to-world pose -> (metadata int64 [n, 3], poses fp64 [n, 4, 4]).  Blank lines are skipped.  Refused with MvsB200Error: a
    short block, a line with the wrong number of values, a non-numeric or non-finite value, a pose whose last row is not exactly
    0 0 0 1."""
    lines = _lines(path)
    if len(lines) % 5:
        _fail(f"{path}: {len(lines)} lines do not make blocks of 5 (metadata and a 4 x 4 pose): the last block is short")
    meta = np.zeros((len(lines) // 5, 3), np.int64)
    poses = np.zeros((len(lines) // 5, 4, 4))
    for b in range(len(meta)):
        line, fields = lines[5 * b]
        meta[b] = _ints(fields, path, line, 3)
        for r in range(4):
            line, fields = lines[5 * b + 1 + r]
            try:
                row = [float(x) for x in fields]
            except ValueError:
                _fail(f"{path}:{line}: numbers expected, got {' '.join(fields)!r}")
            if len(row) != 4 or not np.isfinite(row).all():
                _fail(f"{path}:{line}: a pose row of 4 finite numbers expected, got {' '.join(fields)!r}")
            poses[b, r] = row
        if not np.array_equal(poses[b, 3], [0.0, 0.0, 0.0, 1.0]):
            _fail(f"{path}: pose {b}: last row exactly 0 0 0 1 expected, got {poses[b, 3].tolist()}")
    return meta, poses


def write_trajectory(path, poses, metadata=None):
    """Write poses [n, 4, 4] (camera-to-world) as a trajectory file.  metadata [n, 3] integers; default i, i, i + 1 per camera i, as
    Open3D's LOG writer writes it (the toolbox's reader ignores it).  Values are written with 17 significant digits, so
    read_trajectory gives back the same fp64 poses."""
    p = np.asarray(poses, np.float64)
    if p.ndim != 3 or p.shape[1:] != (4, 4):
        _fail(f"write_trajectory: poses [n, 4, 4] expected, got shape {p.shape}")
    m = np.stack([np.arange(len(p))] * 2 + [np.arange(1, len(p) + 1)], 1) if metadata is None else np.asarray(metadata)
    if m.shape != (len(p), 3) or not np.array_equal(m, np.asarray(m, np.int64)):
        _fail(f"write_trajectory: metadata [{len(p)}, 3] integers expected, got shape {m.shape}")
    with open(path, "w") as f:
        for k in range(len(p)):
            f.write(" ".join(str(int(v)) for v in m[k]) + "\n")
            for r in range(4):
                f.write(" ".join(f"{v:.17g}" for v in p[k, r]) + "\n")


def read_mapping(path):
    """T&T's {scene}_mapping_reference.txt: n_sampled, n_total, then n_sampled lines of two integers -> Mapping.  Refused with
    MvsB200Error: non-integer values, a row that is not two integers, or a row count other than n_sampled."""
    lines = _lines(path)
    if len(lines) < 2:
        _fail(f"{path}: n_sampled and n_total expected on the first two lines")
    n_sampled = _ints(lines[0][1], path, lines[0][0], 1)[0]
    n_total = _ints(lines[1][1], path, lines[1][0], 1)[0]
    rows = np.array([_ints(f, path, line, 2) for line, f in lines[2:]], np.int64).reshape(-1, 2)
    if len(rows) != n_sampled:
        _fail(f"{path}: n_sampled is {n_sampled} but {len(rows)} mapping rows follow")
    return Mapping(n_total, rows)


def load_tnt_trajectory(root, scene):
    """T&T's reference trajectory of one scene -> (COLMAP poses fp64 [n, 4, 4], Mapping or None), read from
        {root}/{scene}/{scene}_COLMAP_SfM.log            the camera poses of T&T's COLMAP reconstruction
        {root}/{scene}/{scene}_mapping_reference.txt     which video frames those cameras are (None when the file is absent)"""
    d = os.path.join(root, scene)
    log = os.path.join(d, f"{scene}_COLMAP_SfM.log")
    if not os.path.exists(log):
        _fail(f"load_tnt_trajectory: {log} not found")
    mp = os.path.join(d, f"{scene}_mapping_reference.txt")
    return read_trajectory(log)[1], (read_mapping(mp) if os.path.exists(mp) else None)


def camera_poses(R, T):
    """MVSNet's world-to-camera extrinsics R [n, 3, 3], T [n, 3] (or [n, 3, 1]) -> camera-to-world poses [R^T | -R^T T; 0 0 0 1]
    fp64 [n, 4, 4], the poses a trajectory file holds."""
    R = _finite(R.detach().cpu() if isinstance(R, torch.Tensor) else R, "R")
    T = _finite(T.detach().cpu() if isinstance(T, torch.Tensor) else T, "T")
    if R.ndim != 3 or R.shape[1:] != (3, 3) or T.shape not in ((len(R), 3), (len(R), 3, 1)):
        _fail(f"camera_poses: R [n, 3, 3] and T [n, 3] expected, got {R.shape} and {T.shape}")
    Rt = R.transpose(0, 2, 1)
    out = np.zeros((len(R), 4, 4))
    out[:, :3, :3] = Rt
    out[:, :3, 3] = -(Rt @ T.reshape(-1, 3, 1))[..., 0]
    out[:, 3, 3] = 1.0
    return out
