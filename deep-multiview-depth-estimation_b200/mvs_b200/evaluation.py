"""Point-cloud evaluation on the library's kernels (csrc/pointcloud.cu): the DTU protocol of accuracy and completeness, the metric
MVSNet is judged by (Yao et al. 2018, Table 1), restated from the official MATLAB scripts (BaseEvalMain_web.m, reducePts_haa.m,
MaxDistCP.m, ComputeStat_web.m) with their quirks, so that the numbers compare with published tables.

    xyz, rgb, _ = fuse_depth_maps(...)                  # or read_ply("scan.ply")
    stl, obs_mask, bb, res, plane = load_dtu_eval("/data/dtu_eval", scan=1)
    stats = evaluate_point_cloud(xyz.cuda(), stl.cuda(), obs_mask, bb, res, plane)

The hot paths are kernels of this library: a uniform grid (fp64 cell keys, a stable torch sort, cell and block ranges), the exact
capped nearest-distance search and the greedy thinning as parallel rounds.  Torch does the plumbing only: the sort, a cumsum, the
permutation bookkeeping, the fp64 mask and plane passes and the fp64 reductions of the statistics.  There is no CPU path."""
from __future__ import annotations

import math
import os

import numpy as np
import torch

from . import _lib
from .ops import _stream, _timed

DST, MAX_DIST, BLOCK = 0.2, 20.0, 60.0          # DTU's values (BaseEvalMain_web.m)
CELLS_PER_POINT = 0.25                           # search grid: one cell per 4 target points (measured, DESIGN §4 K8) ...
KNN_CELLS_PER_POINT = 2.0                        # ... and for k-nearest searches: two cells per point (measured, DESIGN §4 K10)
THIN_CELLS_PER_POINT = 16                        # thinning grid: finer, fewer candidates in the 27 cells around a point ...
CELL_BUDGET = 1 << 26                            # ... and at most 2^26 cells (512 MB of {begin, end} pairs)
_MAX_POINTS = (1 << 31) - 1


def _fail(msg):
    raise _lib.MvsB200Error("evaluation: " + msg)


def _cloud(t, what):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        _fail(f"{what} must be a CUDA tensor; mvs_b200 has no CPU path")
    if t.dim() != 2 or t.shape[1] != 3:
        _fail(f"{what}: points [n, 3] expected, got {tuple(t.shape)}")
    if t.shape[0] >= _MAX_POINTS:
        _fail(f"{what}: at most 2^31 - 1 points (int32 indices), got {t.shape[0]}")
    t = t.detach().to(torch.float32).contiguous()
    if t.numel() and not bool(torch.isfinite(t).all()):
        _fail(f"{what}: coordinates must be finite")
    return t


def _positive(v, what):
    v = float(v)
    if not (v > 0 and math.isfinite(v)):
        _fail(f"{what} must be > 0 and finite, got {v}")
    return v


class Grid:
    """A uniform grid over a cloud: pts [m, 4] (x, y, z, original index) in cell order, cells / blocks {begin, end} into pts,
    fine cells of edge `cell` from `origin`, in `nb` coarse blocks of 8^3 cells per axis; `perm` the sort permutation."""

    def __init__(self, pts, cells, blocks, perm, origin, cell, nb):
        self.pts, self.cells, self.blocks, self.perm = pts, cells, blocks, perm
        self.origin, self.cell, self.nb = origin, cell, nb

    def args(self):
        return (*[float(o) for o in self.origin], float(self.cell), *[int(b) for b in self.nb])

    def slack(self):
        """What the kernels subtract from every distance lower bound: above the fp32 rounding of the cell faces."""
        top = max(max(abs(o), abs(o + 8 * b * self.cell)) for o, b in zip(self.origin, self.nb))
        return 1e-5 * self.cell + 2.4e-7 * top


def cell_size(lo, hi, m, min_cell=0.0, cells_per_point=CELLS_PER_POINT, budget=CELL_BUDGET):
    """The fine cell edge for a cloud of m points in the box [lo, hi]: the box's volume over cells_per_point * m cells (each extent
    taken as at least 1e-3 of the largest, so flat clouds get cells too), at least min_cell, grown by 10 % steps until the grid
    (padded to whole 8^3 blocks) has at most `budget` cells -> (cell, blocks per axis)."""
    ext = [max(float(h) - float(l), 0.0) for l, h in zip(lo, hi)]
    big = max(ext)
    if big > 0:
        vol = math.prod(max(e, 1e-3 * big) for e in ext)
        cell = (vol / max(cells_per_point * m, 1)) ** (1.0 / 3.0)
    else:
        cell = 1.0
    cell = max(cell, float(min_cell), 1e-30)
    while True:
        cell = float(np.float32(cell))
        nb = [(int(math.floor(e / cell)) + 1 + 7) // 8 for e in ext]
        if 512 * math.prod(nb) <= budget:
            return cell, nb
        cell *= 1.1


def build_grid(xyz, cell=None, min_cell=0.0, cells_per_point=CELLS_PER_POINT):
    """Grid over the CUDA cloud xyz [m, 3] fp32, m >= 1 (cell=None: the rule of cell_size)."""
    m = xyz.shape[0]
    lo, hi = (v.cpu().tolist() for v in torch.aminmax(xyz, dim=0))
    if cell is None:
        cell, nb = cell_size(lo, hi, m, min_cell, cells_per_point)
    else:                                   # an explicit cell edge (benchmarks, tests): no budget beyond the kernels' bound
        cell = float(np.float32(max(float(cell), float(min_cell))))
        nb = [(int(math.floor((h - l) / cell)) + 1 + 7) // 8 for l, h in zip(lo, hi)]
        if 512 * math.prod(nb) > _lib.PC_MAX_CELLS:
            _fail(f"a grid of cell {cell} over this cloud has more than {_lib.PC_MAX_CELLS} cells")
    dev = xyz.device
    keys = torch.empty(m, dtype=torch.int32, device=dev)
    args = (*lo, cell, *nb)
    with _timed("pc_grid_keys"):
        _lib.call("mvsb200_pc_grid_keys", xyz.data_ptr(), m, *args, keys.data_ptr(), _stream())
    skeys, perm = torch.sort(keys, stable=True)
    pts = torch.empty((m, 4), dtype=torch.float32, device=dev)
    n_blocks = math.prod(nb)
    cells = torch.zeros((n_blocks * 512, 2), dtype=torch.int32, device=dev)
    blocks = torch.zeros((n_blocks, 2), dtype=torch.int32, device=dev)
    with _timed("pc_grid_cells"):
        _lib.call("mvsb200_pc_grid_cells", xyz.data_ptr(), skeys.data_ptr(), perm.data_ptr(), m, pts.data_ptr(), cells.data_ptr(),
                  blocks.data_ptr(), _stream())
    return Grid(pts, cells, blocks, perm, lo, cell, nb)


def nearest_distance(query, target, max_dist, *, grid=None):
    """For every query point [n, 3] the distance to its nearest target point [m, 3] (CUDA tensors) -> fp32 [n]: exact (fp32
    arithmetic on the fp32 coordinates) where it is below max_dist, +inf where no target point lies within max_dist (and
    everywhere for an empty target).  grid: a build_grid(target) to reuse.  Two calls return the same bits."""
    q = _cloud(query, "query")
    t = _cloud(target, "target")
    max_dist = _positive(max_dist, "max_dist")
    n, m = q.shape[0], t.shape[0]
    out = torch.full((n,), float("inf"), dtype=torch.float32, device=q.device)
    if n == 0 or m == 0:
        return out
    g = grid if grid is not None else build_grid(t)
    with _timed("pc_nearest"):
        _lib.call("mvsb200_pc_nearest", q.data_ptr(), n, g.pts.data_ptr(), g.cells.data_ptr(), g.blocks.data_ptr(), *g.args(),
                  float(g.slack()), max_dist, out.data_ptr(), _stream())
    return out


def nearest_index_into(q, g, max_dist, dist, index):
    """The index-returning search of the fp32 CUDA points q [n, 3], n >= 1, on the grid g, into dist fp32 [n] and index int32 [n]."""
    with _timed("pc_nearest_index"):
        _lib.call("mvsb200_pc_nearest_index", q.data_ptr(), q.shape[0], g.pts.data_ptr(), g.cells.data_ptr(), g.blocks.data_ptr(),
                  *g.args(), float(g.slack()), float(max_dist), dist.data_ptr(), index.data_ptr(), _stream())


def nearest_neighbour(query, target, max_dist, *, grid=None):
    """nearest_distance, and which target point it is -> (dist fp32 [n], index int64 [n]): index[i] is the row of `target` nearest to
    query[i] (the smaller row on an exact tie of the fp32 distance), -1 where dist[i] is +inf.  Same search, same distances."""
    q = _cloud(query, "query")
    t = _cloud(target, "target")
    max_dist = _positive(max_dist, "max_dist")
    n, m = q.shape[0], t.shape[0]
    dist = torch.full((n,), float("inf"), dtype=torch.float32, device=q.device)
    index = torch.full((n,), -1, dtype=torch.int32, device=q.device)
    if n and m:
        nearest_index_into(q, grid if grid is not None else build_grid(t), max_dist, dist, index)
    return dist, index.long()


def knn_k(k):
    """k as an int in [1, PC_KNN_MAX], refused otherwise."""
    if isinstance(k, bool) or int(k) != k or not 1 <= int(k) <= _lib.PC_KNN_MAX:
        _fail(f"k must be an integer in [1, {_lib.PC_KNN_MAX}], got {k!r}")
    return int(k)


def knn_cap(max_dist):
    """max_dist of a k-nearest search: > 0, +inf meaning no cap."""
    v = float(max_dist)
    if not v > 0:
        _fail(f"max_dist must be > 0 (+inf: no cap), got {v}")
    return v


def k_nearest(query, target, k, max_dist=math.inf, *, grid=None):
    """The k nearest target points [m, 3] of every query point [n, 3] (CUDA tensors) -> (dist fp32 [n, k], index int64 [n, k]).

    Row i lists the target points that come first in the total order (d^2, row) among those with d < max_dist, ascending: d^2 is
    the fp32 (dx^2 + dy^2) + dz^2 of nearest_distance and d its square root, so ties are exact and go to the smaller row, and
    k = 1 is nearest_neighbour bit for bit.  A row holds fewer than k points only when the cap or the cloud leaves fewer; it is
    padded with +inf / -1.  1 <= k <= 32; max_dist > 0 (+inf: no cap).  grid: a build_grid(target, cells_per_point=
    KNN_CELLS_PER_POINT) to reuse.  Two calls return the same bits."""
    q = _cloud(query, "query")
    t = _cloud(target, "target")
    k = knn_k(k)
    max_dist = knn_cap(max_dist)
    n, m = q.shape[0], t.shape[0]
    dist = torch.full((n, k), float("inf"), dtype=torch.float32, device=q.device)
    index = torch.full((n, k), -1, dtype=torch.int32, device=q.device)
    if n and m:
        g = grid if grid is not None else build_grid(t, cells_per_point=KNN_CELLS_PER_POINT)
        with _timed("pc_knn"):
            _lib.call("mvsb200_pc_knn", q.data_ptr(), n, g.pts.data_ptr(), g.cells.data_ptr(), g.blocks.data_ptr(), *g.args(),
                      float(g.slack()), max_dist, k, dist.data_ptr(), index.data_ptr(), _stream())
    return dist, index.long()


def _order(order, seed, n):
    if order is None:
        return torch.randperm(n, generator=torch.Generator().manual_seed(int(seed)))
    o = torch.as_tensor(np.asarray(order.cpu() if isinstance(order, torch.Tensor) else order)).reshape(-1)
    if o.dtype.is_floating_point or o.dtype == torch.bool or o.numel() != n:
        _fail(f"order must be a permutation of 0..{n - 1} (integers, {n} of them), got {o.numel()} values of {o.dtype}")
    o = o.to(torch.int64)
    if not torch.equal(torch.sort(o).values, torch.arange(n)):
        _fail(f"order must be a permutation of 0..{n - 1}")
    return o


def thin(xyz, dst=DST, *, order=None, seed=0, cell=None):
    """thin_points, plus the number of parallel rounds it took -> (kept int64 [k] ascending, rounds)."""
    x = _cloud(xyz, "xyz")
    dst = _positive(dst, "dst")
    n = x.shape[0]
    o = _order(order, seed, n)
    dev = x.device
    if n == 0:
        return torch.empty(0, dtype=torch.int64, device=dev), 0
    # cell >= dst: every neighbour lies in the 27 cells around a point
    g = build_grid(x, cell=cell, min_cell=dst * (1 + 1e-3), cells_per_point=THIN_CELLS_PER_POINT)
    rank = torch.empty(n, dtype=torch.int32, device=dev)
    rank[o.to(dev)] = torch.arange(n, dtype=torch.int32, device=dev)
    rank_sorted = rank[g.perm].contiguous()
    counts = torch.empty(n, dtype=torch.int32, device=dev)
    with _timed("pc_thin_count"):
        _lib.call("mvsb200_pc_thin_neighbours", g.pts.data_ptr(), g.cells.data_ptr(), rank_sorted.data_ptr(), n, *g.args(), dst,
                  None, counts.data_ptr(), None, _stream())
    offsets = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=offsets[1:])
    total = int(offsets[-1])
    if total >= _MAX_POINTS:
        _fail(f"{total} pairs within dst: the neighbour lists need int32 positions")
    nbrs = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
    with _timed("pc_thin_list"):
        _lib.call("mvsb200_pc_thin_neighbours", g.pts.data_ptr(), g.cells.data_ptr(), rank_sorted.data_ptr(), n, *g.args(), dst,
                  offsets.data_ptr(), None, nbrs.data_ptr(), _stream())
    state = torch.zeros(n, dtype=torch.uint8, device=dev)
    nxt = torch.empty_like(state)
    undecided = torch.zeros(1, dtype=torch.int32, device=dev)
    rounds = 0
    while True:
        # the lowest-ranked undecided point is decided in every round, so n rounds always suffice
        if rounds > n:
            _fail(f"thinning did not converge in {n} rounds")
        undecided.zero_()
        with _timed("pc_thin_round"):
            _lib.call("mvsb200_pc_thin_round", offsets.data_ptr(), nbrs.data_ptr(), state.data_ptr(), nxt.data_ptr(), n,
                      undecided.data_ptr(), _stream())
        state, nxt = nxt, state
        rounds += 1
        if int(undecided.item()) == 0:
            break
    keep = torch.zeros(n, dtype=torch.bool, device=dev)
    keep[g.perm] = state == 1
    return torch.nonzero(keep).reshape(-1), rounds


def thin_points(xyz, dst=DST, *, order=None, seed=0):
    """reducePts_haa: visit the points of the CUDA cloud xyz [n, 3] in `order` (a permutation of 0..n-1; None: drawn from a CPU
    torch.Generator seeded with `seed`, the same on every machine); a visited point still present is kept and removes every
    other point within dst of it (|p - q| <= dst, inclusive, in fp64 on the fp32 coordinates) -> the int64 indices of the kept
    points, ascending.  For a fixed order the result is the lexicographically first maximal independent set of the "within dst"
    graph, computed exactly by parallel greedy rounds."""
    return thin(xyz, dst, order=order, seed=seed)[0]


def _f64(a, shape, what):
    v = np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a, dtype=np.float64)
    if v.size != math.prod(shape):
        _fail(f"{what}: {math.prod(shape)} values expected, got shape {v.shape}")
    if not np.isfinite(v).all():
        _fail(f"{what} must be finite")
    return v.reshape(shape)


def covered(q, bb, block):
    """MaxDistCP's block grid: q [n, 3] is visited iff BB[0,a] <= q_a < BB[0,a] + (R_a + 1) * block on every axis, with
    R_a = floor((BB[1,a] - BB[0,a]) / block); fp64 on the fp32 values -> bool [n]."""
    bb = torch.as_tensor(bb, dtype=torch.float64, device=q.device)
    R = torch.floor((bb[1] - bb[0]) / block)
    q64 = q.double()
    return ((q64 >= bb[0]) & (q64 < bb[0] + (R + 1) * block)).all(1)


def round_half_away(x):
    """MATLAB's round: halves away from zero (torch.round rounds half to even; floor(x + 0.5) is wrong at -0.5)."""
    return torch.sign(x) * torch.floor(torch.abs(x) + 0.5)


def in_mask(q, obs_mask, bb, res):
    """DataInMask: i_a = round_half_away((q_a - BB[0,a]) / Res), in the mask iff 0 <= i_a < ObsMask.shape[a] and ObsMask[i]."""
    bb = torch.as_tensor(bb, dtype=torch.float64, device=q.device)
    i = round_half_away((q.double() - bb[0]) / float(res))
    shape = torch.tensor(obs_mask.shape, dtype=torch.float64, device=q.device)
    inside = ((i >= 0) & (i < shape)).all(1)
    ii = torch.where(inside[:, None], i, torch.zeros_like(i)).to(torch.int64)
    X, Y, Z = obs_mask.shape
    flat = obs_mask.reshape(-1)[(ii[:, 0] * Y + ii[:, 1]) * Z + ii[:, 2]]
    return inside & flat


def above_plane(s, plane):
    """StlAbovePlane: P[0] x + P[1] y + P[2] z + P[3] > 0 in fp64."""
    P = torch.as_tensor(plane, dtype=torch.float64, device=s.device)
    return s.double() @ P[:3] + P[3] > 0


def _mean_median(v):
    """fp64 mean and MATLAB's median (the mean of the two middle values for an even count); NaN for an empty selection."""
    if v.numel() == 0:
        return float("nan"), float("nan")
    v = v.double()
    s = torch.sort(v).values
    k = s.numel()
    med = s[k // 2] if k % 2 else (s[k // 2 - 1] + s[k // 2]) / 2
    return float(v.sum() / k), float(med)


def evaluate_point_cloud(xyz, stl, obs_mask, bb, res, plane, *, dst=DST, max_dist=MAX_DIST, block=BLOCK, order=None, seed=0,
                         return_details=False):
    """The DTU evaluation of a reconstruction xyz [n, 3] against the ground truth stl [m, 3] (both CUDA tensors, fp32).

    Points are fp32 as fuse_depth_maps and PLY files give them.  Every comparison below is defined on those values promoted to fp64.

    1. Thinning (reducePts_haa).  Given a permutation `order` of the data points, visit them in that order.  A visited point that
       is still present is kept, and it removes every other point q with |p - q| <= dst (inclusive, as rangesearch is).  The
       result is the kept subset in original index order.  MATLAB draws `order` with randperm, which cannot be reproduced: pass
       `order`, or a `seed` from which a CPU torch.Generator draws it, so the result is the same on every machine.  For a fixed
       order the greedy result is the lexicographically first maximal independent set of the "within dst" graph.
    2. Distances (MaxDistCP).  Ddata[i] is the distance from reduced data point i to its nearest point of stl; Dstl[j] the
       distance from stl[j] to its nearest reduced data point.  A distance is exact when it is below max_dist, +inf otherwise.
       Quirk kept: MaxDistCP only visits query points inside its block grid.  Per axis a, with
       R_a = floor((BB[1,a] - BB[0,a]) / block), a point is covered iff BB[0,a] <= q_a < BB[0,a] + (R_a + 1) * block.  An
       uncovered query point gets `block`, so the statistics exclude it.
    3. Masks.  DataInMask: i_a = round_half_away((q_a - BB[0,a]) / Res) (MATLAB's round, zero-based here); the point is in the
       mask iff 0 <= i_a < ObsMask.shape[a] on every axis and ObsMask[i] is true.  StlAbovePlane: P[0]x + P[1]y + P[2]z + P[3] > 0.
    4. Statistics (ComputeStat_web).  accuracy = mean of Ddata over DataInMask & Ddata < max_dist; completeness = mean of Dstl
       over StlAbovePlane & Dstl < max_dist; overall = (accuracy + completeness) / 2; the two medians and all counts.  Sums are in
       fp64; an empty selection gives NaN, as MATLAB's mean([]) does.

    obs_mask: bool [X, Y, Z] (any device); bb [2, 3]; res > 0; plane [4] -> dict with accuracy, completeness, overall,
    median_accuracy, median_completeness, n, n_reduced, n_in_mask, n_accuracy, m, m_above_plane, n_completeness, thin_rounds;
    with return_details also kept (int64), Ddata, Dstl (fp32), DataInMask, StlAbovePlane (bool), on the device of xyz."""
    x = _cloud(xyz, "xyz")
    s = _cloud(stl, "stl")
    dst, max_dist, block = _positive(dst, "dst"), _positive(max_dist, "max_dist"), _positive(block, "block")
    res = _positive(res, "res")
    bb = _f64(bb, (2, 3), "bb")
    if (bb[1] < bb[0]).any():
        _fail(f"bb[1] must be >= bb[0] on every axis, got {bb.tolist()}")
    plane = _f64(plane, (4,), "plane")
    mask = torch.as_tensor(obs_mask.detach() if isinstance(obs_mask, torch.Tensor) else np.asarray(obs_mask))
    if mask.dim() != 3:
        _fail(f"obs_mask: a 3-D mask [X, Y, Z] expected, got {tuple(mask.shape)}")
    mask = mask.to(device=x.device, dtype=torch.bool).contiguous()
    kept, rounds = thin(x, dst, order=order, seed=seed)
    q = x[kept].contiguous()
    d_data = nearest_distance(q, s, max_dist)
    d_stl = nearest_distance(s, q, max_dist)
    d_data = torch.where(covered(q, bb, block), d_data, torch.full_like(d_data, block))
    d_stl = torch.where(covered(s, bb, block), d_stl, torch.full_like(d_stl, block))
    data_in = in_mask(q, mask, bb, res)
    stl_above = above_plane(s, plane)
    sel_a = data_in & (d_data.double() < max_dist)
    sel_c = stl_above & (d_stl.double() < max_dist)
    acc, med_a = _mean_median(d_data[sel_a])
    comp, med_c = _mean_median(d_stl[sel_c])
    out = {"accuracy": acc, "completeness": comp, "overall": (acc + comp) / 2, "median_accuracy": med_a,
           "median_completeness": med_c, "n": x.shape[0], "n_reduced": q.shape[0], "n_in_mask": int(data_in.sum()),
           "n_accuracy": int(sel_a.sum()), "m": s.shape[0], "m_above_plane": int(stl_above.sum()), "n_completeness": int(sel_c.sum()),
           "thin_rounds": rounds}
    if return_details:
        out.update(kept=kept, Ddata=d_data, Dstl=d_stl, DataInMask=data_in, StlAbovePlane=stl_above)
    return out


def load_dtu_eval(dtu_root, scan):
    """DTU's evaluation files for one scan -> (stl fp32 [m, 3] CPU tensor, obs_mask bool [X, Y, Z] CPU tensor, bb fp64 [2, 3],
    res float, plane fp64 [4]), read from
        {dtu_root}/Points/stl/stl{scan:03d}_total.ply
        {dtu_root}/ObsMask/ObsMask{scan}_10.mat    (ObsMask, BB, Res)
        {dtu_root}/ObsMask/Plane{scan}.mat         (P)
    Needs scipy (scipy.io.loadmat), imported here so that `import mvs_b200` does not."""
    import scipy.io
    from .fusion import read_ply
    scan = int(scan)
    paths = [os.path.join(dtu_root, "Points", "stl", f"stl{scan:03d}_total.ply"),
             os.path.join(dtu_root, "ObsMask", f"ObsMask{scan}_10.mat"), os.path.join(dtu_root, "ObsMask", f"Plane{scan}.mat")]
    for p in paths:
        if not os.path.exists(p):
            _fail(f"load_dtu_eval: {p} not found")
    stl, _ = read_ply(paths[0])
    m = scipy.io.loadmat(paths[1])
    for k in ("ObsMask", "BB", "Res"):
        if k not in m:
            _fail(f"load_dtu_eval: {paths[1]} has no variable {k}")
    pm = scipy.io.loadmat(paths[2])
    if "P" not in pm:
        _fail(f"load_dtu_eval: {paths[2]} has no variable P")
    obs = torch.from_numpy(np.ascontiguousarray(np.asarray(m["ObsMask"]).astype(bool)))
    return (stl, obs, _f64(m["BB"], (2, 3), "BB"), float(np.asarray(m["Res"], np.float64).reshape(-1)[0]),
            _f64(pm["P"], (4,), "P"))
