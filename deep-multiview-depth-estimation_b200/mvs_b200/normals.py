"""Oriented point-cloud normals on the library's kernels (csrc/pointcloud.cu, DESIGN §4 K10): an exact k-nearest-neighbour search on
K8's grid, then per point the fp64 covariance of its neighbourhood and the eigenvector of its smallest eigenvalue, in one launch.

    xyz, rgb, masks = fuse_depth_maps(depth, conf, colours, K, R, T, sources)
    nrm = estimate_normals(xyz, viewpoints=point_viewpoints(masks, R, T))      # each normal faces the camera that saw the point
    write_ply("scene.ply", xyz, rgb, normals=nrm)

The normals are what Poisson meshing and normal-shaded viewers need, and what Open3D's estimate_normals gives with
KDTreeSearchParamKNN(knn) (max_dist = inf) or KDTreeSearchParamHybrid(radius, max_nn), up to the differences DESIGN §4 K10 lists.
There is no CPU path."""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _lib
from .evaluation import KNN_CELLS_PER_POINT, _cloud, build_grid, knn_cap, knn_k
from .ops import _stream, _timed


def _fail(msg):
    raise _lib.MvsB200Error("normals: " + msg)


def _viewpoints(viewpoints, n, dev):
    """None -> (0, None); one point [3] -> (1, fp64 [3]); one per point [n, 3] -> (2, fp64 [n, 3]), on dev."""
    if viewpoints is None:
        return 0, None
    v = viewpoints.detach() if isinstance(viewpoints, torch.Tensor) else torch.as_tensor(np.asarray(viewpoints, dtype=np.float64))
    v = v.to(device=dev, dtype=torch.float64).contiguous()
    if tuple(v.shape) in ((3,), (1, 3)):
        mode = 1
    elif tuple(v.shape) == (n, 3):
        mode = 2
    else:
        _fail(f"viewpoints: one point [3] or one per point [{n}, 3] expected, got {tuple(v.shape)}")
    if not bool(torch.isfinite(v).all()):
        _fail("viewpoints must be finite")
    return mode, v.reshape(-1, 3)


def estimate_normals(xyz, k=30, *, max_dist=math.inf, viewpoints=None, grid=None):
    """The normal of every point of the CUDA cloud xyz [n, 3] -> fp32 [n, 3] (DESIGN §4 K10).

    1. N(i): the k points of xyz first in the order (d^2, row) among those with d < max_dist (k_nearest of the cloud on itself;
       the point itself is one of them, at distance 0).
    2. C = sum (p - mu)(p - mu)^T / c with mu = sum p / c, c = |N(i)|, in fp64 on the fp32 coordinates, summed in list order.
    3. The unit eigenvector of C's smallest eigenvalue; the zero vector ("no normal") where c < 3 or trace C = 0.
    4. Its component of largest magnitude made positive (the first such axis on a tie); with viewpoints (one point [3], or one per
       point [n, 3]) then flipped iff n . (v - p) < 0 in fp64.  Rounded to fp32 last.

    k: 1..32 (30 is Open3D's default knn); max_dist > 0, +inf for none; grid: build_grid(xyz, cells_per_point=KNN_CELLS_PER_POINT)
    to reuse (it must be built over xyz itself).  Two calls return the same bits."""
    x = _cloud(xyz, "xyz")
    k = knn_k(k)
    max_dist = knn_cap(max_dist)
    n = x.shape[0]
    mode, v = _viewpoints(viewpoints, n, x.device)
    out = torch.zeros((n, 3), dtype=torch.float32, device=x.device)
    if n == 0:
        return out
    g = grid if grid is not None else build_grid(x, cells_per_point=KNN_CELLS_PER_POINT)
    if g.pts.shape[0] != n:
        _fail(f"grid: built over {g.pts.shape[0]} points, not over this cloud of {n}")
    with _timed("pc_normals"):
        _lib.call("mvsb200_pc_normals", x.data_ptr(), n, g.pts.data_ptr(), g.cells.data_ptr(), g.blocks.data_ptr(), *g.args(),
                  float(g.slack()), max_dist, k, v.data_ptr() if v is not None else None, mode, out.data_ptr(), _stream())
    return out
