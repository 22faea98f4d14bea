"""Scene reconstruction after per-view inference: photometric confidence, multi-view consistency filtering and point-cloud fusion
(MVSNet, Yao et al. 2018, §4.2) on the library's kernels (csrc/fusion.cu, the confidence in csrc/softmax_depth.cu).

    depth, conf, colours = infer_scene(FrozenMVSNet(model), images, K, R, T, d_min, d_int, pairs)
    xyz, rgb, masks = fuse_depth_maps(depth, conf, colours, K, R, T, sources)      # or visibility_fusion: each point once
    write_ply("scene.ply", xyz, rgb)

What a depth means.  The network sweeps the planes n^T (X - C_ref) = d with n = R_ref[:, 2], the third COLUMN of R (geometry.py,
DESIGN §1), so the depth d at pixel p = (x, y, 1) of a view stands for the world point X = C + d / (n^T r) r, r = R^T K^-1 p, and
the depth of a point in view j is n_j^T (X - C_j).  `normal` picks n for every view: "sweep" (the network's depths) or
"optical_axis" (n = R[2, :], true z-depth: ground-truth PFM maps, depth maps from elsewhere).  x, y are the integer pixel indices
of the depth map in the coordinates K is written in, i.e. K at depth (feature) resolution, the K the model takes.  The resampling
offset of the sweep's warp (kornia's w / (w - 1), geometry.py) is a property of that warp, not of the geometry, and is not applied.

Thresholds (MVSNet's values): conf_min 0.8, reproj_px 1.0 (pixels), rel_depth 0.01, min_views 3.  There is no CPU path."""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from .ops import _stream, _timed

NORMALS = ("sweep", "optical_axis")
CONF_MIN, REPROJ_PX, REL_DEPTH, MIN_VIEWS = 0.8, 1.0, 0.01, 3


def _fail(msg):
    raise _lib.MvsB200Error("fusion: " + msg)


def _f64(t, shape, what):
    a = t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
    a = np.asarray(a, dtype=np.float64)
    if a.size != int(np.prod(shape)):
        _fail(f"{what}: {int(np.prod(shape))} values ({'x'.join(map(str, shape))}) expected, got shape {a.shape}")
    return a.reshape(shape)


def camera_fields(K, R, T, normal="sweep"):
    """Per view the fp64 fields of the camera table: [N, 32] = K [R | T] (12), R^T K^-1 (9), C = -R^T T (3), n (3), zeros (5)."""
    if normal not in NORMALS:
        _fail(f'normal must be one of {NORMALS}, got {normal!r}')
    N = (K.numel() if isinstance(K, torch.Tensor) else np.asarray(K).size) // 9
    K, R, T = _f64(K, (N, 3, 3), "K"), _f64(R, (N, 3, 3), "R"), _f64(T, (N, 3, 1), "T")
    Rt = np.transpose(R, (0, 2, 1))
    out = np.zeros((N, _lib.FUSION_CAM_FLOATS))
    out[:, 0:12] = (K @ np.concatenate([R, T], 2)).reshape(N, 12)
    out[:, 12:21] = (Rt @ np.linalg.inv(K)).reshape(N, 9)
    out[:, 21:24] = (-Rt @ T).reshape(N, 3)
    out[:, 24:27] = R[:, :, 2] if normal == "sweep" else R[:, 2, :]
    return out


def source_table(sources, N):
    """Source lists (one per view; -1 or a shorter list pads) -> int32 [N, S], S <= 16."""
    if isinstance(sources, torch.Tensor):
        sources = sources.detach().cpu().numpy()
    rows = [np.asarray(s, dtype=np.int64).reshape(-1) for s in sources]
    if len(rows) != N:
        _fail(f"one source list per view expected ({N}), got {len(rows)}")
    S = max((len(r) for r in rows), default=0)
    if S > _lib.FUSION_MAX_SOURCES:
        _fail(f"at most {_lib.FUSION_MAX_SOURCES} sources per view, got {S}")
    table = np.full((N, max(S, 1)), -1, dtype=np.int32)
    for i, r in enumerate(rows):
        if np.any((r < -1) | (r >= N)):
            _fail(f"view {i}: source ids must lie in [0, {N - 1}] (or be -1), got {r.tolist()}")
        table[i, :len(r)] = r
    return table


def _maps(t, N, c, h, w, what):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        _fail(f"{what} must be a CUDA tensor; mvs_b200 has no CPU path")
    if tuple(t.shape) != (N, c, h, w):
        _fail(f"{what}: [{N}, {c}, {h}, {w}] expected, got {tuple(t.shape)}")
    return t.detach().float().contiguous()


def _prepare(depth, conf, K, R, T, sources, normal):
    """The inputs of the check on the device and its outputs (uninitialised): d, c, cams, source table, mask, count, fused, blocks."""
    if not isinstance(depth, torch.Tensor) or not depth.is_cuda:
        _fail("depth must be a CUDA tensor; mvs_b200 has no CPU path")
    if depth.dim() != 4 or depth.shape[1] != 1:
        _fail(f"depth maps [N, 1, h, w] expected, got {tuple(depth.shape)}")
    N, _, h, w = depth.shape
    dev = depth.device
    d = _maps(depth, N, 1, h, w, "depth")
    c = _maps(conf, N, 1, h, w, "conf")
    cams = torch.from_numpy(camera_fields(K, R, T, normal).astype(np.float32)).to(dev)
    if cams.shape[0] != N:
        _fail(f"one camera per depth map expected ({N}), got {cams.shape[0]}")
    src = source_table(sources, N)
    S = src.shape[1]
    src = torch.from_numpy(src).to(dev)
    mask = torch.empty((N, 1, h, w), dtype=torch.uint8, device=dev)
    count = torch.empty((N, 1, h, w), dtype=torch.int32, device=dev)
    fused = torch.empty((N, 1, h, w), dtype=torch.float32, device=dev)
    blocks = torch.empty((N * -(-h * w // _lib.FUSION_BLOCK_PIXELS),), dtype=torch.int32, device=dev)
    return d, c, cams, src, mask, count, fused, blocks


def _check(depth, conf, K, R, T, sources, normal, conf_min, reproj_px, rel_depth, min_views):
    d, c, cams, src, mask, count, fused, blocks = _prepare(depth, conf, K, R, T, sources, normal)
    N, _, h, w = depth.shape
    with _timed("fusion_check"):
        _lib.call("mvsb200_fusion_check", d.data_ptr(), c.data_ptr(), cams.data_ptr(), src.data_ptr(), N, src.shape[1], h, w,
                  float(conf_min), float(reproj_px), float(rel_depth), int(min_views), mask.data_ptr(), count.data_ptr(),
                  fused.data_ptr(), blocks.data_ptr(), _stream())
    return mask, count, fused, blocks, cams


def _emit(mask, fused, blocks, cams, colours):
    """The kept pixels of every view -> (xyz, rgb), view-major, row-major; the one device-to-host read is the point count."""
    N, _, h, w = mask.shape
    col = _maps(colours, N, 3, h, w, "colours")
    offsets = torch.cumsum(blocks, 0) - blocks                    # exclusive scan, int64
    M = int(offsets[-1] + blocks[-1]) if blocks.numel() else 0
    xyz = torch.empty((M, 3), dtype=torch.float32, device=mask.device)
    rgb = torch.empty((M, 3), dtype=torch.float32, device=mask.device)
    if M:
        with _timed("fusion_emit"):
            _lib.call("mvsb200_fusion_emit", mask.data_ptr(), fused.data_ptr(), col.data_ptr(), cams.data_ptr(), offsets.data_ptr(),
                      N, h, w, xyz.data_ptr(), rgb.data_ptr(), _stream())
    return xyz, rgb


def check_consistency(depth, conf, K, R, T, sources, *, normal="sweep", conf_min=CONF_MIN, reproj_px=REPROJ_PX,
                      rel_depth=REL_DEPTH, min_views=MIN_VIEWS):
    """The filter of fuse_depth_maps without the point cloud -> (masks bool, consistent-source counts int32, fused depths fp32),
    each [N, 1, h, w].  The fused depth of a pixel is (d + the sum of its reprojected depths) / (1 + count)."""
    mask, count, fused, _, _ = _check(depth, conf, K, R, T, sources, normal, conf_min, reproj_px, rel_depth, min_views)
    return mask.bool(), count, fused


def fuse_depth_maps(depth, conf, colours, K, R, T, sources, *, normal="sweep", conf_min=CONF_MIN, reproj_px=REPROJ_PX,
                    rel_depth=REL_DEPTH, min_views=MIN_VIEWS):
    """Filter N depth maps of one scene by photometric and multi-view geometric consistency and fuse the survivors into one point
    cloud -> (xyz fp32 [M, 3], rgb fp32 [M, 3], masks bool [N, 1, h, w]).

    depth, conf [N, 1, h, w] and colours [N, 3, h, w] on a CUDA device; K, R, T per view ([N, 3, 3], [N, 3, 3], [N, 3, 1], K at
    depth resolution); sources: per view the ids of its source views (at most 16; -1 or shorter lists pad).  A pixel is kept when
    conf >= conf_min, its depth d is finite and > 0, and at least min_views sources are consistent: the point projects into the
    source in front of it and inside [0, w-1] x [0, h-1], the four bilinear taps of the source's depth there are finite and > 0,
    and the source point projected back lands within reproj_px pixels of the pixel with a depth within rel_depth * d of d.  The
    point is the fused depth unprojected at the reference pixel, its colour the colours of that pixel.  Points come view-major,
    row-major; two calls on the same inputs return the same bits."""
    mask, count, fused, blocks, cams = _check(depth, conf, K, R, T, sources, normal, conf_min, reproj_px, rel_depth, min_views)
    xyz, rgb = _emit(mask, fused, blocks, cams, colours)
    return xyz, rgb, mask.bool()


def _view_order(order, N):
    if order is None:
        return list(range(N))
    if isinstance(order, torch.Tensor):
        order = order.detach().cpu().numpy()
    a = np.asarray(order)
    if a.ndim != 1 or a.dtype.kind not in "iu" or not np.array_equal(np.sort(a), np.arange(N)):
        _fail(f"visibility_fusion: order must be a permutation of range({N}), got {a.tolist()}")
    return [int(i) for i in a]


def visibility_fusion(depth, conf, colours, K, R, T, sources, *, order=None, normal="sweep", conf_min=CONF_MIN, reproj_px=REPROJ_PX,
                      rel_depth=REL_DEPTH, min_views=MIN_VIEWS):
    """fuse_depth_maps with visibility-based suppression: each surface point is emitted once, by the first view in `order` that
    keeps it, instead of once per view that sees it -> (xyz fp32 [M, 3], rgb fp32 [M, 3], masks bool [N, 1, h, w]).

    Inputs, thresholds and conventions are those of fuse_depth_maps; order is a permutation of range(N) (default: index order).
    A state used [N, h, w] starts all false, and the views are checked one after another in `order`.  In reference view r a pixel
    with used[r] set is not a reference (its mask is false: another view's point has absorbed it); every other pixel runs
    fuse_depth_maps' test unchanged, and when it is kept, each consistent source j gets the pixel nearest the point's projection
    there marked, used[j, floor(v + 1/2), floor(u + 1/2)] = true.  A marked pixel still serves as a source's depth sample for later
    references; it only stops being a reference itself.  The points are fuse_depth_maps' points of the kept pixels, in its order
    (view-major in index order, not in `order`; row-major).  So the masks are a subset of fuse_depth_maps' masks, where a pixel is
    kept its fused depth is the same bits, and the first view in `order` keeps exactly what fuse_depth_maps keeps there.

    This is fusibile-style (greedy suppression in view order), not fusibile: fusibile's disparity threshold and normal test are not
    applied, and no number of fusibile's is claimed.  Refused with MvsB200Error: a view that lists itself among its sources, an
    order that is not a permutation of range(N), and whatever fuse_depth_maps refuses.  One check launch per view in `order`, then
    one compaction; the one device-to-host read is the point count.  Two calls on the same inputs return the same bits."""
    if not isinstance(depth, torch.Tensor) or depth.dim() != 4:
        _fail(f"depth maps [N, 1, h, w] expected, got {type(depth).__name__} {tuple(getattr(depth, 'shape', ()))}")
    N = depth.shape[0]
    own = np.nonzero((source_table(sources, N) == np.arange(N)[:, None]).any(1))[0]
    if own.size:
        _fail(f"visibility_fusion: view {int(own[0])} lists itself among its sources (it would mark the pixels it is reading)")
    views = _view_order(order, N)
    d, c, cams, src, mask, count, fused, blocks = _prepare(depth, conf, K, R, T, sources, normal)
    _, _, h, w = depth.shape
    used = torch.zeros((N, h, w), dtype=torch.uint8, device=depth.device)
    for r in views:
        with _timed("fusion_visibility"):
            _lib.call("mvsb200_fusion_visibility", d.data_ptr(), c.data_ptr(), cams.data_ptr(), src.data_ptr(), N, src.shape[1], h, w,
                      float(conf_min), float(reproj_px), float(rel_depth), int(min_views), r, used.data_ptr(), mask.data_ptr(),
                      count.data_ptr(), fused.data_ptr(), blocks.data_ptr(), _stream())
    xyz, rgb = _emit(mask, fused, blocks, cams, colours)
    return xyz, rgb, mask.bool()


def resize_colours(images, h, w):
    """images fp32 [N, 3, H, W] on a CUDA device -> [N, 3, h, w]: bilinear, align_corners=False (the resize of refine_input)."""
    if not images.is_cuda:
        _fail("images must be a CUDA tensor; mvs_b200 has no CPU path")
    if images.dim() != 4 or images.shape[1] != 3:
        _fail(f"images [N, 3, H, W] expected, got {tuple(images.shape)}")
    x = images.detach().float().contiguous()
    N, _, H, W = x.shape
    out = torch.empty((N, 3, h, w), dtype=torch.float32, device=x.device)
    _lib.call("mvsb200_resize_rgb", x.data_ptr(), N, H, W, h, w, out.data_ptr(), _stream())
    return out


@torch.no_grad()
def infer_scene(frozen, images, K, R, T, d_min, d_int, pairs, n_views=3, batch_size=4, depth="refined"):
    """Run a FrozenMVSNet once per reference view of a scene -> (depth [N, 1, h, w], conf [N, 1, h, w], colours [N, 3, h, w]).

    images [N, 3, H, W] fp32; K (at feature resolution, H/4 x W/4), R, T per view; d_min, d_int one value per view; pairs[i] the
    source views of view i, best first (dtu.read_pairs): view i runs with its first n_views - 1 sources, gathered in b * V + v
    order.  depth: "refined" or "initial"; conf is the photometric confidence of the initial depth map.  The colours are the
    views' images resized to h x w (bilinear, align_corners=False, as refine_input does).

    Only views with equal (d_min, d_int) share a batch of up to batch_size.  The sweep reads its depth table with the reference's
    batch quirk (flat view i takes the row i mod B, geometry.py), which is then inert: every row of a batch is the same."""
    if depth not in ("refined", "initial"):
        _fail(f'depth must be "refined" or "initial", got {depth!r}')
    dev = frozen.device
    imgs = images.to(dev, torch.float32)
    N = imgs.shape[0]
    K, R, T = _f64(K, (N, 3, 3), "K"), _f64(R, (N, 3, 3), "R"), _f64(T, (N, 3, 1), "T")
    dmin, dint = _f64(d_min, (N,), "d_min"), _f64(d_int, (N,), "d_int")
    V = int(n_views)
    if len(pairs) != N:
        _fail(f"one source list per view expected ({N}), got {len(pairs)}")
    views = []
    for i in range(N):
        src = [int(j) for j in np.asarray(pairs[i]).reshape(-1)[:V - 1]]
        if len(src) != V - 1 or not all(0 <= j < N for j in src):
            _fail(f"view {i} needs {V - 1} source views in [0, {N - 1}], pairs gives {np.asarray(pairs[i]).tolist()}")
        views.append([i] + src)
    groups = {}
    for i in range(N):
        groups.setdefault((dmin[i], dint[i]), []).append(i)
    out_d = out_c = None
    for (d0, di), refs in groups.items():
        for b0 in range(0, len(refs), int(batch_size)):
            chunk = refs[b0:b0 + int(batch_size)]
            B = len(chunk)
            idx = [j for i in chunk for j in views[i]]
            dm = torch.full((B, 1, 1, 1), d0, dtype=torch.float32)
            dt = torch.full((B, 1, 1, 1), di, dtype=torch.float32)
            initial, refined, conf = frozen(imgs[idx], torch.from_numpy(K[idx]).float(), torch.from_numpy(R[idx]).float(),
                                            torch.from_numpy(T[idx]).float(), dm, dt, B, V, return_confidence=True)
            if out_d is None:
                out_d = torch.empty((N,) + tuple(initial.shape[1:]), dtype=torch.float32, device=dev)
                out_c = torch.empty_like(out_d)
            out_d[chunk] = refined if depth == "refined" else initial
            out_c[chunk] = conf
    return out_d, out_c, resize_colours(imgs, out_d.shape[2], out_d.shape[3])


def point_viewpoints(masks, R, T):
    """The centre C = -R^T T of the view that emitted each point of a fuse_depth_maps / visibility_fusion cloud -> fp64 [M, 3] on
    the device of masks.  Both emit view-major in index order, so view i's centre repeats once per kept pixel of masks[i]; these
    are the viewpoints estimate_normals takes to make each normal face the camera that saw its point.  masks [N, 1, h, w] (as returned), R [N, 3, 3], T [N, 3, 1]."""
    if not isinstance(masks, torch.Tensor) or masks.dim() != 4 or masks.shape[1] != 1:
        _fail(f"point_viewpoints: masks [N, 1, h, w] expected, got {tuple(getattr(masks, 'shape', ()))}")
    N = masks.shape[0]
    R, T = _f64(R, (N, 3, 3), "R"), _f64(T, (N, 3, 1), "T")
    C = torch.from_numpy((-np.transpose(R, (0, 2, 1)) @ T).reshape(N, 3)).to(masks.device)
    counts = masks.reshape(N, -1).bool().sum(1)
    return torch.repeat_interleave(C, counts, dim=0)


def write_ply(path, xyz, rgb=None, normals=None):
    """Binary little-endian PLY of the points xyz [M, 3] (float x, y, z), when given their normals [M, 3] (float nx, ny, nz, after z
    as Open3D writes them) and their colours rgb [M, 3] in [0, 1] (uchar red, green, blue: x 255, rounded, clamped)."""
    pts = (xyz.detach().cpu().numpy() if isinstance(xyz, torch.Tensor) else np.asarray(xyz)).astype("<f4").reshape(-1, 3)
    fields = [("x", "<f4"), ("y", "<f4"), ("z", "<f4")]
    if normals is not None:
        nrm = (normals.detach().cpu().numpy() if isinstance(normals, torch.Tensor) else np.asarray(normals)).astype("<f4").reshape(-1, 3)
        if nrm.shape[0] != pts.shape[0]:
            _fail(f"write_ply: {pts.shape[0]} points but {nrm.shape[0]} normals")
        fields += [("nx", "<f4"), ("ny", "<f4"), ("nz", "<f4")]
    if rgb is not None:
        col = (rgb.detach().cpu().numpy() if isinstance(rgb, torch.Tensor) else np.asarray(rgb)).astype(np.float64).reshape(-1, 3)
        if col.shape[0] != pts.shape[0]:
            _fail(f"write_ply: {pts.shape[0]} points but {col.shape[0]} colours")
        fields += [("red", "u1"), ("green", "u1"), ("blue", "u1")]
    rec = np.empty(pts.shape[0], dtype=fields)
    rec["x"], rec["y"], rec["z"] = pts[:, 0], pts[:, 1], pts[:, 2]
    if normals is not None:
        rec["nx"], rec["ny"], rec["nz"] = nrm[:, 0], nrm[:, 1], nrm[:, 2]
    if rgb is not None:
        c8 = np.clip(np.rint(col * 255.0), 0, 255).astype(np.uint8)
        rec["red"], rec["green"], rec["blue"] = c8[:, 0], c8[:, 1], c8[:, 2]
    props = "".join(f"property float {n}\n" for n in "xyz")
    if normals is not None:
        props += "".join(f"property float {n}\n" for n in ("nx", "ny", "nz"))
    if rgb is not None:
        props += "".join(f"property uchar {n}\n" for n in ("red", "green", "blue"))
    header = f"ply\nformat binary_little_endian 1.0\nelement vertex {pts.shape[0]}\n{props}end_header\n"
    with open(path, "wb") as f:
        f.write(header.encode("ascii"))
        f.write(rec.tobytes())


_PLY_TYPES = {"char": "i1", "int8": "i1", "uchar": "u1", "uint8": "u1", "short": "i2", "int16": "i2", "ushort": "u2", "uint16": "u2",
              "int": "i4", "int32": "i4", "uint": "u4", "uint32": "u4", "float": "f4", "float32": "f4", "double": "f8", "float64": "f8"}


def read_ply(path):
    """The vertex element of a PLY file (binary little-endian or ASCII) -> (xyz fp32 [n, 3], rgb uint8 [n, 3] or None), CPU tensors.
    Scalar properties of any PLY type are read; x, y, z become fp32 and red, green, blue uint8 (as stored by write_ply, whose output
    reads back bit for bit); other scalar properties are skipped.  Refused with MvsB200Error: big-endian files, list properties in
    the vertex element (or in an element before it), and a missing x, y or z."""
    with open(path, "rb") as f:
        raw = f.read()
    end = raw.find(b"end_header")
    if not raw.startswith(b"ply") or end < 0:
        _fail(f"read_ply: {path} is not a PLY file")
    body_at = raw.index(b"\n", end) + 1
    fmt, elements = None, []
    for line in raw[:end].decode("ascii", errors="replace").splitlines()[1:]:
        tok = line.split()
        if not tok or tok[0] in ("comment", "obj_info"):
            continue
        if tok[0] == "format":
            fmt = tok[1]
        elif tok[0] == "element":
            elements.append((tok[1], int(tok[2]), []))
        elif tok[0] == "property":
            if not elements:
                _fail(f"read_ply: {path}: property before any element")
            if tok[1] == "list":
                elements[-1][2].append((tok[-1], None))
            elif tok[1] in _PLY_TYPES:
                elements[-1][2].append((tok[2], _PLY_TYPES[tok[1]]))
            else:
                _fail(f"read_ply: {path}: unknown property type {tok[1]!r}")
    if fmt == "binary_big_endian":
        _fail(f"read_ply: {path}: big-endian PLY files are not supported")
    if fmt not in ("binary_little_endian", "ascii"):
        _fail(f"read_ply: {path}: unknown format {fmt!r}")
    names = [e[0] for e in elements]
    if "vertex" not in names:
        _fail(f"read_ply: {path} has no vertex element")
    vi = names.index("vertex")
    for name, count, props in elements[:vi + 1]:
        if any(t is None for _, t in props):
            _fail(f"read_ply: {path}: list property in the element {name!r} (only scalar properties can be read)")
    _, n, props = elements[vi]
    pnames = [p for p, _ in props]
    for c in "xyz":
        if c not in pnames:
            _fail(f"read_ply: {path}: the vertex element has no property {c!r}")
    if fmt == "ascii":
        lines = raw[body_at:].decode("ascii").splitlines()
        skip = sum(c for _, c, _ in elements[:vi])
        rows = [l.split() for l in lines[skip:skip + n]]
        if len(rows) != n or any(len(r) != len(props) for r in rows):
            _fail(f"read_ply: {path}: {n} vertex lines of {len(props)} values expected")
        cols = {p: np.array([r[k] for r in rows], dtype=np.float64 if t[0] == "f" else np.int64).astype(t)
                for k, (p, t) in enumerate(props)}
    else:
        at = body_at + sum(c * sum(np.dtype("<" + t).itemsize for _, t in pr) for _, c, pr in elements[:vi])
        rec = np.frombuffer(raw, dtype=[(p, "<" + t) for p, t in props], count=n, offset=at)
        cols = {p: rec[p] for p in pnames}
    xyz = torch.from_numpy(np.stack([cols[c] for c in "xyz"], 1).astype(np.float32))
    rgb = None
    if all(c in cols for c in ("red", "green", "blue")):
        rgb = torch.from_numpy(np.stack([cols[c] for c in ("red", "green", "blue")], 1).astype(np.uint8))
    return xyz, rgb
