"""Host-side operators of the plane-sweep path: thin autograd wrappers over the C ABI (include/mvs_b200.h).

PyTorch is used for device memory, streams and autograd bookkeeping only; every computation below is a
kernel of libmvs_b200.so.  All ops raise on CPU tensors -- there is no fallback.
"""
from __future__ import annotations

import torch

from . import _lib
from . import geometry

_DT = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16}


def _stream():
    return torch.cuda.current_stream().cuda_stream


# bench.py sets EVENTS = {} to have every kernel launch bracketed by CUDA events on its launching stream
EVENTS = None


class _timed:
    def __init__(self, name, work=None):
        self.name, self.work = name, work          # work: algorithmic FLOPs (tensor kernels) or bytes of this launch

    def __enter__(self):
        if EVENTS is not None:
            self.start = torch.cuda.Event(enable_timing=True)
            self.start.record()

    def __exit__(self, *exc):
        if EVENTS is not None:
            end = torch.cuda.Event(enable_timing=True)
            end.record()
            EVENTS.setdefault(self.name, []).append((self.start, end, self.work))
        return False


# --------------------------------------------------------------------------------------------------
# weight gradients off the critical path of the backward pass
# --------------------------------------------------------------------------------------------------
# A weight gradient reads the layer's saved input and its output gradient, and nothing later in the backward pass reads it.
# Inside loss.backward() the convolution nodes therefore launch it on a side stream and return None for the weight; the
# tensor-core weight-gradient kernels then run under the streaming BatchNorm / data-gradient kernels that follow on the
# launching stream.  One end-of-backward callback joins the side stream and adds every such gradient into its parameter's
# .grad, as AccumulateGrad would (allocated in the parameter's layout, or added in place -- a FlatGradAllReduce view stays one),
# so .grad is complete on the current stream when backward() returns.  torch.autograd.grad, backward(inputs=...) without the
# weight, and double backward keep the plain path: the node returns the gradient.
WGRAD_FORK = True
_SIDE = {}
_PENDING = {}


def _side_stream(device):
    """One side stream per device.  0 is the lowest priority CUDA offers (the default and torch's streams sit there too)."""
    st = _SIDE.get(device)
    if st is None:
        st = _SIDE[device] = torch.cuda.Stream(device, priority=0)
    return st


def _will_accumulate(p):
    """p (a leaf) receives its gradient through AccumulateGrad in the running backward pass."""
    try:
        return p.is_leaf and p.requires_grad and torch._C._will_engine_execute_node(torch.autograd.graph.get_gradient_edge(p).node)
    except RuntimeError:                     # torch.autograd.grad: the engine captures leaf gradients instead of accumulating them
        return False


def _wgrad_targets(w):
    """[(leaf parameter, map from w's gradient to the parameter's)] when every parameter behind w accumulates in this pass."""
    if not WGRAD_FORK or torch.is_grad_enabled() or not w.is_cuda:
        return None
    targets = [(w, None)] if w.is_leaf else getattr(w, "_mvs_wgrad_to", None)
    if not targets or not all(_will_accumulate(p) for p, _ in targets):
        return None
    return targets


class wgrad_fork:
    """`with wgrad_fork(w, reads) as f: f.result = <weight gradient of w>` inside a backward node; then return f.grad() for w.
    Forked, the body launches on the side stream, after all work the launching stream has issued so far; `reads` (the tensors
    the body reads) stay allocated until the side stream is done with them."""

    def __init__(self, w, reads):
        self.targets, self.reads, self.result = _wgrad_targets(w), reads, None

    def __enter__(self):
        if self.targets is not None:
            cur = torch.cuda.current_stream()
            self.side = _side_stream(cur.device)
            self.side.wait_stream(cur)
            for t in self.reads:
                t.record_stream(self.side)
            self._guard = torch.cuda.stream(self.side)
            self._guard.__enter__()
        return self

    def __exit__(self, *exc):
        if self.targets is not None:
            self._guard.__exit__(*exc)
            if exc[0] is None:
                task = torch._C._current_graph_task_id()
                if task not in _PENDING:
                    _PENDING[task] = []
                    torch.autograd.Variable._execution_engine.queue_callback(lambda: _join(task))
                _PENDING[task].append((self.side, self.result, self.targets))
        return False

    def grad(self):
        return self.result if self.targets is None else None


def _join(task):
    """End of the backward pass: the current stream waits for the side stream(s), then every forked gradient goes into .grad."""
    pending = _PENDING.pop(task)
    cur = {}
    with torch.no_grad():
        for side, g, targets in pending:
            st = cur.get(side)
            if st is None:
                st = cur[side] = torch.cuda.current_stream(side.device)
                st.wait_stream(side)
            g.record_stream(st)
            for p, to_param in targets:
                gp = g if to_param is None else to_param(g)
                if p.grad is None:
                    p.grad = torch.empty_like(p).copy_(gp)
                else:
                    p.grad.add_(gp)


def _need_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise _lib.MvsB200Error(f"{what} must live on a CUDA device (got {t.device}); mvs_b200 has no CPU path")


def _ptr(t):
    return None if t is None else t.data_ptr()


# --------------------------------------------------------------------------------------------------
# feature-map layout
# --------------------------------------------------------------------------------------------------
def _features_nhwc(feat: torch.Tensor) -> torch.Tensor:
    """[N,C,h,w] fp32 (any strides) -> tensor whose memory is N x h x w x C.  Zero-copy when the encoder
    already emits channels_last."""
    N, C, h, w = feat.shape
    if feat.dtype != torch.float32:
        feat = feat.float()
    if feat.permute(0, 2, 3, 1).is_contiguous():
        return feat.permute(0, 2, 3, 1)
    src = feat.contiguous()
    dst = torch.empty((N, h, w, C), dtype=torch.float32, device=feat.device)
    _lib.call("mvsb200_nchw_to_nhwc_f32", src.data_ptr(), dst.data_ptr(), N, C, h, w, _stream())
    return dst


def _grad_nchw(g_nhwc: torch.Tensor) -> torch.Tensor:
    N, h, w, C = g_nhwc.shape
    out = torch.empty((N, C, h, w), dtype=torch.float32, device=g_nhwc.device)
    _lib.call("mvsb200_nhwc_to_nchw_f32", g_nhwc.data_ptr(), out.data_ptr(), N, C, h, w, _stream())
    return out


# --------------------------------------------------------------------------------------------------
# K1 / K2
# --------------------------------------------------------------------------------------------------
class _WarpVariance(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, view_params, tinv, B, V, D, out_dtype):
        _need_cuda(feat, "feature_maps")
        N, C, h, w = feat.shape
        if N != B * V:
            raise ValueError(f"feature_maps has {N} views, expected batch_size*n_views = {B * V}")
        nhwc = _features_nhwc(feat.detach())
        cost = torch.empty((B, C, D, h, w), dtype=out_dtype, device=feat.device, memory_format=torch.channels_last_3d)
        with _timed("warp_variance_fwd"):
            _lib.call("mvsb200_warp_variance_fwd", nhwc.data_ptr(), view_params.data_ptr(), tinv.data_ptr(),
                      cost.data_ptr(), _DT[out_dtype], B, V, C, D, h, w, _stream())
        ctx.save_for_backward(nhwc, view_params, tinv)
        ctx.dims = (B, V, C, D, h, w)
        ctx.feat_was_nhwc = feat.permute(0, 2, 3, 1).is_contiguous()
        return cost

    @staticmethod
    def backward(ctx, gcost):
        nhwc, view_params, tinv = ctx.saved_tensors
        B, V, C, D, h, w = ctx.dims
        if gcost.dtype not in _DT:
            gcost = gcost.float()
        gcost = gcost.contiguous(memory_format=torch.channels_last_3d)
        g_nhwc = torch.empty((B * V, h, w, C), dtype=torch.float32, device=gcost.device)
        with _timed("warp_variance_bwd"):
            _lib.call("mvsb200_warp_variance_bwd", nhwc.data_ptr(), view_params.data_ptr(), tinv.data_ptr(),
                      gcost.data_ptr(), _DT[gcost.dtype], g_nhwc.data_ptr(), B, V, C, D, h, w, _stream())
        gfeat = g_nhwc.permute(0, 3, 1, 2) if ctx.feat_was_nhwc else _grad_nchw(g_nhwc)
        return gfeat, None, None, None, None, None, None


class PlaneSweep:
    """Geometry of one homography_warping call, resident on the device: what the fused kernel needs
    instead of the N*D 3x3 matrices the reference builds (homography.py:40-75)."""

    def __init__(self, K, R, T, d_min, d_int, batch_size, n_views, d_num, d_scale, h, w, device,
                 bug_compatible=True):
        self.B, self.V, self.D, self.h, self.w = batch_size, n_views, d_num, h, w
        self.d_scale, self.bug_compatible = d_scale, bug_compatible
        self.d_batch_0 = geometry.depth_table(d_min, d_int, d_num, d_scale)            # CPU [B,D,1,1]
        params, tinv = geometry.view_tables(K, R, T, self.d_batch_0, batch_size, n_views, h, w, bug_compatible)
        packed = torch.from_numpy(params).pin_memory() if torch.cuda.is_available() else torch.from_numpy(params)
        self.view_params = packed.to(device, non_blocking=True)
        self.tinv = torch.from_numpy(tinv).to(device)
        self.d_batch_dev = self.d_batch_0.to(device)
        self._stage = None

    def update(self, K, R, T, d_min, d_int):
        """New cameras / depth range into the SAME device buffers (static addresses: the sweep of a captured CUDA graph is
        re-targeted by this call; one pinned staging buffer, three asynchronous copies on the current stream)."""
        self.d_batch_0 = geometry.depth_table(d_min, d_int, self.D, self.d_scale)
        params, tinv = geometry.view_tables(K, R, T, self.d_batch_0, self.B, self.V, self.h, self.w, self.bug_compatible)
        n1, n2, n3 = params.size, tinv.size, self.d_batch_0.numel()
        on_gpu = self.view_params.is_cuda
        if self._stage is None:
            self._stage = torch.empty(n1 + n2 + n3, dtype=torch.float32)
            if on_gpu:
                self._stage = self._stage.pin_memory()
                self._stage_free = torch.cuda.Event()
        elif on_gpu:
            self._stage_free.synchronize()                 # the previous update's copies have left the staging buffer
        st = self._stage
        st[:n1].copy_(torch.from_numpy(params).reshape(-1))
        st[n1:n1 + n2].copy_(torch.from_numpy(tinv).reshape(-1))
        st[n1 + n2:].copy_(self.d_batch_0.reshape(-1))
        self.view_params.view(-1).copy_(st[:n1], non_blocking=True)
        self.tinv.view(-1).copy_(st[n1:n1 + n2], non_blocking=True)
        self.d_batch_dev.view(-1).copy_(st[n1 + n2:], non_blocking=True)
        if on_gpu:
            self._stage_free.record()
        return self


def warp_variance(feat: torch.Tensor, sweep: PlaneSweep, out_dtype=torch.float32) -> torch.Tensor:
    """features [B*V,32,h,w] -> variance cost volume [B,32,D,h,w] (channels_last_3d strides)."""
    return _WarpVariance.apply(feat, sweep.view_params, sweep.tinv, sweep.B, sweep.V, sweep.D, out_dtype)


def warp_materialize(feat: torch.Tensor, sweep: PlaneSweep) -> torch.Tensor:
    """Parity/debug: the [B*V,C,D,h,w] warped volumes the reference's homography_warping returns."""
    _need_cuda(feat, "feature_maps")
    N, C, h, w = feat.shape
    nhwc = _features_nhwc(feat.detach())
    out = torch.empty((N, C, sweep.D, h, w), dtype=torch.float32, device=feat.device)
    _lib.call("mvsb200_warp_materialize", nhwc.data_ptr(), sweep.view_params.data_ptr(), sweep.tinv.data_ptr(),
              out.data_ptr(), sweep.B, sweep.V, C, sweep.D, h, w, _stream())
    return out


class _VarianceViews(torch.autograd.Function):
    @staticmethod
    def forward(ctx, warped, n_views):
        _need_cuda(warped, "warped_feature_maps")
        bn, c, d, h, w = warped.shape
        x = warped.detach().float().contiguous()
        B, M = bn // n_views, c * d * h * w
        out = torch.empty((B, c, d, h, w), dtype=torch.float32, device=warped.device)
        _lib.call("mvsb200_variance_views_fwd", x.data_ptr(), out.data_ptr(), B, n_views, M, _stream())
        ctx.save_for_backward(x)
        ctx.n_views = n_views
        return out

    @staticmethod
    def backward(ctx, gout):
        (x,) = ctx.saved_tensors
        V = ctx.n_views
        B, M = x.shape[0] // V, x[0].numel()
        gx = torch.empty_like(x)
        g = gout.float().contiguous()
        _lib.call("mvsb200_variance_views_bwd", x.data_ptr(), g.data_ptr(), gx.data_ptr(), B, V, M, _stream())
        return gx, None


def variance_views(warped: torch.Tensor, n_views: int) -> torch.Tensor:
    return _VarianceViews.apply(warped, n_views)


# --------------------------------------------------------------------------------------------------
# K4
# --------------------------------------------------------------------------------------------------
def _as_bdhw(t: torch.Tensor):
    B, one, D, h, w = t.shape
    if one != 1:
        raise ValueError(f"expected a [B,1,D,h,w] volume, got {tuple(t.shape)}")
    return t.reshape(B, D, h, w).contiguous(), (B, D, h, w)


class _SoftmaxRanks(torch.autograd.Function):
    """prob = softmax_D(logits); also produces the kept-plane ranks (non-differentiable side output)."""

    @staticmethod
    def forward(ctx, logits, n_est):
        _need_cuda(logits, "logits")
        x, (B, D, h, w) = _as_bdhw(logits.detach().float())
        prob = torch.empty_like(x)
        n_keep = min(n_est, D)
        ranks = torch.empty((B, n_keep, h, w), dtype=torch.int32, device=x.device)
        with _timed("softmax_ranks_fwd"):
            _lib.call("mvsb200_softmax_depth_fwd", x.data_ptr(), 1, None, prob.data_ptr(), ranks.data_ptr(), None,
                      B, D, h, w, n_est, _stream())
        ctx.save_for_backward(prob)
        ctx.dims = (B, D, h, w)
        ctx.mark_non_differentiable(ranks)
        ctx.set_materialize_grads(False)          # no zero tensors (one fill launch each) for outputs nobody differentiates
        return prob.view(B, 1, D, h, w), ranks

    @staticmethod
    def backward(ctx, gprob, _granks):
        if gprob is None:
            return None, None
        (prob,) = ctx.saved_tensors
        B, D, h, w = ctx.dims
        g = gprob.float().reshape(B, D, h, w).contiguous()
        out = torch.empty_like(prob)
        _lib.call("mvsb200_softmax_bwd", prob.data_ptr(), g.data_ptr(), out.data_ptr(), B, D, h, w, _stream())
        return out.view(B, 1, D, h, w), None


class _DepthFromProb(torch.autograd.Function):
    """depth = sum_kept d P / sum_kept P.  `ranks` may be None (computed here from the probabilities)."""

    @staticmethod
    def forward(ctx, prob, depths, ranks, n_est):
        _need_cuda(prob, "prob_volume")
        p, (B, D, h, w) = _as_bdhw(prob.detach().float())
        depths = depths.detach().to(device=p.device, dtype=torch.float32).reshape(B, D).contiguous()
        depth = torch.empty((B, h, w), dtype=torch.float32, device=p.device)
        n_keep = min(n_est, D)
        if ranks is None:
            ranks = torch.empty((B, n_keep, h, w), dtype=torch.int32, device=p.device)
            _lib.call("mvsb200_softmax_depth_fwd", p.data_ptr(), 0, depths.data_ptr(), None, ranks.data_ptr(),
                      depth.data_ptr(), B, D, h, w, n_est, _stream())
        else:
            _lib.call("mvsb200_depth_from_ranks", p.data_ptr(), ranks.data_ptr(), depths.data_ptr(), depth.data_ptr(),
                      B, D, h, w, n_keep, _stream())
        ctx.save_for_backward(p, ranks, depths)
        ctx.dims = (B, D, h, w, n_keep)
        return depth.view(B, 1, h, w)

    @staticmethod
    def backward(ctx, gdepth):
        p, ranks, depths = ctx.saved_tensors
        B, D, h, w, n_keep = ctx.dims
        g = gdepth.float().reshape(B, h, w).contiguous()
        gprob = torch.empty_like(p)
        _lib.call("mvsb200_depth_bwd", p.data_ptr(), ranks.data_ptr(), depths.data_ptr(), g.data_ptr(),
                  gprob.data_ptr(), B, D, h, w, n_keep, _stream())
        return gprob.view(B, 1, D, h, w), None, None, None


def softmax_over_depth(logits: torch.Tensor, n_est: int = 5) -> torch.Tensor:
    """CostVolumeReg.Norm replacement.  The returned prob tensor carries the kept-plane ranks so that
    extract_depth_map needs no second pass over the volume."""
    prob, ranks = _SoftmaxRanks.apply(logits, int(n_est))
    prob._mvs_ranks = (ranks, int(n_est), prob._version)
    return prob


def depth_from_prob(prob: torch.Tensor, d_batch: torch.Tensor, n_est: int = 5) -> torch.Tensor:
    """extract_depth_map replacement: prob [B,1,D,h,w], d_batch [B,D,1,1] -> [B,1,h,w]."""
    stash = getattr(prob, "_mvs_ranks", None)
    ranks = None
    if stash is not None and stash[1] == int(n_est) and stash[2] == prob._version:
        ranks = stash[0]
    return _DepthFromProb.apply(prob, d_batch, ranks, int(n_est))


def softmax_depth(logits: torch.Tensor, d_batch: torch.Tensor, n_est: int = 5):
    """Fully fused forward (one launch): logits -> (prob, depth).  Inference helper; no autograd."""
    _need_cuda(logits, "logits")
    x, (B, D, h, w) = _as_bdhw(logits.detach().float())
    depths = d_batch.detach().to(device=x.device, dtype=torch.float32).reshape(B, D).contiguous()
    prob = torch.empty_like(x)
    depth = torch.empty((B, h, w), dtype=torch.float32, device=x.device)
    _lib.call("mvsb200_softmax_depth_fwd", x.data_ptr(), 1, depths.data_ptr(), prob.data_ptr(), None, depth.data_ptr(),
              B, D, h, w, int(n_est), _stream())
    return prob.view(B, 1, D, h, w), depth.view(B, 1, h, w)


def softmax_depth_confidence(logits: torch.Tensor, d_batch: torch.Tensor, n_est: int = 5):
    """Fused forward (one launch): logits [B,1,D,h,w] -> (prob, ranks, depth, conf).  prob, ranks and depth are bit-identical to
    softmax_over_depth + depth_from_prob; conf [B,1,h,w] is the confidence of depth_confidence.  Inference only; no autograd."""
    _need_cuda(logits, "logits")
    x, (B, D, h, w) = _as_bdhw(logits.detach().float())
    depths = d_batch.detach().to(device=x.device, dtype=torch.float32).reshape(B, D).contiguous()
    prob = torch.empty_like(x)
    ranks = torch.empty((B, min(int(n_est), D), h, w), dtype=torch.int32, device=x.device)
    depth = torch.empty((B, h, w), dtype=torch.float32, device=x.device)
    conf = torch.empty_like(depth)
    with _timed("softmax_depth_conf_fwd"):
        _lib.call("mvsb200_softmax_depth_conf_fwd", x.data_ptr(), 1, depths.data_ptr(), prob.data_ptr(), ranks.data_ptr(),
                  depth.data_ptr(), conf.data_ptr(), B, D, h, w, int(n_est), _stream())
    return prob.view(B, 1, D, h, w), ranks, depth.view(B, 1, h, w), conf.view(B, 1, h, w)


def depth_confidence(prob: torch.Tensor, depth: torch.Tensor, d_batch: torch.Tensor) -> torch.Tensor:
    """MVSNet's photometric confidence of an existing probability volume prob [B,1,D,h,w] and depth map [B,1,h,w]: the
    probability mass of the planes k0-1 .. k0+2 (clipped to the sweep) with k0 = floor((depth - d_0) / (d_1 - d_0)), summed in
    ascending order in fp32 -> [B,1,h,w].  1 when D = 1; NaN where the depth or a summed probability is not finite.  No autograd."""
    _need_cuda(prob, "prob_volume")
    p, (B, D, h, w) = _as_bdhw(prob.detach().float())
    if depth.shape != (B, 1, h, w):
        raise _lib.MvsB200Error(f"depth_confidence: depth map [{B}, 1, {h}, {w}] expected, got {tuple(depth.shape)}")
    dep = depth.detach().to(device=p.device, dtype=torch.float32).contiguous()
    depths = d_batch.detach().to(device=p.device, dtype=torch.float32).reshape(B, D).contiguous()
    conf = torch.empty((B, 1, h, w), dtype=torch.float32, device=p.device)
    with _timed("depth_confidence"):
        _lib.call("mvsb200_depth_confidence", p.data_ptr(), dep.data_ptr(), depths.data_ptr(), conf.data_ptr(), B, D, h, w, _stream())
    return conf


# --------------------------------------------------------------------------------------------------
# K3b: train-mode BatchNorm3d + ReLU on channel-last volumes
# --------------------------------------------------------------------------------------------------
_BN_WS = {}


def _ws_key(device):
    """Scratch buffers are per (device, launching stream): kernels of one stream are ordered, two streams (or a replaying graph
    captured on its own stream and eager launches) never share scratch memory."""
    return (device, torch.cuda.current_stream(device).cuda_stream)


def _bn_workspace(device):
    key = _ws_key(device)
    ws = _BN_WS.get(key)
    if ws is None:
        ws = torch.empty(int(_lib.load().mvsb200_bn_workspace_floats()), dtype=torch.float32, device=device)
        _BN_WS[key] = ws
    return ws


def _rows(x: torch.Tensor):
    """[B,C,D,h,w] volume -> (tensor whose memory is M x C rows, M, C)."""
    if x.dtype not in _DT:
        x = x.float()
    x = x.contiguous(memory_format=torch.channels_last_3d)
    B, C, D, h, w = x.shape
    return x, B * D * h * w, C


def _geo12(alloc, canvas, crop):
    import ctypes
    (d0, d1), (h0, h1), (w0, w1) = crop
    return (ctypes.c_int * 12)(*alloc, *canvas, d0, h0, w0, d1 - d0, h1 - h0, w1 - w0)


class _BatchNormReLU(torch.autograd.Function):
    """y = ReLU(BatchNorm_train(x)) with batch statistics (model.py:101-121).  Returns (y, mean, biased var).
    `canvas` = (D,h,w): the statistics volume, sitting at the origin of x's (possibly larger) allocation.
    `crop` = ((d0,d1),(h0,h1),(w0,w1)): y (and the incoming gradient) exist only on that box of the canvas."""

    @staticmethod
    def forward(ctx, x, weight, bias, eps, relu, crop, canvas, running=None, momentum=0.1, partials=None, add=None, s2d=False):
        _need_cuda(x, "BatchNorm input")
        _need_cuda(weight, "BatchNorm weight")
        xr, _, C = _rows(x.detach())
        dev = xr.device
        B = xr.shape[0]
        alloc = tuple(xr.shape[2:])
        canvas = alloc if canvas is None else tuple(canvas)
        plain = crop is None and canvas == alloc
        M = B * canvas[0] * canvas[1] * canvas[2]
        box = crop if crop is not None else tuple((0, n) for n in canvas)
        geo = None if plain else _geo12(alloc, canvas, box)
        # one [5, C] buffer: mean, biased variance, invstd, scale, shift -- all written by the statistics' finalize launch,
        # which also performs the running-statistics update of torch.nn.BatchNorm when `running` is given
        vec = torch.empty((5, C), dtype=torch.float32, device=dev)
        mean, var, invstd, scale, shift = vec[0], vec[1], vec[2], vec[3], vec[4]
        gamma = weight.detach().float().contiguous()
        beta = bias.detach().float().contiguous()
        rm = rv = nbt = None
        if running is not None:
            rm, rv, nbt = running
            if not (rm.is_cuda and rm.dtype == torch.float32 and rm.is_contiguous() and rv.dtype == torch.float32 and rv.is_contiguous()
                    and (nbt is None or (nbt.is_cuda and nbt.dtype == torch.int64))):
                raise _lib.MvsB200Error("BatchNorm running statistics must be contiguous fp32 CUDA tensors (int64 counter)")
        ws = _bn_workspace(dev)
        if partials is not None and tuple(partials[2]) == canvas and partials[0].shape[-1] == C:
            # the producer kernel (transposed convolution) already summed what it stored: finalize only, no pass over the canvas
            with _timed("bn_stats"):
                _lib.call("mvsb200_bn_finalize_affine", partials[0].data_ptr(), int(partials[1]), M, C, gamma.data_ptr(), beta.data_ptr(),
                          float(eps), float(momentum), _ptr(rm), _ptr(rv), _ptr(nbt), mean.data_ptr(), var.data_ptr(), invstd.data_ptr(),
                          scale.data_ptr(), shift.data_ptr(), _stream())
        else:
            with _timed("bn_stats"):
                _lib.call("mvsb200_bn_stats_affine", xr.data_ptr(), _DT[xr.dtype], M, C, ws.data_ptr(), geo if canvas != alloc else None,
                          gamma.data_ptr(), beta.data_ptr(), float(eps), float(momentum), _ptr(rm), _ptr(rv), _ptr(nbt),
                          mean.data_ptr(), var.data_ptr(), invstd.data_ptr(), scale.data_ptr(), shift.data_ptr(), _stream())
        (d0, d1), (h0, h1), (w0, w1) = box
        y = torch.empty_like(xr) if plain else torch.empty((B, C, d1 - d0, h1 - h0, w1 - w0), dtype=xr.dtype, device=dev,
                                                           memory_format=torch.channels_last_3d)
        ctx.s2d = None
        if s2d:
            # stacked maps [1, C, N, H, W] -> the normalised maps in the space-to-depth form [1, 4C, N, H/2, W/2] (nets2d.py: the
            # input of a 5x5 stride-2 layer), written by the apply pass itself; the backward reads its gradient from that form
            if not plain or add is not None or xr.shape[0] != 1 or xr.dtype != torch.bfloat16 or alloc[1] % 2 or alloc[2] % 2:
                raise _lib.MvsB200Error(f"BatchNorm with space-to-depth output: dense stacked bf16 maps of even size expected, got "
                                        f"{tuple(xr.shape)} {xr.dtype}")
            Nm, H, W = alloc
            y = torch.empty((1, 4 * C, Nm, H // 2, W // 2), dtype=xr.dtype, device=dev, memory_format=torch.channels_last_3d)
            with _timed("bn_relu_fwd"):
                _lib.call("mvsb200_bn_relu_fwd_s2d", xr.data_ptr(), _DT[xr.dtype], scale.data_ptr(), shift.data_ptr(), y.data_ptr(),
                          int(relu), M, C, H, W, _stream())
            ctx.s2d = (H, W)
        elif add is not None:
            # skip addition folded into the apply pass (model.py:117-123): the addend lives where y does
            if add.shape != y.shape or add.dtype != y.dtype:
                raise _lib.MvsB200Error(f"BatchNorm + skip addition: addend {tuple(add.shape)} {add.dtype} for an output "
                                        f"{tuple(y.shape)} {y.dtype}")
            ad = add.detach().contiguous(memory_format=torch.channels_last_3d)
            with _timed("bn_relu_fwd"):
                _lib.call("mvsb200_bn_relu_add_apply", xr.data_ptr(), _DT[xr.dtype], scale.data_ptr(), shift.data_ptr(), ad.data_ptr(),
                          y.data_ptr(), int(relu), M, C, None if plain else geo, _stream())
        elif plain:
            with _timed("bn_relu_fwd"):
                _lib.call("mvsb200_bn_relu_fwd", xr.data_ptr(), _DT[xr.dtype], scale.data_ptr(), shift.data_ptr(),
                          y.data_ptr(), int(relu), M, C, _stream())
        else:
            with _timed("bn_relu_fwd"):
                _lib.call("mvsb200_bn_relu_fwd_crop", xr.data_ptr(), _DT[xr.dtype], scale.data_ptr(), shift.data_ptr(),
                          y.data_ptr(), int(relu), M, C, geo, _stream())
        ctx.has_add = add is not None
        ctx.save_for_backward(xr, scale, shift, mean, invstd, gamma)
        ctx.relu, ctx.dims, ctx.geo = bool(relu), (M, C), (None if plain else (alloc, canvas, box))
        ctx.mark_non_differentiable(mean, var)
        ctx.set_materialize_grads(False)          # no zero tensors (one fill launch each) for outputs nobody differentiates
        return y, mean, var

    @staticmethod
    def backward(ctx, gy, _gm, _gv):
        if gy is None:
            return (None,) * 12
        xr, scale, shift, mean, invstd, gamma = ctx.saved_tensors
        M, C = ctx.dims
        if gy.dtype not in _DT:
            gy = gy.float()
        gy = gy.contiguous(memory_format=torch.channels_last_3d)
        dev = xr.device
        dbeta = torch.empty(C, dtype=torch.float32, device=dev)
        dgamma = torch.empty(C, dtype=torch.float32, device=dev)
        dx = torch.empty_like(xr)
        with _timed("bn_relu_bwd"):
            if ctx.s2d is not None:
                gy = gy.to(torch.bfloat16).contiguous(memory_format=torch.channels_last_3d)
                _lib.call("mvsb200_bn_relu_bwd_s2d", xr.data_ptr(), gy.data_ptr(), scale.data_ptr(), shift.data_ptr(), mean.data_ptr(),
                          invstd.data_ptr(), gamma.data_ptr(), _bn_workspace(dev).data_ptr(), dbeta.data_ptr(), dgamma.data_ptr(),
                          dx.data_ptr(), int(ctx.relu), M, C, ctx.s2d[0], ctx.s2d[1], _stream())
            elif ctx.geo is None:
                _lib.call("mvsb200_bn_relu_bwd", xr.data_ptr(), _DT[xr.dtype], gy.data_ptr(), _DT[gy.dtype],
                          scale.data_ptr(), shift.data_ptr(), mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                          _bn_workspace(dev).data_ptr(), dbeta.data_ptr(), dgamma.data_ptr(), dx.data_ptr(),
                          int(ctx.relu), M, C, _stream())
            else:
                _lib.call("mvsb200_bn_relu_bwd_crop", xr.data_ptr(), _DT[xr.dtype], gy.data_ptr(), _DT[gy.dtype],
                          scale.data_ptr(), shift.data_ptr(), mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                          _bn_workspace(dev).data_ptr(), dbeta.data_ptr(), dgamma.data_ptr(), dx.data_ptr(),
                          int(ctx.relu), M, C, _geo12(*ctx.geo), _stream())
        # the skip addend's gradient is the incoming gradient itself
        return dx, dgamma, dbeta, None, None, None, None, None, None, None, (gy if ctx.has_add else None), None


def batchnorm_relu_train(x, weight, bias, eps=1e-5, relu=True, crop=None, canvas=None, running=None, momentum=0.1, partials=None, add=None,
                         s2d=False):
    """-> (y, batch mean [C], biased batch variance [C]); y has x's dtype (fp32 or bf16), channels_last_3d.
    canvas = (D,h,w) <= x's spatial dims: the statistics volume (x may carry allocation slack beyond it);
    crop = ((d0,d1),(h0,h1),(w0,w1)): full-canvas statistics, y only on that box.
    running = (running_mean, running_var, num_batches_tracked): updated in place as torch.nn.BatchNorm does in train mode
    (momentum, unbiased variance), inside the statistics' finalize launch.
    partials = (per-CTA sums [n, 2, C], n, (D,h,w)) left by the kernel that produced x (conv3d_sm100.conv_transpose3d_s2): the
    statistics are finalized from them, x is not read for them.
    add = a tensor of y's shape and dtype: y = ReLU(BatchNorm(x)) + add in the same pass (the decoder's skip additions), bit-identical
    to adding it to the stored y afterwards; its gradient is y's.
    s2d: x is a stack of maps [1, C, N, H, W]; y leaves in the space-to-depth form [1, 4C, N, H/2, W/2] (nets2d.space_to_depth of
    the normalised maps, written by the apply pass itself)."""
    if crop is not None:
        crop = tuple((int(a), int(b)) for a, b in crop)
    if canvas is not None:
        canvas = tuple(int(n) for n in canvas)
    return _BatchNormReLU.apply(x, weight, bias, float(eps), bool(relu), crop, canvas, running, float(momentum), partials, add, bool(s2d))


def affine_relu(x, scale, shift, relu=True):
    """Eval-mode BatchNorm(+ReLU): y = max(x*scale + shift, 0) with given per-channel fp32 vectors (no autograd)."""
    _need_cuda(x, "BatchNorm input")
    xr, M, C = _rows(x.detach())
    y = torch.empty_like(xr)
    _lib.call("mvsb200_bn_relu_fwd", xr.data_ptr(), _DT[xr.dtype], scale.float().contiguous().data_ptr(),
              shift.float().contiguous().data_ptr(), y.data_ptr(), int(relu), M, C, _stream())
    return y


# --------------------------------------------------------------------------------------------------
# K3c: the output convolution 8 -> 1 (model.py:91,123)
# --------------------------------------------------------------------------------------------------
_CO_WS = {}


def _conv_out_workspace(device):
    key = _ws_key(device)
    ws = _CO_WS.get(key)
    if ws is None:
        ws = torch.empty(int(_lib.load().mvsb200_conv_out_workspace_floats()), dtype=torch.float32, device=device)
        _CO_WS[key] = ws
    return ws


class _ConvOut(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z, weight):
        _need_cuda(z, "conv_out input")
        _need_cuda(weight, "conv_out weight")
        B, C, D, h, w = z.shape
        zc = z.detach().to(torch.bfloat16).contiguous(memory_format=torch.channels_last_3d)
        w27 = weight.detach().float()[0].permute(1, 2, 3, 0).reshape(27, 8).contiguous()
        out = torch.empty((B, 1, D, h, w), dtype=torch.float32, device=z.device)
        with _timed("conv_out_fwd"):
            _lib.call("mvsb200_conv_out_fwd", zc.data_ptr(), w27.data_ptr(), out.data_ptr(), B, D, h, w, _stream())
        ctx.save_for_backward(zc, w27)
        ctx.wdtype, ctx.zdtype, ctx.w_arg = weight.dtype, z.dtype, weight
        return out

    @staticmethod
    def backward(ctx, gout):
        zc, w27 = ctx.saved_tensors
        B, _, D, h, w = zc.shape
        g = gout.float().contiguous()
        gz = gw = None
        if ctx.needs_input_grad[0]:
            gz = torch.empty_like(zc)
            with _timed("conv_out_dgrad"):
                _lib.call("mvsb200_conv_out_dgrad", g.data_ptr(), w27.data_ptr(), gz.data_ptr(), B, D, h, w, _stream())
            gz = gz.to(ctx.zdtype)
        if ctx.needs_input_grad[1]:
            with wgrad_fork(ctx.w_arg, (zc, g)) as f:
                gw27 = torch.empty_like(w27)
                with _timed("conv_out_wgrad"):
                    _lib.call("mvsb200_conv_out_wgrad", zc.data_ptr(), g.data_ptr(), _conv_out_workspace(zc.device).data_ptr(),
                              gw27.data_ptr(), B, D, h, w, _stream())
                f.result = gw27.reshape(3, 3, 3, 8).permute(3, 0, 1, 2).unsqueeze(0).to(ctx.wdtype)
            gw = f.grad()
        return gz, gw


def conv_out(z: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
    """Conv3d(8, 1, 3, padding=1, bias=False) on a [B,8,D,h,w] volume -> fp32 logits [B,1,D,h,w]."""
    if z.shape[1] != 8 or tuple(weight.shape) != (1, 8, 3, 3, 3):
        raise ValueError(f"conv_out expects 8 -> 1 channels, got input {tuple(z.shape)} and weight {tuple(weight.shape)}")
    return _ConvOut.apply(z, weight)


# --------------------------------------------------------------------------------------------------
# K3d: per-channel sums and affine+ReLU over boxes (the stride-2 branches' BatchNorm on their central box)
# --------------------------------------------------------------------------------------------------
_AF_WS = {}


def _affine_workspace(device):
    key = _ws_key(device)
    ws = _AF_WS.get(key)
    if ws is None:
        ws = torch.empty(int(_lib.load().mvsb200_affine_workspace_floats()), dtype=torch.float32, device=device)
        _AF_WS[key] = ws
    return ws


def _box_view(x: torch.Tensor):
    """A [B,C,D,h,w] view with unit channel stride (made so if needed) -> (tensor, strides4, dims4 ctypes arrays)."""
    import ctypes
    if x.dtype not in _DT:
        x = x.float()
    if x.stride(1) != 1 or any(s % 8 for s in (x.stride(0), x.stride(2), x.stride(3), x.stride(4))) or x.data_ptr() % 16:
        x = x.contiguous(memory_format=torch.channels_last_3d)
    B, C, D, h, w = x.shape
    strides = (ctypes.c_int64 * 4)(x.stride(0), x.stride(2), x.stride(3), x.stride(4))
    dims = (ctypes.c_int * 4)(B, D, h, w)
    return x, strides, dims


class _ChannelSums(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        _need_cuda(x, "channel_sums input")
        xv, strides, dims = _box_view(x.detach())
        C = xv.shape[1]
        s1 = torch.empty(C, dtype=torch.float32, device=xv.device)
        s2 = torch.empty(C, dtype=torch.float32, device=xv.device)
        with _timed("channel_sums"):
            _lib.call("mvsb200_channel_sums", xv.data_ptr(), _DT[xv.dtype], strides, dims, C,
                      _affine_workspace(xv.device).data_ptr(), s1.data_ptr(), s2.data_ptr(), _stream())
        ctx.save_for_backward(xv)
        return s1, s2

    @staticmethod
    def backward(ctx, g1, g2):
        (xv,) = ctx.saved_tensors
        _, strides, dims = _box_view(xv)
        gx = torch.empty(xv.shape, dtype=xv.dtype, device=xv.device, memory_format=torch.channels_last_3d)
        with _timed("channel_sums_bwd"):
            _lib.call("mvsb200_channel_sums_bwd", xv.data_ptr(), _DT[xv.dtype], strides, dims, xv.shape[1],
                      g1.float().contiguous().data_ptr(), g2.float().contiguous().data_ptr(), gx.data_ptr(), _stream())
        return gx


def channel_sums(x: torch.Tensor):
    """(sum x, sum x^2) per channel over a [B,C,D,h,w] box (any view with unit channel stride); differentiable."""
    return _ChannelSums.apply(x)


def _geo13(xv, in_origin, out_origin, out_dims):
    import ctypes
    B, _, D, h, w = xv.shape
    return (ctypes.c_int * 13)(B, D, h, w, *in_origin, *out_origin, *out_dims)


class _AffineReLUGeo(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, scale, shift, in_origin, out_origin, out_dims, relu):
        _need_cuda(x, "affine_relu_geo input")
        xv, strides, _ = _box_view(x.detach())
        B, C = xv.shape[:2]
        sc, sh = scale.detach().float().contiguous(), shift.detach().float().contiguous()
        y = torch.empty((B, C) + tuple(out_dims), dtype=xv.dtype, device=xv.device, memory_format=torch.channels_last_3d)
        with _timed("affine_relu_geo_fwd"):
            _lib.call("mvsb200_affine_relu_geo_fwd", xv.data_ptr(), _DT[xv.dtype], strides, _geo13(xv, in_origin, out_origin, out_dims),
                      C, sc.data_ptr(), sh.data_ptr(), y.data_ptr(), int(relu), _stream())
        ctx.save_for_backward(xv, sc, sh)
        ctx.geo, ctx.relu = (tuple(in_origin), tuple(out_origin), tuple(out_dims)), bool(relu)
        return y

    @staticmethod
    def backward(ctx, gy):
        xv, sc, sh = ctx.saved_tensors
        _, strides, _ = _box_view(xv)
        C = xv.shape[1]
        if gy.dtype not in _DT:
            gy = gy.float()
        gy = gy.contiguous(memory_format=torch.channels_last_3d)
        gx = torch.empty(xv.shape, dtype=xv.dtype, device=xv.device, memory_format=torch.channels_last_3d)
        gscale = torch.empty(C, dtype=torch.float32, device=xv.device)
        gshift = torch.empty(C, dtype=torch.float32, device=xv.device)
        with _timed("affine_relu_geo_bwd"):
            _lib.call("mvsb200_affine_relu_geo_bwd", xv.data_ptr(), _DT[xv.dtype], strides, _geo13(xv, *ctx.geo), C,
                      sc.data_ptr(), sh.data_ptr(), gy.data_ptr(), _DT[gy.dtype], _affine_workspace(xv.device).data_ptr(),
                      gscale.data_ptr(), gshift.data_ptr(), gx.data_ptr(), int(ctx.relu), _stream())
        return gx, gscale, gshift, None, None, None, None


def affine_relu_geo(x, scale, shift, in_origin, out_origin, out_dims, relu=True):
    """y(p) = max(xv(p)*scale + shift, 0) on the output box; xv = x inside the input box, 0 outside (one frame).
    Differentiable w.r.t. x, scale and shift."""
    return _AffineReLUGeo.apply(x, scale, shift, tuple(int(v) for v in in_origin), tuple(int(v) for v in out_origin),
                                tuple(int(v) for v in out_dims), bool(relu))


# --------------------------------------------------------------------------------------------------
# K3d, fused: train-mode BatchNorm3d + ReLU of a stride-2 branch on its central box (model.py:104-110)
# --------------------------------------------------------------------------------------------------
class BoxGradDest:
    """Where the gradients of the stacked stride-2 branch outputs are wanted: the padded, channel-stacked, channel-last buffer
    the strided convolution's backward reads (conv3d_sm100._Conv3dS2Box).  The fused box BatchNorm backward writes its result
    straight into the branch's slice of that buffer (allocated, zeroed once, on first use), so the three strided copies and
    the zero-fill of an assembled buffer disappear."""

    def __init__(self, shape, box, splits, device, zero=True):
        self.shape, self.box, self.splits, self.device = tuple(shape), tuple(box), tuple(splits), device
        self.buffer = None
        self.zero = zero                 # False: the box is the whole buffer, every element gets written
        self.filled = [False] * len(splits)

    def dest(self, k):
        if self.buffer is None:
            self.buffer = torch.empty(self.shape, dtype=torch.bfloat16, device=self.device, memory_format=torch.channels_last_3d)
            if self.zero:
                self.buffer.zero_()
        c0 = sum(self.splits[:k])
        return self.buffer[(slice(None), slice(c0, c0 + self.splits[k])) + self.box]

    def holds(self, k, g):
        """g is exactly this holder's slice k (written by the fused backward)."""
        if self.buffer is None or not self.filled[k] or g is None:
            return False
        d = self.dest(k)
        return g.data_ptr() == d.data_ptr() and g.shape == d.shape and g.stride() == d.stride() and g.dtype == d.dtype


class _BoxBatchNormReLU(torch.autograd.Function):
    """X, scale, shift = BatchNorm_train+ReLU of the box tensor S whose canvas (n_full voxels per channel) is zero outside the
    box: mean = sum S / n_full, var = sum S^2 / n_full - mean^2 (the zeros count), X on the output box (data where the input box
    is, relu(shift) around it).  scale / shift are differentiable outputs too (the next layer's analytic statistics use
    relu(shift)).  Backward: ONE reduction pass (gscale, gshift), the per-channel algebra, ONE apply pass
    gS = g*scale + dL/d(sum S) + 2 S dL/d(sum S^2) -- written into `grad_dest` when given."""

    @staticmethod
    def forward(ctx, S, weight, bias, n_full, eps, in_origin, out_origin, out_dims, grad_dest, running=None, momentum=0.1, sums_in=None):
        _need_cuda(S, "box BatchNorm input")
        _need_cuda(weight, "BatchNorm weight")
        xv, strides, dims = _box_view(S.detach())
        C = xv.shape[1]
        dev = xv.device
        if sums_in is not None and sums_in[0].shape == (C,) and sums_in[0].dtype == torch.float32 and sums_in[0].is_contiguous() \
                and sums_in[1].is_contiguous():
            sums = sums_in                          # left by the producing convolution's epilogue: no pass over S
        else:
            sums = torch.empty((2, C), dtype=torch.float32, device=dev)
            with _timed("channel_sums"):
                _lib.call("mvsb200_channel_sums", xv.data_ptr(), _DT[xv.dtype], strides, dims, C, _affine_workspace(dev).data_ptr(),
                          sums[0].data_ptr(), sums[1].data_ptr(), _stream())
        # the per-channel algebra (fp64 inside) and the running-statistics update in one launch
        vec = torch.empty((4, C), dtype=torch.float32, device=dev)
        scale, shift, mean, var = vec[0], vec[1], vec[2], vec[3]
        stat64 = torch.empty((2, C), dtype=torch.float64, device=dev)       # mean, 1/sqrt(var + eps): the backward's operands
        gamma = weight.detach().float().contiguous()
        beta = bias.detach().float().contiguous()
        rm = rv = nbt = None
        if running is not None:
            rm, rv, nbt = running
        _lib.call("mvsb200_box_bn_algebra_fwd", sums[0].data_ptr(), sums[1].data_ptr(), None, None, C, float(n_full), gamma.data_ptr(),
                  beta.data_ptr(), float(eps), float(momentum), _ptr(rm), _ptr(rv), _ptr(nbt), scale.data_ptr(), shift.data_ptr(),
                  mean.data_ptr(), var.data_ptr(), stat64.data_ptr(), _stream())
        B = xv.shape[0]
        y = torch.empty((B, C) + tuple(out_dims), dtype=xv.dtype, device=dev, memory_format=torch.channels_last_3d)
        with _timed("affine_relu_geo_fwd"):
            _lib.call("mvsb200_affine_relu_geo_fwd", xv.data_ptr(), _DT[xv.dtype], strides, _geo13(xv, in_origin, out_origin, out_dims),
                      C, scale.data_ptr(), shift.data_ptr(), y.data_ptr(), 1, _stream())
        ctx.save_for_backward(xv, scale, shift, stat64, gamma)
        ctx.geo, ctx.n_full, ctx.grad_dest = (tuple(in_origin), tuple(out_origin), tuple(out_dims)), float(n_full), grad_dest
        ctx.mark_non_differentiable(mean, var)
        ctx.set_materialize_grads(False)          # no zero tensors (one fill launch each) for outputs nobody differentiates
        return y, scale, shift, mean, var

    @staticmethod
    def backward(ctx, gy, g_scale_ext, g_shift_ext, _gm, _gv):
        xv, scale, shift, stat64, gamma = ctx.saved_tensors
        _, strides, _ = _box_view(xv)
        C, dev, n = xv.shape[1], xv.device, ctx.n_full
        if gy is None:
            gy = torch.empty((xv.shape[0], C) + ctx.geo[2], dtype=xv.dtype, device=dev, memory_format=torch.channels_last_3d).zero_()
        if gy.dtype not in _DT:
            gy = gy.float()
        gy = gy.contiguous(memory_format=torch.channels_last_3d)
        red = torch.empty((2, C), dtype=torch.float32, device=dev)          # gscale, gshift over the box
        geo = _geo13(xv, *ctx.geo)
        with _timed("box_bn_relu_bwd"):
            _lib.call("mvsb200_box_bn_relu_bwd_reduce", xv.data_ptr(), _DT[xv.dtype], strides, geo, C, scale.data_ptr(), shift.data_ptr(),
                      gy.data_ptr(), _DT[gy.dtype], _affine_workspace(dev).data_ptr(), red[0].data_ptr(), red[1].data_ptr(), 1, _stream())
        # per-channel algebra (fp64 inside, one launch): (a, b2) = (dL/d sum S, 2 dL/d sum S^2), gradients of gamma and beta
        ext = [None if g is None else g.detach().float().contiguous() for g in (g_scale_ext, g_shift_ext)]
        out = torch.empty((4, C), dtype=torch.float32, device=dev)
        a, b2, g_gamma, g_beta = out[0], out[1], out[2], out[3]
        _lib.call("mvsb200_box_bn_algebra_bwd", red[0].data_ptr(), red[1].data_ptr(), _ptr(ext[0]), _ptr(ext[1]), stat64.data_ptr(),
                  gamma.data_ptr(), C, float(n), a.data_ptr(), b2.data_ptr(), g_gamma.data_ptr(), g_beta.data_ptr(), _stream())
        dest = ctx.grad_dest
        if dest is not None and xv.dtype == torch.bfloat16:
            holder, k = dest
            gx = holder.dest(k)
            holder.filled[k] = True
        else:
            gx = torch.empty(xv.shape, dtype=xv.dtype, device=dev, memory_format=torch.channels_last_3d)
        import ctypes
        ostr = (ctypes.c_int64 * 4)(gx.stride(0), gx.stride(2), gx.stride(3), gx.stride(4))
        with _timed("box_bn_relu_bwd"):
            _lib.call("mvsb200_box_bn_relu_bwd_apply", xv.data_ptr(), _DT[xv.dtype], strides, geo, C, scale.data_ptr(), shift.data_ptr(),
                      a.data_ptr(), b2.data_ptr(), gy.data_ptr(), _DT[gy.dtype], gx.data_ptr(), ostr, 1, _stream())
        return gx, g_gamma, g_beta, None, None, None, None, None, None, None, None, None


def box_batchnorm_relu(S, weight, bias, n_full, eps, in_origin, out_origin, out_dims, grad_dest=None, running=None, momentum=0.1,
                       sums=None):
    """-> (X on the output box, scale [C], shift [C], batch mean [C], biased batch variance [C]) -- see _BoxBatchNormReLU.
    running = (running_mean, running_var, num_batches_tracked): updated in place as torch.nn.BatchNorm does in train mode.
    sums = (sum S [C], sum S^2 [C]) fp32 when the kernel that produced S already has them (conv3d_sm100: the stride-2
    convolution's epilogue): the statistics pass over S is skipped."""
    return _BoxBatchNormReLU.apply(S, weight, bias, float(n_full), float(eps), tuple(int(v) for v in in_origin),
                                   tuple(int(v) for v in out_origin), tuple(int(v) for v in out_dims), grad_dest, running, float(momentum),
                                   sums)


class _OutsideSums(torch.autograd.Function):
    """(A1, A2) fp64 [Cout]: what a stride-1, padding-1 convolution with weight W [Cout, Cin, 3, 3, 3] contributes to its BatchNorm
    sums OUTSIDE its computed box, where its input is the per-channel constant bg [Cin]: 27 border classes of cnt [3, 3, 3] voxels
    each (regulariser._outside_geometry).  One launch forward, two backward (mvsb200_outside_sums_*) where a five-operand einsum
    and its fp64 follow-up stood."""

    @staticmethod
    def forward(ctx, W, bg, cnt):
        _need_cuda(W, "convolution weight")
        Wf = W.detach().float().contiguous()
        bgf = bg.detach().float().contiguous()
        cf = cnt.detach().float().contiguous()
        Cout, Cin = Wf.shape[:2]
        if Wf.shape[2:] != (3, 3, 3) or bgf.numel() != Cin or cf.numel() != 27:
            raise _lib.MvsB200Error(f"outside_sums: W {tuple(Wf.shape)}, bg {tuple(bgf.shape)}, cnt {tuple(cf.shape)}")
        out = torch.empty((2, Cout), dtype=torch.float64, device=Wf.device)
        val = torch.empty((Cout, 27), dtype=torch.float64, device=Wf.device)
        _lib.call("mvsb200_outside_sums_fwd", Wf.data_ptr(), bgf.data_ptr(), cf.data_ptr(), Cout, Cin, val.data_ptr(), out[0].data_ptr(),
                  out[1].data_ptr(), _stream())
        ctx.save_for_backward(Wf, bgf, cf, val)
        ctx.meta = (W.dtype, bg.dtype, bg.shape)
        ctx.set_materialize_grads(False)
        return out[0], out[1]

    @staticmethod
    def backward(ctx, gA1, gA2):
        if gA1 is None and gA2 is None:
            return None, None, None
        Wf, bgf, cf, val = ctx.saved_tensors
        Cout, Cin = Wf.shape[:2]
        g1 = None if gA1 is None else gA1.detach().double().contiguous()
        g2 = None if gA2 is None else gA2.detach().double().contiguous()
        gW = torch.empty_like(Wf)
        gbg = torch.empty(Cin, dtype=torch.float32, device=Wf.device)
        dt = torch.empty((Cout, 27), dtype=torch.float32, device=Wf.device)
        _lib.call("mvsb200_outside_sums_bwd", Wf.data_ptr(), bgf.data_ptr(), cf.data_ptr(), val.data_ptr(), _ptr(g1), _ptr(g2), Cout, Cin,
                  dt.data_ptr(), gW.data_ptr(), gbg.data_ptr(), _stream())
        wd, bd, bshape = ctx.meta
        return gW.to(wd), gbg.to(bd).reshape(bshape), None


def outside_sums(W, bg, cnt):
    """-> (A1, A2) fp64 [Cout], see _OutsideSums."""
    return _OutsideSums.apply(W, bg, cnt)


class _BoxStatsAffine(torch.autograd.Function):
    """(scale, shift) of a train-mode BatchNorm from the per-channel sums (t1, t2) of a tensor over a box plus the closed-form
    sums (A1, A2, fp64) of what it holds outside the box: mean = (t1 + A1)/n, var = (t2 + A2)/n - mean^2, scale = gamma/sqrt(var +
    eps), shift = beta - mean scale, running statistics updated in place -- one launch forward, one backward
    (mvsb200_box_bn_algebra_fwd / _bwd) where ~25 + ~40 [C]-sized torch launches stood (conv_{1,2,3}_1, regulariser.py)."""

    @staticmethod
    def forward(ctx, t1, t2, A1, A2, weight, bias, n_full, eps, running, momentum):
        C, dev = t1.shape[0], t1.device
        t1, t2 = t1.detach().float().contiguous(), t2.detach().float().contiguous()
        A1, A2 = A1.detach().double().contiguous(), A2.detach().double().contiguous()
        vec = torch.empty((4, C), dtype=torch.float32, device=dev)
        stat64 = torch.empty((2, C), dtype=torch.float64, device=dev)
        gamma, beta = weight.detach().float().contiguous(), bias.detach().float().contiguous()
        rm, rv, nbt = running if running is not None else (None, None, None)
        _lib.call("mvsb200_box_bn_algebra_fwd", t1.data_ptr(), t2.data_ptr(), A1.data_ptr(), A2.data_ptr(), C, float(n_full),
                  gamma.data_ptr(), beta.data_ptr(), float(eps), float(momentum), _ptr(rm), _ptr(rv), _ptr(nbt), vec[0].data_ptr(),
                  vec[1].data_ptr(), vec[2].data_ptr(), vec[3].data_ptr(), stat64.data_ptr(), _stream())
        ctx.save_for_backward(stat64, gamma)
        ctx.n_full = float(n_full)
        return vec[0], vec[1]

    @staticmethod
    def backward(ctx, g_scale, g_shift):
        stat64, gamma = ctx.saved_tensors
        C, dev = gamma.shape[0], gamma.device
        zero = None
        if g_scale is None or g_shift is None:
            zero = torch.zeros(C, dtype=torch.float32, device=dev)
        gs = zero if g_scale is None else g_scale.detach().float().contiguous()
        gh = zero if g_shift is None else g_shift.detach().float().contiguous()
        out = torch.empty((4, C), dtype=torch.float32, device=dev)
        _lib.call("mvsb200_box_bn_algebra_bwd", gs.data_ptr(), gh.data_ptr(), None, None, stat64.data_ptr(), gamma.data_ptr(), C,
                  ctx.n_full, out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(), out[3].data_ptr(), _stream())
        g1, g2 = out[0], out[1] * 0.5                      # dL/d(sum), dL/d(sum of squares): the same for t and A
        return g1, g2, g1.double(), g2.double(), out[2], out[3], None, None, None, None


def box_stats_affine(t1, t2, A1, A2, weight, bias, n_full, eps, running=None, momentum=0.1):
    """-> (scale [C], shift [C]) -- see _BoxStatsAffine."""
    return _BoxStatsAffine.apply(t1, t2, A1, A2, weight, bias, float(n_full), float(eps), running, float(momentum))


class _BoxLink:
    """Connects the two autograd nodes of a box BatchNorm whose statistics go through differentiable per-channel algebra outside
    (conv_k_1: its statistics also depend on the filter and on the constant around the box): the affine node's backward only
    REDUCES (gscale, gshift) and leaves (gy, scale, shift, geometry) here; the statistics node's backward -- which autograd
    runs afterwards, its incoming gradients depend on gscale / gshift -- then makes the ONE apply pass
    gT = gy*mask*scale + g1 + 2 T g2 instead of an affine data gradient, a statistics gradient and their sum."""

    def __init__(self):
        self.pending = None          # (gy, scale, shift, geo, relu) left by the affine backward
        self.sums_done = False


class _BoxSumsLinked(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, link):
        _need_cuda(x, "channel_sums input")
        xv, strides, dims = _box_view(x.detach())
        C = xv.shape[1]
        s1 = torch.empty(C, dtype=torch.float32, device=xv.device)
        s2 = torch.empty(C, dtype=torch.float32, device=xv.device)
        with _timed("channel_sums"):
            _lib.call("mvsb200_channel_sums", xv.data_ptr(), _DT[xv.dtype], strides, dims, C,
                      _affine_workspace(xv.device).data_ptr(), s1.data_ptr(), s2.data_ptr(), _stream())
        ctx.save_for_backward(xv)
        ctx.link = link
        return s1, s2

    @staticmethod
    def backward(ctx, g1, g2):
        (xv,) = ctx.saved_tensors
        _, strides, dims = _box_view(xv)
        C, dev = xv.shape[1], xv.device
        link = ctx.link
        g1 = (torch.zeros(C, device=dev) if g1 is None else g1.float()).contiguous()
        g2 = (torch.zeros(C, device=dev) if g2 is None else g2.float()).contiguous()
        gx = torch.empty(xv.shape, dtype=xv.dtype, device=dev, memory_format=torch.channels_last_3d)
        link.sums_done = True
        if link.pending is None:                     # the affine node had no incoming gradient (or runs later): statistics only
            with _timed("channel_sums_bwd"):
                _lib.call("mvsb200_channel_sums_bwd", xv.data_ptr(), _DT[xv.dtype], strides, dims, C, g1.data_ptr(), g2.data_ptr(),
                          gx.data_ptr(), _stream())
            return gx, None
        gy, sc, sh, geo, relu = link.pending
        link.pending = None
        import ctypes
        ostr = (ctypes.c_int64 * 4)(gx.stride(0), gx.stride(2), gx.stride(3), gx.stride(4))
        b2 = (2.0 * g2).contiguous()
        with _timed("box_bn_relu_bwd"):
            _lib.call("mvsb200_box_bn_relu_bwd_apply", xv.data_ptr(), _DT[xv.dtype], strides, _geo13(xv, *geo), C, sc.data_ptr(),
                      sh.data_ptr(), g1.data_ptr(), b2.data_ptr(), gy.data_ptr(), _DT[gy.dtype], gx.data_ptr(), ostr, int(relu), _stream())
        return gx, None


class _AffineReLUGeoLinked(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, scale, shift, in_origin, out_origin, out_dims, relu, link):
        _need_cuda(x, "affine_relu_geo input")
        xv, strides, _ = _box_view(x.detach())
        B, C = xv.shape[:2]
        sc, sh = scale.detach().float().contiguous(), shift.detach().float().contiguous()
        y = torch.empty((B, C) + tuple(out_dims), dtype=xv.dtype, device=xv.device, memory_format=torch.channels_last_3d)
        with _timed("affine_relu_geo_fwd"):
            _lib.call("mvsb200_affine_relu_geo_fwd", xv.data_ptr(), _DT[xv.dtype], strides, _geo13(xv, in_origin, out_origin, out_dims),
                      C, sc.data_ptr(), sh.data_ptr(), y.data_ptr(), int(relu), _stream())
        ctx.save_for_backward(xv, sc, sh)
        ctx.geo, ctx.relu, ctx.link = (tuple(in_origin), tuple(out_origin), tuple(out_dims)), bool(relu), link
        return y

    @staticmethod
    def backward(ctx, gy):
        xv, sc, sh = ctx.saved_tensors
        _, strides, _ = _box_view(xv)
        C, dev, link = xv.shape[1], xv.device, ctx.link
        if gy.dtype not in _DT:
            gy = gy.float()
        gy = gy.contiguous(memory_format=torch.channels_last_3d)
        gscale = torch.empty(C, dtype=torch.float32, device=dev)
        gshift = torch.empty(C, dtype=torch.float32, device=dev)
        if link.sums_done:                           # the statistics node already ran (no dependency on this one): classic form
            gx = torch.empty(xv.shape, dtype=xv.dtype, device=dev, memory_format=torch.channels_last_3d)
            with _timed("affine_relu_geo_bwd"):
                _lib.call("mvsb200_affine_relu_geo_bwd", xv.data_ptr(), _DT[xv.dtype], strides, _geo13(xv, *ctx.geo), C,
                          sc.data_ptr(), sh.data_ptr(), gy.data_ptr(), _DT[gy.dtype], _affine_workspace(dev).data_ptr(),
                          gscale.data_ptr(), gshift.data_ptr(), gx.data_ptr(), int(ctx.relu), _stream())
            return gx, gscale, gshift, None, None, None, None, None
        with _timed("box_bn_relu_bwd"):
            _lib.call("mvsb200_box_bn_relu_bwd_reduce", xv.data_ptr(), _DT[xv.dtype], strides, _geo13(xv, *ctx.geo), C, sc.data_ptr(),
                      sh.data_ptr(), gy.data_ptr(), _DT[gy.dtype], _affine_workspace(dev).data_ptr(), gscale.data_ptr(),
                      gshift.data_ptr(), int(ctx.relu), _stream())
        link.pending = (gy, sc, sh, ctx.geo, ctx.relu)   # the data gradient is made by the statistics node's backward
        return None, gscale, gshift, None, None, None, None, None


def box_batchnorm_linked(x):
    """-> (link, (sum x, sum x^2)) for a box BatchNorm whose per-channel algebra stays outside; pass `link` to
    affine_relu_geo_linked for the normalisation of the same tensor."""
    link = _BoxLink()
    return link, _BoxSumsLinked.apply(x, link)


def affine_relu_geo_linked(x, scale, shift, in_origin, out_origin, out_dims, link, relu=True):
    return _AffineReLUGeoLinked.apply(x, scale, shift, tuple(int(v) for v in in_origin), tuple(int(v) for v in out_origin),
                                      tuple(int(v) for v in out_dims), bool(relu), link)


# --------------------------------------------------------------------------------------------------
# f3: the training loss (scripts/loss.py:4-41), one launch forward, one backward
# --------------------------------------------------------------------------------------------------
class _MaskedL1Loss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, gt, initial, refined):
        for t, what in ((gt, "ground-truth depth"), (initial, "initial depth map"), (refined, "refined depth map")):
            _need_cuda(t, what)
        if not (gt.shape == initial.shape == refined.shape):
            raise _lib.MvsB200Error(f"loss_fcn: shapes differ: {tuple(gt.shape)}, {tuple(initial.shape)}, {tuple(refined.shape)}")
        g_, a0, a1 = (t.detach().float().contiguous() for t in (gt, initial, refined))
        B = g_.shape[0]
        n = g_.numel() // B
        ws = torch.zeros(int(_lib.load().mvsb200_masked_l1_workspace_floats(B)), dtype=torch.float32, device=g_.device)
        out3 = torch.empty(3, dtype=torch.float32, device=g_.device)
        with _timed("masked_l1_loss"):
            _lib.call("mvsb200_masked_l1_fwd", g_.data_ptr(), a0.data_ptr(), a1.data_ptr(), B, n, ws.data_ptr(), out3.data_ptr(), _stream())
        ctx.save_for_backward(g_, a0, a1, ws)
        ctx.shapes = (initial.shape, refined.shape, initial.dtype, refined.dtype)
        ctx.set_materialize_grads(False)
        return out3[0], out3[1], out3[2]

    @staticmethod
    def backward(ctx, g_loss, g_acc0, g_acc1):
        g_, a0, a1, ws = ctx.saved_tensors
        B = g_.shape[0]
        n = g_.numel() // B
        g3 = torch.zeros(3, dtype=torch.float32, device=g_.device)
        for k, g in enumerate((g_loss, g_acc0, g_acc1)):
            if g is not None:
                g3[k] = g.detach().float().reshape(())
        ga0, ga1 = torch.empty_like(a0), torch.empty_like(a1)
        with _timed("masked_l1_loss"):
            _lib.call("mvsb200_masked_l1_bwd", g_.data_ptr(), a0.data_ptr(), a1.data_ptr(), ws.data_ptr(), g3.data_ptr(), B, n,
                      ga0.data_ptr(), ga1.data_ptr(), _stream())
        s0, s1, d0, d1 = ctx.shapes
        return None, ga0.view(s0).to(d0), ga1.view(s1).to(d1)


def masked_l1_loss(gt, initial, refined):
    """(loss, initial_acc, refined_acc) of scripts/loss.py:4-41 -- masked L1 on both depth maps, mask = (gt != 0), per-sample
    normalisation by the number of valid pixels -- one launch forward and one backward (SURVEY §8 row f3)."""
    return _MaskedL1Loss.apply(gt, initial, refined)
