"""The 2D convolutions either side of the hot path on the path's own tensor-core kernels (SURVEY §8 rows f1 and f2).

Reference: /root/reference/scripts/model.py:22-65 (`FeatureEncoder`: eight Conv2d -- 3x3 stride 1 and two 5x5 stride 2 -- on
3 / 8 / 16 / 32 channels, BatchNorm2d + ReLU after all but the last) and :129-152 (`DepthRefinement`, see refine.py).

Layout: a batch of maps [N, C, H, W] travels as channel-last bf16 rows stacked as the planes of ONE volume, [1, C, N, H, W]
(memory N x H x W x C).  On that volume

  * a 3x3 convolution (padding 1) IS the 3x3x3 convolution whose filter has only its middle depth slice: the filter operand is
    packed straight from the Conv2d parameter (mvsb200_pack_filter, middle slice of the kdn layout), forward and data gradient
    run conv3d_s1_kdn_kernel in its PLANAR mode (mvsb200_conv2d_rows_fwd): MMAs of N = Cout on the middle slice's row block, one
    slab per map, the accumulator is the output plane -- 9 MMAs per 128 pixels and K step, what a native 2D kernel issues
    (MVSB200_CONV2D=volume keeps the three-slice form for A/B) -- and the weight gradient runs conv3d_s1_wgrad_tc_kernel with
    the depth-tap mask 2 (mvsb200_conv3d_s1_wgrad_ex);
  * a 5x5 stride-2 convolution (padding 2) is a 3x3 stride-1 convolution of the space-to-depth form [1, 4C, N, H/2, W/2] of its
    input: tap k = 2t + p of an axis reads parity class p at j - 1 + t, so the effective filter [co, (py, px, c), ty, tx] is a
    zero-padded re-indexing of the [co, c, 5, 5] parameter (25 of its 36 taps are real);
  * BatchNorm2d + ReLU over (N, H, W) is BatchNorm3d + ReLU over the volume: the fused K3b kernels, the module's running
    statistics updated in place.

Maps of different samples are neighbouring planes of the volume and never meet: the planar forward reads one plane per output
plane, the weight gradient computes the middle depth taps only.  Train mode, bf16 operands, fp32 accumulation; eval-mode BatchNorm and fp32 stay on the module's torch layers."""
from __future__ import annotations

import ctypes

import torch
import torch.nn.functional as F

from . import _lib, ops
from .ops import _need_cuda, _stream, _timed

_CL3 = torch.channels_last_3d


def _n_rows(c):
    return 16 if c <= 16 else (32 if c <= 32 else 64)


def _pack2d(w, role, n_rows, n_cols, out=None):
    """Conv2d weight [co, ci, 3, 3] (dense fp32) -> the bf16 [(kh, kw)][kd][row][col] filter operand of the kdn kernel in one
    launch: middle depth slice = the 3x3 filter, the other slices and the padded rows / columns zero.  role "fwd": rows = co,
    columns = ci; "dgrad": taps flipped, rows = ci, columns = co.  out: the buffer to write (the filter is re-packed in place)."""
    from .conv3d_sm100 import _FLIP, _NAT, _kdn_order
    co, ci = w.shape[:2]
    taps = [t - 9 if 9 <= t < 18 else -1 for t in _kdn_order(_NAT if role == "fwd" else _FLIP)]
    rows_real, cols_real, sr, sc = (co, ci, 9 * ci, 9) if role == "fwd" else (ci, co, 9, 9 * ci)
    if out is None:
        out = torch.empty((27, n_rows, n_cols), dtype=torch.bfloat16, device=w.device)
    _lib.call("mvsb200_pack_filter", w.data_ptr(), out.data_ptr(), 27, n_rows, n_cols, rows_real, cols_real, 0, sr, sc,
              (ctypes.c_int * 27)(*taps), _stream())
    return out


def _PLANAR():
    import os
    return os.environ.get("MVSB200_CONV2D", "planar") != "volume"


def _conv_rows(x, wk, c_out, work):
    """3x3 convolution (padding 1) of the stacked maps x [1, c, N, H, W] with a packed filter -> [1, c_out, N, H, W]."""
    _, c, N, H, W = x.shape
    y = torch.empty((1, c_out, N, H, W), dtype=torch.bfloat16, device=x.device, memory_format=_CL3)
    with _timed("conv2d_tc", work):
        if _PLANAR():
            _lib.call("mvsb200_conv2d_rows_fwd", x.data_ptr(), wk.data_ptr(), y.data_ptr(), N, H, W, c, c_out, c_out, _n_rows(c_out),
                      _stream())
        else:       # MVSB200_CONV2D=volume: the maps as one volume under the three-slice filter (zero kd = 0 / 2 slices); A/B form
            _lib.call("mvsb200_conv3d_s1_fwd_kdn", x.data_ptr(), wk.data_ptr(), y.data_ptr(), 1, N, H, W, c, N, H, W, c_out, c_out,
                      _n_rows(c_out), -1, -1, -1, _stream())
    return y


class _Conv2dRows(torch.autograd.Function):
    """Conv2d(ci, co, 3, padding=1, bias=False) on stacked channel-last maps: x [1, cx, N, H, W] bf16 (cx >= ci, surplus
    channels zero), w [co, ci, 3, 3] fp32 -> [1, cy, N, H, W] (cy >= co, surplus channels zero)."""

    @staticmethod
    def forward(ctx, x, w, cy):
        _need_cuda(x, "maps")
        if x.dtype != torch.bfloat16 or w.dtype != torch.float32 or x.shape[0] != 1:
            raise _lib.MvsB200Error(f"2D convolution: stacked bf16 rows [1, C, N, H, W] and an fp32 weight expected, got {x.dtype} "
                                    f"{tuple(x.shape)}, {w.dtype}")
        x = x.detach().contiguous(memory_format=_CL3)
        wf = w.detach().contiguous()
        co, ci = wf.shape[:2]
        _, cx, N, H, W = x.shape
        if ci > cx or co > cy or cx not in (8, 16, 32, 64) or cy not in (8, 16, 32, 64):
            raise _lib.MvsB200Error(f"2D convolution: {ci} -> {co} channels on rows of {cx} -> {cy}")
        y = _conv_rows(x, _pack2d(wf, "fwd", _n_rows(cy), max(cx, 16)), cy, 2.0 * 9 * ci * co * N * H * W)
        ctx.save_for_backward(x, wf)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        co, ci = w.shape[:2]
        _, cx, N, H, W = x.shape
        cy = gy.shape[1]
        gy = gy.to(torch.bfloat16).contiguous(memory_format=_CL3)
        work = 2.0 * 9 * ci * co * N * H * W
        gx = gw = None
        if ctx.needs_input_grad[0]:
            gx = _conv_rows(gy, _pack2d(w, "dgrad", _n_rows(cx), max(cy, 16)), cx, work)
        if ctx.needs_input_grad[1]:
            gw27 = torch.empty((27, max(cx, 16), cy), dtype=torch.float32, device=gy.device)
            with _timed("conv2d_wgrad_tc", work):
                _lib.call("mvsb200_conv3d_s1_wgrad_ex", x.data_ptr(), gy.data_ptr(), gw27.data_ptr(), 1, N, H, W, cx, N, H, W, cy,
                          -1, -1, -1, 2, _stream())
            gw = gw27[9:18, :ci, :co].reshape(3, 3, ci, co).permute(3, 2, 0, 1)      # a view: the accumulation into .grad reads it strided
        return gx, gw, None


def conv3x3(x, w, cy=None):
    """Conv2d 3x3 / padding 1 on stacked rows (see _Conv2dRows); cy defaults to the layer's width rounded up to 8."""
    co = w.shape[0]
    return _Conv2dRows.apply(x, w, int(cy) if cy is not None else max(8, (co + 7) // 8 * 8))


class _SpaceToDepth(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        _, C, N, H, W = x.shape
        if H % 2 or W % 2 or C % 8:
            raise _lib.MvsB200Error(f"space-to-depth: even maps of a multiple of 8 channels expected, got {tuple(x.shape)}")
        x = x.detach().contiguous(memory_format=_CL3)
        y = torch.empty((1, 4 * C, N, H // 2, W // 2), dtype=x.dtype, device=x.device, memory_format=_CL3)
        with _timed("s2d_rows"):
            _lib.call("mvsb200_s2d_rows_bf16", x.data_ptr(), y.data_ptr(), N, H // 2, W // 2, C, 0, _stream())
        return y

    @staticmethod
    def backward(ctx, gy):
        _, C4, N, h, w = gy.shape
        gy = gy.to(torch.bfloat16).contiguous(memory_format=_CL3)
        gx = torch.empty((1, C4 // 4, N, 2 * h, 2 * w), dtype=gy.dtype, device=gy.device, memory_format=_CL3)
        with _timed("s2d_rows"):
            _lib.call("mvsb200_s2d_rows_bf16", gy.data_ptr(), gx.data_ptr(), N, h, w, C4 // 4, 1, _stream())
        return gx


def space_to_depth(x):
    """[1, C, N, 2h, 2w] -> [1, 4C, N, h, w], channel (py*2 + px)*C + c of pixel (j, i) = channel c of pixel (2j + py, 2i + px)."""
    return _SpaceToDepth.apply(x)


def k5s2_as_3x3(w5):
    """Conv2d weight [co, ci, 5, 5] (stride 2, padding 2) -> the [co, 4ci, 3, 3] filter of the same convolution on the
    space-to-depth form of its input (differentiable re-indexing; the 11 taps that fall outside the 5x5 support are zero)."""
    co, ci = w5.shape[:2]
    w6 = F.pad(w5.float(), (0, 1, 0, 1))
    return w6.view(co, ci, 3, 2, 3, 2).permute(0, 3, 5, 1, 2, 4).reshape(co, 4 * ci, 3, 3)


def image_rows(images):
    """fp32 images [N, 3, H, W] (any strides) -> stacked bf16 rows [1, 8, N, H, W], channels 3..7 zero (no gradient)."""
    _need_cuda(images, "input images")
    if images.dtype != torch.float32 or images.dim() != 4 or images.shape[1] != 3:
        raise _lib.MvsB200Error(f"image_rows: fp32 [N, 3, H, W] expected, got {images.dtype} {tuple(images.shape)}")
    N, _, H, W = images.shape
    rows = torch.empty((1, 8, N, H, W), dtype=torch.bfloat16, device=images.device, memory_format=_CL3)
    with _timed("image_rows"):
        _lib.call("mvsb200_image_to_rows8", images.data_ptr(), (ctypes.c_int64 * 4)(*images.stride()), N, H, W, rows.data_ptr(), _stream())
    return rows


def _bn_relu(y, bn, s2d=False):
    """BatchNorm2d + ReLU of the stacked maps on the fused K3b kernels; s2d: the result leaves in the space-to-depth form (the
    input of a 5x5 stride-2 layer), written by the apply pass itself -- MVSB200_S2D=separate keeps the permutation a pass of its own."""
    import os
    fused = s2d and os.environ.get("MVSB200_S2D", "fused") != "separate"
    out, _, _ = ops.batchnorm_relu_train(y, bn.weight, bn.bias, bn.eps, relu=True,
                                         running=(bn.running_mean, bn.running_var, bn.num_batches_tracked), momentum=bn.momentum,
                                         s2d=fused)
    return space_to_depth(out) if s2d and not fused else out


_ENC_LAYERS = ((3, 8, 3, 1), (8, 8, 3, 1), (8, 16, 5, 2), (16, 16, 3, 1), (16, 16, 3, 1), (16, 32, 5, 2), (32, 32, 3, 1), (32, 32, 3, 1))


def encoder_layout_error(module):
    """None when FeatureEncoder `module` has the reference's layout (eight bias-free fp32 Conv2d of _ENC_LAYERS, seven
    BatchNorm2d), else what differs."""
    convs = [m for m in getattr(module, "model", ()) if isinstance(m, torch.nn.Conv2d)]
    bns = [m for m in getattr(module, "model", ()) if isinstance(m, torch.nn.BatchNorm2d)]
    if len(convs) != 8 or len(bns) != 7:
        return f"feature encoder: {len(convs)} Conv2d / {len(bns)} BatchNorm2d layers, the reference has 8 / 7"
    for i, (c, (ci, co, k, s)) in enumerate(zip(convs, _ENC_LAYERS)):
        if (c.in_channels, c.out_channels, c.kernel_size, c.stride, c.padding) != (ci, co, (k, k), (s, s), (k // 2, k // 2)) \
                or c.bias is not None or c.weight.dtype != torch.float32:
            return f"feature encoder: convolution {i} is not the reference's {ci} -> {co}, {k}x{k}, stride {s}, bias-free fp32 layer"
    for i, (b, (_, co, _, _)) in enumerate(zip(bns, _ENC_LAYERS)):
        if b.num_features != co:
            return f"feature encoder: BatchNorm {i} has {b.num_features} channels, the reference {co}"
    return None


def encoder_ok(module, images) -> bool:
    """Whether FeatureEncoder `module` can run on the library's kernels: the reference's eight layers, train-mode BatchNorm, fp32
    images on the GPU whose sides are multiples of 4."""
    from . import conv3d_sm100
    if not (images.is_cuda and images.dtype == torch.float32 and images.dim() == 4 and module.training
            and images.shape[2] % 4 == 0 and images.shape[3] % 4 == 0 and min(images.shape[2:]) >= 12):
        return False
    return encoder_layout_error(module) is None and conv3d_sm100.available()


def encode_native(module, images):
    """model.py:22-65 on `module` (a FeatureEncoder: Sequential of Conv2d / BatchNorm2d(+ReLU) groups) -> feature maps
    [N, 32, H/4, W/4] bf16 in channels-last memory (the layout K1 stages).  Parameters, running statistics and state_dict keys
    are the module's own."""
    convs = [m for m in module.model if isinstance(m, torch.nn.Conv2d)]
    bns = [m for m in module.model if isinstance(m, torch.nn.BatchNorm2d)]
    x = image_rows(images)
    x = _bn_relu(conv3x3(x, convs[0].weight), bns[0])
    x = _bn_relu(conv3x3(x, convs[1].weight), bns[1], s2d=True)
    x = _bn_relu(conv3x3(x, k5s2_as_3x3(convs[2].weight)), bns[2])
    x = _bn_relu(conv3x3(x, convs[3].weight), bns[3])
    x = _bn_relu(conv3x3(x, convs[4].weight), bns[4], s2d=True)
    x = _bn_relu(conv3x3(x, k5s2_as_3x3(convs[5].weight)), bns[5])
    x = _bn_relu(conv3x3(x, convs[6].weight), bns[6])
    x = conv3x3(x, convs[7].weight)
    return x.squeeze(0).permute(1, 0, 2, 3)


def encode_features(module, images, bf16=True):
    """`self.feature_encoder(nn_input)` of model.py:181 as a call a host application can bind: feature maps [N, 32, H/4, W/4].
    `module` is the application's own FeatureEncoder (the reference's class or harness.FeatureEncoder: same Sequential, same
    state_dict).  bf16 with train-mode BatchNorm on a GPU runs encode_native (bf16 maps in channels-last memory, the layout K1
    stages); fp32, eval-mode BatchNorm or MVSB200_ENCODER=torch evaluate the module's own torch layers."""
    import os
    amp = bool(bf16) and images.is_cuda
    if amp and os.environ.get("MVSB200_ENCODER", "native") == "native" and encoder_ok(module, images):
        return encode_native(module, images)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        return module(images.contiguous(memory_format=torch.channels_last) if images.is_cuda else images)
