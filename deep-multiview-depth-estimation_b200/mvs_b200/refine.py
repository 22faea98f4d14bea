"""Depth refinement (SURVEY §8 row f2): the step right after the hot path, on the library's own kernels.

Reference: /root/reference/scripts/model.py:129-152 (`DepthRefinement`: Conv2d 4->32, 32->32, 32->32 with BatchNorm2d + ReLU,
Conv2d 32->1, residual added to the normalised depth) and :190-205 (normalise the initial depth map, resize the reference image
to the feature resolution, concatenate, refine, de-normalise).

  refine_input / refine_output   the glue as ONE launch each way (csrc/refine.cu) instead of ~10 elementwise / resize / concat
                                 launches forward and as many backward; the network's input leaves as bf16 channel-last rows of
                                 16 channels (4 carry data), the layout the K = 16 tensor-core convolution reads.
  refine_native                  the four 3x3 convolutions -- forward, data gradient, weight gradient -- on the tcgen05 stride-1
                                 kernels of the regulariser (nets2d.py: the maps are the planes of one volume, a 3x3 filter is
                                 the middle depth slice of a 3x3x3 one, packed straight from the Conv2d parameter), BatchNorm +
                                 ReLU the fused K3b kernels with the module's running statistics.  No library convolution is
                                 left in the refinement network.

Train mode, bf16 only (what the train step and the bf16 inference path run); DepthRefinement.forward keeps the stock torch layers for
eval-mode BatchNorm and fp32."""
from __future__ import annotations

import ctypes

import torch

from . import _lib, ops
from .ops import _need_cuda, _stream, _timed

_CP = 16      # channels per row of the network's input (4 real)
_CR = 8       # channels per row of the last convolution's output (1 real)


def _per_sample(t, B, what):
    t = t.detach().to(torch.float32).reshape(-1)
    if t.numel() != B:
        raise _lib.MvsB200Error(f"{what}: one value per sample expected ({B}), got {t.numel()}")
    return t.contiguous()


class _RefineInput(torch.autograd.Function):
    @staticmethod
    def forward(ctx, initial, images, n_views, d_min, span):
        _need_cuda(initial, "initial depth map")
        _need_cuda(images, "input images")
        if images.dtype != torch.float32 or images.dim() != 4 or images.shape[1] != 3:
            raise _lib.MvsB200Error(f"refine_input: images must be fp32 [N, 3, H, W], got {images.dtype} {tuple(images.shape)}")
        B, _, h, w = initial.shape
        if images.shape[0] < (B - 1) * n_views + 1:
            raise _lib.MvsB200Error(f"refine_input: {images.shape[0]} images for {B} samples of {n_views} views")
        x = initial.detach().float().contiguous()
        rows = torch.empty((1, _CP, B, h, w), dtype=torch.bfloat16, device=x.device, memory_format=torch.channels_last_3d)
        norm = torch.empty_like(x)
        with _timed("refine_glue"):
            _lib.call("mvsb200_refine_input_fwd", x.data_ptr(), images.data_ptr(), (ctypes.c_int64 * 4)(*images.stride()), int(n_views),
                      images.shape[2], images.shape[3], d_min.data_ptr(), span.data_ptr(), B, h, w, _CP, rows.data_ptr(),
                      norm.data_ptr(), _stream())
        ctx.save_for_backward(span)
        ctx.meta = (initial.shape, initial.dtype)
        return rows, norm

    @staticmethod
    def backward(ctx, g_rows, g_norm):
        (span,) = ctx.saved_tensors
        shape, dtype = ctx.meta
        B, n = shape[0], shape[2] * shape[3]
        if g_rows is not None:
            g_rows = g_rows.to(torch.bfloat16).contiguous(memory_format=torch.channels_last_3d)
        if g_norm is not None:
            g_norm = g_norm.float().contiguous()
        gi = torch.empty(shape, dtype=torch.float32, device=span.device)
        with _timed("refine_glue"):
            _lib.call("mvsb200_refine_input_bwd", ops._ptr(g_rows), _CP, ops._ptr(g_norm), span.data_ptr(), B, n, gi.data_ptr(), _stream())
        return gi.to(dtype), None, None, None, None


class _RefineOutput(torch.autograd.Function):
    @staticmethod
    def forward(ctx, res_rows, norm, d_min, span):
        _, cr, B, h, w = res_rows.shape
        r = res_rows.detach().contiguous(memory_format=torch.channels_last_3d)
        if r.dtype != torch.bfloat16:
            raise _lib.MvsB200Error(f"refine_output: bf16 rows expected, got {r.dtype}")
        nm = norm.detach().float().contiguous()
        out = torch.empty((B, 1, h, w), dtype=torch.float32, device=r.device)
        with _timed("refine_glue"):
            _lib.call("mvsb200_refine_output_fwd", r.data_ptr(), cr, nm.data_ptr(), d_min.data_ptr(), span.data_ptr(), B, h * w,
                      out.data_ptr(), _stream())
        ctx.save_for_backward(span)
        ctx.meta = (res_rows.shape, norm.shape)
        return out

    @staticmethod
    def backward(ctx, g):
        (span,) = ctx.saved_tensors
        rs, ns = ctx.meta
        _, cr, B, h, w = rs
        g = g.float().contiguous()
        g_rows = torch.empty(rs, dtype=torch.bfloat16, device=g.device, memory_format=torch.channels_last_3d)
        g_norm = torch.empty(ns, dtype=torch.float32, device=g.device)
        with _timed("refine_glue"):
            _lib.call("mvsb200_refine_output_bwd", g.data_ptr(), span.data_ptr(), B, h * w, cr, g_rows.data_ptr(), g_norm.data_ptr(),
                      _stream())
        return g_rows, g_norm, None, None


def refine_input(initial, images, n_views, d_min, span):
    """(rows, norm): rows = bf16 [1, 16, B, h, w] channel-last (the maps stacked as planes, nets2d.py): channel 0 the normalised
    depth (initial - d_min) / span, 1..3 the reference image of every sample (images[b * n_views], fp32 [N, 3, H, W], any
    strides) resized bilinearly to h x w, the rest zeros; norm = the normalised depth in fp32 [B, 1, h, w] (model.py:190-200).
    d_min / span: one value per sample."""
    B = initial.shape[0]
    return _RefineInput.apply(initial, images, int(n_views), _per_sample(d_min, B, "d_min"), _per_sample(span, B, "depth span"))


def refine_output(res_rows, norm, d_min, span):
    """(res_rows[0, 0] + norm) * span + d_min -> fp32 [B, 1, h, w] (model.py:150-151, :203); res_rows [1, c, B, h, w]."""
    B = res_rows.shape[2]
    return _RefineOutput.apply(res_rows, norm, _per_sample(d_min, B, "d_min"), _per_sample(span, B, "depth span"))


def layout_ok(module) -> bool:
    """Whether DepthRefinement `module` has the reference's layers: four bias-free 3x3 Conv2d 4 -> 32 -> 32 -> 32 -> 1."""
    convs = [m for m in getattr(module, "model", ()) if isinstance(m, torch.nn.Conv2d)]
    return (len(convs) == 4 and convs[0].in_channels == 4 and convs[-1].out_channels == 1
            and all(c.kernel_size == (3, 3) and c.stride == (1, 1) and c.padding == (1, 1) and c.bias is None for c in convs)
            and all(c.out_channels == 32 for c in convs[:3]))


def native_ok(module, x_like) -> bool:
    """Whether DepthRefinement `module` can run on the library's kernels: train-mode BatchNorm, CUDA, the reference's widths."""
    from . import conv3d_sm100
    return x_like.is_cuda and module.training and layout_ok(module) and conv3d_sm100.available()


def refine_native(module, initial, images, n_views, d_min, span):
    """model.py:190-205 on `module` (a DepthRefinement: Sequential of Conv2d / BatchNorm2d(+ReLU) triples): normalise, build the
    network's input, four convolutions with BatchNorm + ReLU between them, residual, de-normalise -> refined depth fp32
    [B, 1, h, w].  Parameters, running statistics and their state_dict keys are the module's own."""
    from .nets2d import _bn_relu, conv3x3
    convs = [m for m in module.model if isinstance(m, torch.nn.Conv2d)]
    bns = [m for m in module.model if isinstance(m, torch.nn.BatchNorm2d)]
    x, norm = refine_input(initial, images, n_views, d_min, span)
    for k in range(3):
        x = _bn_relu(conv3x3(x, convs[k].weight), bns[k])
    return refine_output(conv3x3(x, convs[3].weight, _CR), norm, d_min, span)


def refine_depth(module, initial, nn_input, n_views, d_min, d_int, d_num, d_scale, bf16=True):
    """The lines of `MVSNet.forward` after `extract_depth_map` (model.py:190-205) as one call a host application can bind:
    -> refined depth map fp32 [B, 1, h, w].  `module` is the application's own DepthRefinement (the reference's class or
    harness.DepthRefinement: same Sequential, same state_dict).  bf16 (the train-step precision) with train-mode BatchNorm on a
    GPU runs refine_native; anything else (fp32, eval-mode BatchNorm, MVSB200_REFINE=torch) evaluates the module's own torch
    layers around torch glue, as the reference does."""
    dev = initial.device
    return refine_spans(module, initial, nn_input, n_views, d_min.to(dev), d_int.to(dev) * d_num * d_scale, bf16)


def refine_spans(module, initial, nn_input, n_views, d_trans, span, bf16=True):
    """refine_depth on a depth offset and span (d_int * D_NUM * D_SCALE) per sample that already live on the device -- the form
    a captured CUDA graph replays."""
    import os
    import torch.nn.functional as F
    amp = bool(bf16) and nn_input.is_cuda
    if amp and os.environ.get("MVSB200_REFINE", "native") == "native" and nn_input.dtype == torch.float32 and native_ok(module, initial):
        return refine_native(module, initial, nn_input, n_views, d_trans, span)
    norm = (initial - d_trans) / span
    h, w = initial.shape[-2:]
    ref_img = F.interpolate(nn_input[::n_views], (h, w), mode="bilinear", align_corners=False)       # == nn_input[ref_views]
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        refined = module(torch.cat((norm, ref_img), 1))
    return refined.float() * span + d_trans
