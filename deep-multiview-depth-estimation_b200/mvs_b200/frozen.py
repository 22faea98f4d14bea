"""Eval-mode inference of a whole MVSNet on the library's kernels: FrozenMVSNet.

In eval mode every BatchNorm is a fixed per-channel affine map y = x * scale + shift with scale = w / sqrt(running_var + eps),
shift = b - running_mean * scale.  It needs no statistics pass, so it rides in the epilogue of the convolution in front of it
(conv3d_s1_kdn_kernel and deconv3d_s2_tc_kernel in their affine forms, csrc/conv3d_tc.cu).  It also frees the transposed
convolutions deconv_3_0 / deconv_2_0 from their dense canvases: only their central box C is read (regulariser.py), and without
batch statistics only C has to be written.

    model.eval()                 unchanged: encoder and refinement on the modules' torch layers, regulariser on the train-path
                                 kernels with separate BatchNorm passes
    FrozenMVSNet(model)          the same function on bf16 operands / fp32 accumulation, every convolution and BatchNorm on this
                                 library's kernels; the filters are packed and the BatchNorm vectors computed once, refresh()
                                 rewrites them in place from the bound module (a captured graph then replays the new values)

The bound module is only read: parameters, buffers and its training flag stay as they are.  Out of scope: gradients, fp32, the
depth-slab split (harness.DepthSlabMVSNet).

Layer sequence (scripts/model.py:20-65, :100-126, :129-152, :190-205):
  encoder      image rows -> 8 planar 3x3 convolutions (the 5x5 stride-2 layers on the space-to-depth form of their input),
               the first seven with BatchNorm + ReLU in the epilogue
  sweep        K1 (warp + variance) -> bf16 cost volume
  regulariser  conv_0_0 + BN_0 (epilogue) -> y0;  stacked stride-2 branches onto C -> affine_relu_geo (BN_k, the constant ring
               around C) -> conv_k_1 + BN_k (epilogue), output exactly on C -> enc[k];
               deconv_3_0 + BN_2 + enc[2] on C;  deconv_2_0 + BN_1 + enc[1] on C;  deconv_1_0 + BN_0 + y0 on the canvas;
               K3c (conv_out) -> K4 (softmax over depth)
  refinement   refine_input glue -> 3 planar convolutions with BatchNorm + ReLU epilogues -> last convolution -> refine_output
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib, api, nets2d, ops, refine
from .conv3d_sm100 import _NAT, _kdn_order, _n_rows, _pack
from .ops import _stream, _timed
from .regulariser import central_region

_CL3 = torch.channels_last_3d
_BRANCHES = ((1, 16), (2, 32), (3, 64))                # conv_k_0 / conv_k_1 / BN_k widths of the regulariser


def _fail(msg):
    raise _lib.MvsB200Error("FrozenMVSNet: " + msg)


def _reg_layout_error(reg):
    """None when `reg` has the layout of CostVolumeReg (in_ch 32, base_filt 8), else what differs."""
    conv, convT, bn = torch.nn.Conv3d, torch.nn.ConvTranspose3d, torch.nn.BatchNorm3d
    want = {"conv_0_0": (conv, 32, 8, 1), "conv_1_0": (conv, 32, 16, 2), "conv_2_0": (conv, 32, 32, 2), "conv_3_0": (conv, 32, 64, 2),
            "conv_1_1": (conv, 16, 16, 1), "conv_2_1": (conv, 32, 32, 1), "conv_3_1": (conv, 64, 64, 1),
            "deconv_3_0": (convT, 64, 32, 2), "deconv_2_0": (convT, 32, 16, 2), "deconv_1_0": (convT, 16, 8, 2),
            "conv_out": (conv, 8, 1, 1)}
    for name, (kind, ci, co, s) in want.items():
        m = getattr(reg, name, None)
        if not isinstance(m, kind) or (m.in_channels, m.out_channels, m.kernel_size, m.stride, m.padding) != (ci, co, (3,) * 3, (s,) * 3, (1,) * 3) \
                or m.bias is not None or m.weight.dtype != torch.float32:
            return f"cost_volume_reg.{name} is not the reference's {ci} -> {co}, 3x3x3, stride {s}, bias-free fp32 layer"
    for k, c in enumerate((8, 16, 32, 64)):
        m = getattr(reg, f"BN_{k}", None)
        if not isinstance(m, bn) or m.num_features != c or m.running_mean is None or m.weight is None:
            return f"cost_volume_reg.BN_{k} is not a {c}-channel BatchNorm3d with running statistics and an affine map"
    return None


class FrozenMVSNet:
    """MVSNet.forward with eval-mode BatchNorm (running statistics) on the library's kernels, under no_grad.

    model: a harness.MVSNet, or any module whose feature_encoder, cost_volume_reg and depthmap_refine have the reference's layout.
    d_num / d_scale: the depth sweep (default: the model's own).  Anything the kernels cannot run raises MvsB200Error naming the
    reason: a module on the CPU, precision "fp32", a layout other than the reference's; at forward also CPU tensors and images
    whose sides are not multiples of 4 or are below 12.  There is no fallback."""

    def __init__(self, model, d_num=None, d_scale=None):
        enc, reg, ref = (getattr(model, n, None) for n in ("feature_encoder", "cost_volume_reg", "depthmap_refine"))
        if enc is None or reg is None or ref is None:
            _fail("the model needs feature_encoder, cost_volume_reg and depthmap_refine modules")
        why = nets2d.encoder_layout_error(enc) or _reg_layout_error(reg)
        if why is None and not refine.layout_ok(ref):
            why = "depthmap_refine is not the reference's 4 -> 32 -> 32 -> 32 -> 1 stack of bias-free 3x3 Conv2d"
        if why is not None:
            _fail(why)
        if "fp32" in (getattr(model, "precision", None), getattr(reg, "precision", None)):
            _fail('precision "fp32" is not supported: the frozen model computes on bf16 operands with fp32 accumulation')
        params = list(model.parameters()) + list(model.buffers())
        if not all(t.is_cuda for t in params):
            _fail("the model lives (partly) on the CPU; mvs_b200 has no CPU path")
        self.model = model
        self.d_num = int(d_num if d_num is not None else model.d_num)
        self.d_scale = d_scale if d_scale is not None else model.d_scale
        self.n_depth_est = int(getattr(model, "n_depth_est", getattr(reg, "n_depth_est", 5)))
        self.after_encoder_event = None                  # harness.GraphedInference records it after the encoder
        self.device = reg.conv_out.weight.device
        self._enc_convs = [m for m in enc.model if isinstance(m, torch.nn.Conv2d)]
        self._enc_bns = [m for m in enc.model if isinstance(m, torch.nn.BatchNorm2d)]
        self._ref_convs = [m for m in ref.model if isinstance(m, torch.nn.Conv2d)]
        self._ref_bns = [m for m in ref.model if isinstance(m, torch.nn.BatchNorm2d)]
        self._w, self._bn = {}, {}
        self._geo = {}
        self.refresh()

    # ------------------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def refresh(self):
        """Re-read the bound module's weights and running statistics: every packed filter and every BatchNorm scale / shift
        vector is rewritten IN PLACE (same addresses), so a CUDA graph captured over this object replays the new values."""
        reg = self.model.cost_volume_reg
        # 2D layers: the kdn filter operand of the planar kernel ([9][3][n_rows][Cin], middle depth slice)
        for i, (c, (ci, co, k, _)) in enumerate(zip(self._enc_convs, nets2d._ENC_LAYERS)):
            w = c.weight if k == 3 else nets2d.k5s2_as_3x3(c.weight)
            cx = 8 if i == 0 else (4 * ci if k == 5 else ci)            # channels per input row (images: 8, 3 real)
            self._w[f"enc{i}"] = nets2d._pack2d(w.detach().float().contiguous(), "fwd", _n_rows(co), max(cx, 16), out=self._w.get(f"enc{i}"))
        for i, c in enumerate(self._ref_convs):
            cy = 32 if i < 3 else refine._CR
            cx = refine._CP if i == 0 else 32
            self._w[f"ref{i}"] = nets2d._pack2d(c.weight.detach().float().contiguous(), "fwd", _n_rows(cy), cx, out=self._w.get(f"ref{i}"))
        # regulariser: conv_0_0 / conv_k_1 as kdn operands, the stacked branches as one [27][112][32] operand, the transposed
        # convolutions as [28][n_rows][Cin] (tap 27 all zeros), conv_out as the [27][8] fp32 table of K3c
        self._w["conv_0_0"] = _pack(reg.conv_0_0.weight, 0, 16, _kdn_order(_NAT), out=self._w.get("conv_0_0"))
        for k, c in _BRANCHES:
            self._w[f"conv_{k}_1"] = _pack(getattr(reg, f"conv_{k}_1").weight, 0, _n_rows(c), _kdn_order(_NAT), out=self._w.get(f"conv_{k}_1"))
        w_cat = torch.cat([getattr(reg, f"conv_{k}_0").weight.detach() for k, _ in _BRANCHES], 0)
        self._w["stacked"] = _pack(w_cat, 0, 112, _NAT, out=self._w.get("stacked"))
        for name in ("deconv_3_0", "deconv_2_0", "deconv_1_0"):
            w = getattr(reg, name).weight
            self._w[name] = _pack(w, 1, _n_rows(w.shape[1]), _NAT + [-1], out=self._w.get(name))
        w27 = reg.conv_out.weight.detach().float()[0].permute(1, 2, 3, 0).reshape(27, 8)
        if "conv_out" in self._w:
            self._w["conv_out"].copy_(w27)
        else:
            self._w["conv_out"] = w27.contiguous()
        # BatchNorm scale / shift in fp64, stored as fp32
        bns = {f"enc{i}": b for i, b in enumerate(self._enc_bns)}
        bns.update({f"ref{i}": b for i, b in enumerate(self._ref_bns)})
        bns.update({f"BN_{k}": getattr(reg, f"BN_{k}") for k in range(4)})
        for name, b in bns.items():
            scale = b.weight.detach().double() / torch.sqrt(b.running_var.detach().double() + b.eps)
            shift = b.bias.detach().double() - b.running_mean.detach().double() * scale
            if name in self._bn:
                self._bn[name][0].copy_(scale)
                self._bn[name][1].copy_(shift)
            else:
                self._bn[name] = (scale.float().contiguous(), shift.float().contiguous())

    # ------------------------------------------------------------------------------------------------------------------
    def __call__(self, *args, **kwargs):
        return self.forward(*args, **kwargs)

    @torch.no_grad()
    def forward(self, nn_input, K_batch, R_batch, T_batch, d_min, d_int, batch_size, n_views, sweep=None, return_confidence=False):
        """MVSNet.forward (model.py:168-207) -> (initial, refined) depth maps fp32 [B, 1, H/4, W/4].  sweep: an ops.PlaneSweep
        already holding this batch's geometry on the device, as in harness.MVSNet.forward.  return_confidence: also return
        the photometric confidence of the initial depth map (ops.depth_confidence) -> (initial, refined, confidence); the
        depth-axis softmax, depth and confidence then run as one launch, and initial and refined stay bit-identical."""
        if not nn_input.is_cuda:
            _fail(f"the input images live on {nn_input.device}; mvs_b200 has no CPU path")
        if nn_input.dtype != torch.float32 or nn_input.dim() != 4 or nn_input.shape[1] != 3:
            _fail(f"fp32 images [N, 3, H, W] expected, got {nn_input.dtype} {tuple(nn_input.shape)}")
        H, W = nn_input.shape[2:]
        if H % 4 or W % 4 or min(H, W) < 12:
            _fail(f"image sides must be multiples of 4 and at least 12, got {H} x {W}")
        feats = self.encode(nn_input).float()
        ev = self.after_encoder_event
        if ev is not None and torch.cuda.is_current_stream_capturing():
            ev.record()
        warped, d_batch, _ = api.homography_warping(K_batch, R_batch, T_batch, d_min, d_int, feats, batch_size, n_views, self.d_num,
                                                    self.d_scale, sweep=sweep)
        cost = api.assemble_cost_volume(warped, n_views, torch.bfloat16)
        conf = None
        if return_confidence:
            _, _, initial, conf = ops.softmax_depth_confidence(self.logits(cost), d_batch, self.n_depth_est)
        else:
            initial = api.extract_depth_map(self.regularise(cost), d_batch, self.n_depth_est)
        dev = initial.device
        refined = self.refine(initial, nn_input, n_views, d_min.to(dev), d_int.to(dev) * self.d_num * self.d_scale)
        return (initial, refined) if conf is None else (initial, refined, conf)

    # ------------------------------------------------------------------------------------------------------------------
    def _conv2d(self, x, wname, cy, bn=None):
        """3x3 / padding-1 convolution of stacked maps x [1, cx, N, H, W] -> [1, cy, N, H, W]; bn: BatchNorm + ReLU epilogue."""
        _, cx, N, H, Wd = x.shape
        y = torch.empty((1, cy, N, H, Wd), dtype=torch.bfloat16, device=x.device, memory_format=_CL3)
        with _timed("conv2d_tc"):
            if bn is None:
                _lib.call("mvsb200_conv2d_rows_fwd", x.data_ptr(), self._w[wname].data_ptr(), y.data_ptr(), N, H, Wd, cx, cy, cy,
                          _n_rows(cy), _stream())
            else:
                sc, sh = self._bn[bn]
                _lib.call("mvsb200_conv3d_s1_fwd_kdn_affine", x.data_ptr(), self._w[wname].data_ptr(), y.data_ptr(), 1, N, H, Wd, cx,
                          N, H, Wd, cy, cy, _n_rows(cy), 0, -1, -1, 1, sc.data_ptr(), sh.data_ptr(), _stream())
        return y

    def encode(self, images):
        """model.py:20-65 -> feature maps [N, 32, H/4, W/4] bf16 (channels-last memory)."""
        x = nets2d.image_rows(images)
        for i, (_, co, k, _) in enumerate(nets2d._ENC_LAYERS):
            if k == 5:
                x = nets2d.space_to_depth(x)
            x = self._conv2d(x, f"enc{i}", co, f"enc{i}" if i < 7 else None)
        return x.squeeze(0).permute(1, 0, 2, 3)

    def refine(self, initial, images, n_views, d_trans, span):
        """model.py:190-205 -> refined depth fp32 [B, 1, h, w]."""
        x, norm = refine.refine_input(initial, images, n_views, d_trans, span)
        for i in range(3):
            x = self._conv2d(x, f"ref{i}", 32, f"ref{i}")
        return refine.refine_output(self._conv2d(x, "ref3", refine._CR), norm, d_trans, span)

    # ------------------------------------------------------------------------------------------------------------------
    def _geometry(self, dims):
        g = self._geo.get(dims)
        if g is None:
            reg = [central_region(n) for n in dims]
            C_lo = tuple(lo for lo, _, _ in reg)
            C_dims = tuple(hi - lo + 1 for lo, hi, _ in reg)
            E_lo = tuple(max(0, lo - 1) for lo in C_lo)
            E_dims = tuple(min(n - 1, lo + m) - e + 1 for n, lo, m, e in zip(dims, C_lo, C_dims, E_lo))
            off = tuple(lo - 1 - e for lo, e in zip(C_lo, E_lo))       # conv_k_1 on E -> exactly C (TMA zero fill past E)
            pads = tuple(L for _, _, L in reg)
            g = self._geo[dims] = (C_lo, C_dims, E_lo, E_dims, off, pads)
        return g

    def _kdn(self, x, wname, cout, out_dims, off, bn):
        B, cin = x.shape[:2]
        y = torch.empty((B, cout) + tuple(out_dims), dtype=torch.bfloat16, device=x.device, memory_format=_CL3)
        sc, sh = self._bn[bn]
        with _timed("conv3d_s1_tc", 2.0 * 27 * cin * cout * y.numel() / cout):
            _lib.call("mvsb200_conv3d_s1_fwd_kdn_affine", x.data_ptr(), self._w[wname].data_ptr(), y.data_ptr(), B, *x.shape[2:], cin,
                      *out_dims, cout, cout, _n_rows(cout), *off, 0, sc.data_ptr(), sh.data_ptr(), _stream())
        return y

    def _deconv(self, x, wname, bn, canvas, pads, win_lo, win_dims, add):
        B, cin = x.shape[:2]
        cout = self.model.cost_volume_reg.get_submodule(wname).out_channels
        y = torch.empty((B, cout) + tuple(win_dims), dtype=torch.bfloat16, device=x.device, memory_format=_CL3)
        sc, sh = self._bn[bn]
        ys = (ctypes.c_int64 * 4)(y.stride(0), y.stride(2), y.stride(3), y.stride(4))
        win = (ctypes.c_int * 6)(*win_lo, *win_dims)
        with _timed("deconv3d_s2_tc"):
            _lib.call("mvsb200_deconv3d_s2_fwd_affine", x.data_ptr(), self._w[wname].data_ptr(), y.data_ptr(), B, *x.shape[2:], cin,
                      *canvas, cout, _n_rows(cout), *pads, win, ys, sc.data_ptr(), sh.data_ptr(), add.data_ptr(), _stream())
        return y

    def regularise(self, cost):
        """CostVolumeReg.forward in eval mode: bf16 cost volume [B, 32, D, h, w] (channels-last) -> probability volume
        [B, 1, D, h, w] fp32."""
        return ops.softmax_over_depth(self.logits(cost), self.n_depth_est)

    def logits(self, cost):
        """regularise() up to (excluding) the depth softmax: fp32 logits [B, 1, D, h, w]."""
        B, cin, D, h, w = cost.shape
        if not cost.is_cuda or cost.dtype != torch.bfloat16 or cin != 32 or min(D, h, w) < 3:
            _fail(f"bf16 CUDA cost volume [B, 32, D, h, w] with D, h, w >= 3 expected, got {cost.dtype} {tuple(cost.shape)} on {cost.device}")
        x = cost.contiguous(memory_format=_CL3)
        dims = (D, h, w)
        C_lo, C_dims, E_lo, E_dims, off, pads = self._geometry(dims)
        y0 = self._kdn(x, "conv_0_0", 8, dims, (-1, -1, -1), "BN_0")
        S = torch.empty((B, 112) + C_dims, dtype=torch.bfloat16, device=x.device, memory_format=_CL3)
        with _timed("conv3d_s2_tc", 2.0 * 27 * 32 * S.numel()):
            _lib.call("mvsb200_conv3d_s2_fwd", x.data_ptr(), self._w["stacked"].data_ptr(), S.data_ptr(), B, D, h, w, 32, *C_dims, 112, 112,
                      112, *pads, _stream())
        enc, c0 = {}, 0
        for k, c in _BRANCHES:
            sc, sh = self._bn[f"BN_{k}"]
            # BN_k + ReLU of the branch on C, its constant relu(shift) on the ring E \ C (the zero canvas outside C, normalised)
            X = ops.affine_relu_geo(S[:, c0:c0 + c], sc, sh, C_lo, E_lo, E_dims)
            enc[k] = self._kdn(X, f"conv_{k}_1", c, C_dims, off, f"BN_{k}")
            c0 += c
        s3 = self._deconv(enc[3], "deconv_3_0", "BN_2", dims, pads, C_lo, C_dims, enc[2])
        s2 = self._deconv(s3, "deconv_2_0", "BN_1", dims, pads, C_lo, C_dims, enc[1])
        z = self._deconv(s2, "deconv_1_0", "BN_0", dims, pads, (0, 0, 0), dims, y0)
        logits = torch.empty((B, 1, D, h, w), dtype=torch.float32, device=x.device)
        with _timed("conv_out_fwd"):
            _lib.call("mvsb200_conv_out_fwd", z.data_ptr(), self._w["conv_out"].data_ptr(), logits.data_ptr(), B, D, h, w, _stream())
        return logits
