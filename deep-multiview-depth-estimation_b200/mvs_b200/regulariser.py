"""CostVolumeReg drop-in (reference: /root/reference/scripts/model.py:68-126, factories :223-247).

Same constructor, same parameter / buffer names (state_dict compatible: conv_0_0.weight ... BN_3.num_batches_tracked),
same construction order (so ``torch.manual_seed(s); CostVolumeReg()`` draws the same initial weights), same
forward contract ``cv[B,32,D,h,w] -> prob[B,1,D,h,w]``.

What is different is HOW MUCH is computed.  The reference's "U-Net" never changes resolution: its stride-2
convolutions use padding ``dim/2+1`` (scripts/config.py:20), so every tensor is a full D x h x w canvas
(SURVEY App. A.5).  But on that canvas
  * a stride-2 conv output is exactly 0 outside a central box C (per axis [ceil((p-2)/2), floor((n-1+p)/2)],
    ~1/8 of the voxels); after BatchNorm+ReLU the outside is one constant per channel;
  * a stride-2 transposed conv only READS the box C of its input.
Hence: conv_{1,2,3}_0 are evaluated on C only; conv_{1,2,3}_1 are evaluated on C dilated by one voxel (the
part that sees real data), the rest of their canvas is 27 closed-form constants per channel that enter the
BatchNorm statistics analytically; the transposed convs run from C.  Dense full-canvas work remains only for
conv_0_0, the three transposed-conv outputs (their batch statistics are over the full canvas) and conv_out.
Results are those of the reference network (same statistics, same zero regions), with ~7x fewer FLOPs than
the dense canvases cuDNN executes for the reference (DESIGN.md §K3).

The convolutions themselves go through ``conv_backend`` (mvs_b200.conv3d).

Precision (``precision=``), i.e. what ``CostVolumeReg()`` -- the call of scripts/model.py:161 -- computes in:
  "bf16" (default)  the native path: bf16 operands, fp32 accumulation on the tcgen05 kernels of libmvs_b200.so (BASELINE
                    north_star "bf16/tf32 in, fp32 accumulate"); fp32 volumes in and out, parameters stay fp32.  Tolerance
                    against the reference's fp32 network: probability volume 1e-2 relative (max-norm), the north_star figure
                    for the bf16 convolution path; tests/test_gpu_parity.py, tests/test_gpu_fullsize.py.
  "fp32"            explicit opt-in for parity diagnostics at 1e-4: fp32 volumes through the library convolutions with TF32
                    switched off INSIDE the module (it does not depend on torch.backends.cudnn.allow_tf32).
"""
from __future__ import annotations

import os

import sys

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, ops
from . import conv3d as conv_backends


def default_device():
    """The reference's constructor default is ``device=DEVICE`` (scripts/model.py:70, scripts/config.py:24): the host
    application's ``config.DEVICE`` when that module is loaded, else the current CUDA device, else the CPU (parameters can be
    built there; forward needs CUDA)."""
    cfg = sys.modules.get("config")
    dev = getattr(cfg, "DEVICE", None)
    if isinstance(dev, (torch.device, str)):
        return torch.device(dev)
    if torch.cuda.is_available():
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


def central_region(n: int):
    """Per-axis geometry of the reference's stride-2 layers on a canvas of size n.
    Returns (lo, hi, L): output box [lo, hi] that can be non-zero / input box a transposed conv reads,
    and L = p - 2*lo, the left padding of the equivalent small conv."""
    p = n // 2 + 1                      # scripts/config.py:20
    lo = (p - 1) // 2                   # ceil((p-2)/2)
    hi = min(n - 1, (n - 1 + p) // 2)
    return lo, hi, p - 2 * lo


def _bview(v):
    return v.view(1, -1, 1, 1, 1)


class CostVolumeReg(nn.Module):
    def __init__(self, in_ch=32, base_filt=8, device=None, precision="bf16", conv_backend="auto", n_depth_est=5):
        super().__init__()
        if device is None:
            device = default_device()
        f = base_filt
        mk = lambda i, o, s: nn.Conv3d(i, o, 3, stride=s, padding=1, bias=False, device=device)
        mkT = lambda i, o: nn.ConvTranspose3d(i, o, 3, stride=2, padding=1, bias=False, device=device)
        # construction order == reference (model.py:76-95) so default init consumes the RNG identically
        self.conv_0_0 = mk(in_ch, f, 1)
        self.conv_1_0 = mk(in_ch, f * 2, 2)
        self.conv_2_0 = mk(in_ch, f * 4, 2)
        self.conv_3_0 = mk(in_ch, f * 8, 2)
        self.conv_1_1 = mk(f * 2, f * 2, 1)
        self.conv_2_1 = mk(f * 4, f * 4, 1)
        self.conv_3_1 = mk(f * 8, f * 8, 1)
        self.deconv_3_0 = mkT(f * 8, f * 4)
        self.deconv_2_0 = mkT(f * 4, f * 2)
        self.deconv_1_0 = mkT(f * 2, f)
        self.conv_out = mk(f, 1, 1)
        self.ReLU = nn.ReLU()
        bn = lambda c: nn.BatchNorm3d(c, eps=1e-5, momentum=0.1, track_running_stats=True, device=device)
        self.BN_0, self.BN_1, self.BN_2, self.BN_3 = bn(f), bn(f * 2), bn(f * 4), bn(f * 8)
        self.Norm = nn.Softmax(2)       # kept for state/printing parity; forward uses the fused K4 kernel
        if precision not in ("fp32", "bf16"):
            raise ValueError("precision must be 'fp32' or 'bf16'")
        self.precision = precision
        self.conv_backend = conv_backend
        self.n_depth_est = int(n_depth_est)

    # ------------------------------------------------------------------------------------------
    def forward(self, cv: torch.Tensor) -> torch.Tensor:
        if not cv.is_cuda:
            raise _lib.MvsB200Error("CostVolumeReg.forward needs a CUDA tensor; mvs_b200 has no CPU path")
        if not self.conv_out.weight.is_cuda:
            raise _lib.MvsB200Error("CostVolumeReg parameters live on the CPU; build the module with device=cuda or move it "
                                    "with .to(device) -- mvs_b200 has no CPU path")
        # precision="fp32" means fp32: that mode's library convolutions run with TF32 off in forward AND backward, whatever
        # the process-wide torch.backends flags say (conv3d.ExactTorchConvBackend); the bf16 mode runs on this library's kernels
        be = conv_backends.ExactTorchConvBackend if self.precision == "fp32" else conv_backends.get(self.conv_backend)
        logits = self.logits(cv, be)
        return ops.softmax_over_depth(logits, self.n_depth_est)

    # ------------------------------------------------------------------------------------------
    def _w(self, name, dtype):
        w = getattr(self, name).weight
        return w if w.dtype == dtype else w.to(dtype)

    def _bn_dense(self, bn: nn.BatchNorm3d, x, crop=None, canvas=None, add=None):
        """BatchNorm (+ReLU) over a full canvas.  `canvas` = (D,h,w): the canvas sits at the origin of x, which may be one
        plane/line/column larger (un-cropped transposed conv); `crop` (three slices): only that box of the result is
        produced.  On the GPU in train mode this is the fused channel-last kernel family of libmvs_b200.so (K3b); the
        torch expressions below serve eval mode and the CPU unit tests of the canvas algebra."""
        if x.is_cuda and bn.training:
            box = None if crop is None else tuple((c.start, c.stop) for c in crop)
            # the running statistics (momentum, unbiased variance, counter) are updated inside the statistics' finalize launch
            y, _, _ = ops.batchnorm_relu_train(x, bn.weight, bn.bias, bn.eps, relu=True, crop=box, canvas=canvas,
                                               running=(bn.running_mean, bn.running_var, bn.num_batches_tracked), momentum=bn.momentum,
                                               partials=getattr(x, "_mvs_bn_partials", None),
                                               add=None if add is None else add.to(x.dtype))
            return y
        if canvas is not None:
            x = x[..., :canvas[0], :canvas[1], :canvas[2]]
        if x.is_cuda:
            if not torch.is_grad_enabled() or not (x.requires_grad or bn.weight.requires_grad):
                scale = bn.weight * torch.rsqrt(bn.running_var + bn.eps)
                y = ops.affine_relu(x, scale, bn.bias - bn.running_mean * scale, relu=True)
                y = y if crop is None else y[(slice(None), slice(None)) + tuple(crop)]
                return y if add is None else y + add.to(y.dtype)
        y = F.batch_norm(x, bn.running_mean, bn.running_var, bn.weight, bn.bias, bn.training, bn.momentum, bn.eps)
        if bn.training:
            bn.num_batches_tracked += 1
        y = F.relu(y)
        y = y if crop is None else y[(slice(None), slice(None)) + tuple(crop)]
        return y if add is None else y + add.to(y.dtype)

    def _bn_affine(self, bn: nn.BatchNorm3d, mean, var, n_full):
        """scale/shift of BatchNorm given full-canvas batch statistics (train) or the running ones (eval)."""
        if bn.training:
            with torch.no_grad():
                m = bn.momentum
                bn.running_mean.mul_(1 - m).add_(mean.detach(), alpha=m)
                bn.running_var.mul_(1 - m).add_(var.detach() * (n_full / max(n_full - 1, 1)), alpha=m)
                bn.num_batches_tracked += 1
        else:
            mean, var = bn.running_mean, bn.running_var
        scale = bn.weight * torch.rsqrt(var + bn.eps)
        return scale, bn.bias - mean * scale

    def logits(self, cv: torch.Tensor, be) -> torch.Tensor:
        """Everything up to (excluding) the depth softmax.  `be` is a conv backend (mvs_b200.conv3d)."""
        B, _, D, h, w = cv.shape
        dims = (D, h, w)
        if min(dims) < 2:
            raise ValueError("CostVolumeReg needs D, h, w >= 2")
        dt = torch.bfloat16 if self.precision == "bf16" else torch.float32
        x = cv if cv.dtype == dt else cv.to(dt)
        # a backend that packs its own filters takes the fp32 parameters as they are (no bf16 copies of the weights, no casts
        # of their gradients)
        wdt = torch.float32 if getattr(be, "fp32_weights", False) else dt
        n_full = B * D * h * w
        reg = [central_region(n) for n in dims]
        C = tuple(slice(lo, hi + 1) for lo, hi, _ in reg)                     # central box on the canvas
        train = self.BN_0.training

        # the three stride-2 branches all read cv (model.py:104-110): ONE convolution with the weights stacked along
        # Cout (16+32+64 = 112) reads the cost volume once instead of three times; with conv_0_0 they form one autograd node
        # (the cost volume's gradient is accumulated inside the kernels, not by an elementwise pass of autograd)
        w_parts = [self._w(f"conv_{k}_0", wdt) for k in (1, 2, 3)]
        w_cat = torch.cat(w_parts, 0)
        # where a weight gradient of w_cat computed off the launching stream goes (ops.wgrad_fork): the rows of each branch
        rows = [0]
        for p in w_parts:
            rows.append(rows[-1] + p.shape[0])
        w_cat._mvs_wgrad_to = [(p, (lambda g, a=a, b=b: g[a:b])) for p, a, b in zip(w_parts, rows, rows[1:])]
        widths = [self.conv_1_0.out_channels, self.conv_2_0.out_channels, self.conv_3_0.out_channels]
        box_pads, box_dims = tuple(L for _, _, L in reg), tuple(hi - lo + 1 for lo, hi, _ in reg)
        S_parts = None
        entry = be.entry_convs(x, self._w("conv_0_0", wdt), w_cat, box_pads, box_dims, widths) if hasattr(be, "entry_convs") else None
        if entry is not None:
            c00, S_parts = entry
        else:
            c00 = be.conv3d(x, self._w("conv_0_0", wdt), 1, (1, 1, 1))
        y0 = self._bn_dense(self.BN_0, c00)

        # ---- encoder branches: stride-2 conv on C, then stride-1 conv on C (+1 ring for the statistics)
        P = tuple(L if L >= 2 else L + 2 for _, _, L in reg)                  # symmetric pad with P == L (mod 2)
        off = tuple((Pp - L) // 2 for Pp, (_, _, L) in zip(P, reg))
        cut = tuple(slice(o, o + (hi - lo + 1)) for o, (lo, hi, _) in zip(off, reg))
        E_lo = [max(0, lo - 1) for lo, _, _ in reg]
        E_hi = [min(n - 1, hi + 1) for (_, hi, _), n in zip(reg, dims)]
        F_lo = [max(0, e - 1) for e in E_lo]
        F_hi = [min(n - 1, e + 1) for e, n in zip(E_hi, dims)]
        zpad, bgpad, inner = [], [], []
        for ax in (2, 1, 0):                                                  # F.pad order: w, h, d
            lo, hi, _ = reg[ax]
            zpad += [1 if E_lo[ax] == 0 else 0, 1 if E_hi[ax] == dims[ax] - 1 else 0]
            bgpad += [lo - F_lo[ax], F_hi[ax] - hi]
        for ax in range(3):
            lo, hi, _ = reg[ax]
            inner.append(slice(lo - E_lo[ax], lo - E_lo[ax] + (hi - lo + 1)))  # C inside E
        enc = {}
        if S_parts is None and hasattr(be, "conv3d_s2_box"):                  # tcgen05 stride-2 kernel, straight onto the box
            S_parts = be.conv3d_s2_box(x, w_cat, box_pads, box_dims, widths)
        if S_parts is None:
            S_parts = torch.split(be.conv3d(x, w_cat, 2, P)[(slice(None), slice(None)) + cut], widths, 1)
        S_split = dict(zip((1, 2, 3), S_parts))
        C_lo = [lo for lo, _, _ in reg]
        C_dims = [hi - lo + 1 for lo, hi, _ in reg]
        F_dims = [F_hi[ax] - F_lo[ax] + 1 for ax in range(3)]
        E_dims = [E_hi[ax] - E_lo[ax] + 1 for ax in range(3)]
        for k, bn in ((1, self.BN_1), (2, self.BN_2), (3, self.BN_3)):
            S = S_split[k]
            Wk = self._w(f"conv_{k}_1", wdt)
            if x.is_cuda:
                # GPU: statistics and normalisation of the box tensors in libmvs_b200.so (K3d), per-channel algebra here
                if train:
                    # fused op: one statistics pass + one normalise pass forward; backward = one reduction + one apply pass that
                    # writes the branch's gradient straight into the strided convolution's padded gradient buffer
                    # (the running statistics are updated inside the op's per-channel algebra launch)
                    X, scale, shift, mean, var = ops.box_batchnorm_relu(S, bn.weight, bn.bias, n_full, bn.eps, C_lo, F_lo, F_dims,
                                                                        getattr(S, "_mvs_grad_dest", None),
                                                                        running=(bn.running_mean, bn.running_var, bn.num_batches_tracked),
                                                                        momentum=bn.momentum, sums=getattr(S, "_mvs_box_sums", None))
                    bg = F.relu(shift)                                        # everywhere else on the canvas
                else:
                    scale, shift = self._bn_affine(bn, None, None, n_full)
                    bg = F.relu(shift)
                    X = ops.affine_relu_geo(S, scale, shift, C_lo, F_lo, F_dims)
                # (X: conv_k_1 input over F = C dilated by 2 (clipped): data on C, BatchNorm'd zero (= bg) around it)
                if any(zpad):
                    X = F.pad(X, zpad)                                        # canvas border -> zero padding
                T = be.conv3d(X if X.dtype == dt else X.to(dt), Wk, 1, (0, 0, 0))      # output exactly on E
                if train:
                    # statistics node and normalisation node linked: the backward makes one reduction and one apply pass
                    link, (t1, t2) = ops.box_batchnorm_linked(T)
                    # what the layer's output sums to outside E (27 closed-form border classes of a convolution of the constant
                    # bg) joins the sums over E inside the per-channel algebra launch, which also updates the running statistics
                    if os.environ.get("MVSB200_OUTSIDE_SUMS", "fused") == "fused":
                        A1, A2 = ops.outside_sums(Wk, bg, self._outside_geometry(dims, E_lo, E_hi, B, Wk.device)[1])
                    else:                                                     # the torch expressions (A/B, and the form the test checks against)
                        val, cnt = self._outside_classes(Wk.float(), bg, dims, E_lo, E_hi, B)
                        vc = val.double() * cnt.double()
                        A1, A2 = vc.sum((1, 2, 3)), (vc * val).sum((1, 2, 3))
                    scale, shift = ops.box_stats_affine(t1, t2, A1, A2, bn.weight, bn.bias, n_full,
                                                        bn.eps, running=(bn.running_mean, bn.running_var, bn.num_batches_tracked),
                                                        momentum=bn.momentum)
                    enc[k] = ops.affine_relu_geo_linked(T, scale, shift, E_lo, C_lo, C_dims, link)   # on C, storage dtype of the path
                else:
                    scale, shift = self._bn_affine(bn, None, None, n_full)
                    enc[k] = ops.affine_relu_geo(T, scale, shift, E_lo, C_lo, C_dims)
                continue
            Sf = S.float()
            if train:
                mean = Sf.sum((0, 2, 3, 4)) / n_full
                n_c = Sf.numel() // Sf.shape[1]
                var = ((Sf - _bview(mean)).pow(2).sum((0, 2, 3, 4)) + (n_full - n_c) * mean.pow(2)) / n_full
            else:
                mean = var = None
            scale, shift = self._bn_affine(bn, mean, var, n_full)
            a = F.relu(Sf * _bview(scale) + _bview(shift))                    # on C
            bg = F.relu(shift)                                                # everywhere else on the canvas
            # conv_k_1 input over F = C dilated by 2 (clipped): background constant + real data on C
            X = F.pad(a - _bview(bg), bgpad) + _bview(bg)
            X = F.pad(X, zpad)                                                # canvas border -> zero padding
            T = be.conv3d(X.to(dt).contiguous(memory_format=torch.channels_last_3d), Wk, 1, (0, 0, 0))   # output exactly on E
            Tf = T.float()
            if train:
                mean, var = self._stats_with_constant_outside(Tf, Wk.float(), bg, dims, E_lo, E_hi, B, n_full)
            scale, shift = self._bn_affine(bn, mean if train else None, var if train else None, n_full)
            Tc = Tf[(slice(None), slice(None)) + tuple(inner)]
            enc[k] = F.relu(Tc * _bview(scale) + _bview(shift))               # on C, fp32

        # ---- decoder: transposed convs read only C; their outputs are dense canvases (statistics are dense)
        Lp = tuple(L for _, _, L in reg)

        def up(z, name, bn, crop=None, add=None):
            # channel-last operands keep the library on its NDHWC kernels (no layout-conversion passes over the canvas)
            U = be.conv_transpose3d_alloc(z.to(dt).contiguous(memory_format=torch.channels_last_3d), self._w(name, wdt), 2, Lp, dims)
            # U holds the canvas at its origin (+ up to one slack plane/line/column); `add`: the skip addition (model.py:117-123)
            # rides on the normalisation's apply pass
            return self._bn_dense(bn, U, crop, dims, add)

        # the transposed convs' canvases are normalised with full-canvas statistics but only their box C is read
        # skip additions in the storage dtype of the path (bf16 path: one more bf16 rounding instead of two fp32 round trips
        # of the box tensors per addition, forward and backward)
        s3 = up(enc[3], "deconv_3_0", self.BN_2, C, enc[2])                  # c3 + enc[2]
        s2 = up(s3, "deconv_2_0", self.BN_1, C, enc[1])                      # c2 + enc[1]
        z = up(s2, "deconv_1_0", self.BN_0, None, y0)                        # y1 + y0
        if z.is_cuda and dt == torch.bfloat16 and z.shape[1] == 8 and self.conv_out.out_channels == 1:
            return ops.conv_out(z, self.conv_out.weight)              # K3c: 8 -> 1 is streaming work, not a GEMM
        return be.conv3d(z, self._w("conv_out", dt), 1, (1, 1, 1)).float()

    _GEO = {}

    @classmethod
    def _outside_geometry(cls, dims, E_lo, E_hi, B, dev):
        """([3,3] tap-valid mask per edge class, [3,3,3] voxel counts of the 27 border classes outside the box E), built once
        per geometry and device: forward then performs no host-to-device copy (CUDA-graph capturable)."""
        key = (tuple(dims), tuple(E_lo), tuple(E_hi), int(B), str(dev))
        hit = cls._GEO.get(key)
        if hit is None:
            M = torch.tensor([[0., 1., 1.], [1., 1., 1.], [1., 1., 0.]], device=dev)   # [edge class][tap valid]
            full = [torch.tensor([1., n - 2., 1.], device=dev) for n in dims]
            inside = []
            for ax, n in enumerate(dims):
                lo_edge = 1.0 if E_lo[ax] == 0 else 0.0
                hi_edge = 1.0 if E_hi[ax] == n - 1 else 0.0
                inside.append(torch.tensor([lo_edge, (E_hi[ax] - E_lo[ax] + 1) - lo_edge - hi_edge, hi_edge], device=dev))
            cnt = B * (torch.einsum("a,b,c->abc", *full) - torch.einsum("a,b,c->abc", *inside))
            hit = cls._GEO[key] = (M, cnt)
        return hit

    @classmethod
    def _outside_classes(cls, Wf, bg, dims, E_lo, E_hi, B):
        """Values and voxel counts of the 27 border classes of a stride-1, pad-1 conv output outside the box E when its
        input is the per-channel constant `bg` there: ([Cout,3,3,3] values, [3,3,3] counts)."""
        M, cnt = cls._outside_geometry(dims, E_lo, E_hi, B, Wf.device)
        val = torch.einsum("oidhw,ad,bh,cw,i->oabc", Wf, M, M, M, bg)                   # [Cout,3,3,3]
        return val, cnt

    @classmethod
    def _stats_from_sums_with_constant_outside(cls, t1, t2, Wf, bg, dims, E_lo, E_hi, B, n_full):
        """Same statistics as _stats_with_constant_outside, from the per-channel sums (sum T, sum T^2) over E."""
        val, cnt = cls._outside_classes(Wf, bg, dims, E_lo, E_hi, B)
        val, cnt = val.double(), cnt.double()
        n_e = float(B)
        for ax in range(3):
            n_e *= (E_hi[ax] - E_lo[ax] + 1)
        mean = (t1.double() + (val * cnt).sum((1, 2, 3))) / n_full
        inside = t2.double() - 2.0 * mean * t1.double() + n_e * mean * mean
        outside = ((val - mean.view(-1, 1, 1, 1)).pow(2) * cnt).sum((1, 2, 3))
        var = ((inside + outside) / n_full).clamp_min(0)
        return mean.float(), var.float()

    @staticmethod
    def _stats_with_constant_outside(T, Wf, bg, dims, E_lo, E_hi, B, n_full):
        """Batch mean / biased variance over the FULL canvas of a stride-1, pad-1 conv whose input is the
        per-channel constant `bg` everywhere outside the computed box E (T holds the output on E).
        Outside E the output takes one of 27 values per channel (which taps fall off the canvas)."""
        dev = T.device
        M = torch.tensor([[0., 1., 1.], [1., 1., 1.], [1., 1., 0.]], device=dev)       # [edge class][tap valid]
        val = torch.einsum("oidhw,ad,bh,cw,i->oabc", Wf, M, M, M, bg)                   # [Cout,3,3,3]
        full = [torch.tensor([1., n - 2., 1.], device=dev) for n in dims]
        inside = []
        for ax, n in enumerate(dims):
            lo_edge = 1.0 if E_lo[ax] == 0 else 0.0
            hi_edge = 1.0 if E_hi[ax] == n - 1 else 0.0
            inside.append(torch.tensor([lo_edge, (E_hi[ax] - E_lo[ax] + 1) - lo_edge - hi_edge, hi_edge], device=dev))
        cnt = B * (torch.einsum("a,b,c->abc", *full) - torch.einsum("a,b,c->abc", *inside))
        mean = (T.sum((0, 2, 3, 4)) + (val * cnt).sum((1, 2, 3))) / n_full
        dev_out = (val - mean.view(-1, 1, 1, 1)).pow(2) * cnt
        var = ((T - _bview(mean)).pow(2).sum((0, 2, 3, 4)) + dev_out.sum((1, 2, 3))) / n_full
        return mean, var
