"""tcgen05 convolution backend of the regulariser (K3): 3x3x3 convolutions of bf16 channel-last volumes on the implicit-GEMM
kernels of libmvs_b200.so (csrc/conv3d_tc.cu).

  stride 1 (conv_0_0, conv_{1,2,3}_1)      forward and data gradient: conv3d_s1_kdn_kernel (depth tap folded into the MMA N
                                           extent; MVSB200_CONV_S1=taps selects the one-MMA-per-tap kernel); weight gradient:
                                           conv3d_s1_wgrad_tc_kernel
  stride 2 (conv_{1,2,3}_0, stacked)       forward: conv3d_s2_tc_kernel; gradients: library (a tcgen05 strided weight gradient is
                                           opt-in, MVSB200_S2_WGRAD=tcgen05)
  stride-2 transposed (deconv_{3,2,1}_0)   forward: deconv3d_s2_tc_kernel (one launch; MVSB200_DECONV=classes selects one launch
                                           per output-parity class); data gradient: conv3d_s2_tc_kernel; weight gradient: library
Operands the kernels do not take (8- and 1-channel rows, fp32 volumes) go to the cuDNN backend; DESIGN.md §4 lists which
layer runs where.

Reference layers: scripts/model.py:223-234 (Conv3d / ConvTranspose3d factories), :101-121 (their use).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import _lib, conv3d as conv_backends
from .ops import _stream, _timed, wgrad_fork

_CIN_OK = (16, 32, 64)


def _n_rows(c):
    return 16 if c <= 16 else (32 if c <= 32 else 64)


_SMS = {}


def _sm_count(device):
    d = torch.device(device)
    key = d.index if d.index is not None else torch.cuda.current_device()
    if key not in _SMS:
        _SMS[key] = torch.cuda.get_device_properties(key).multi_processor_count
    return _SMS[key]


_NAT = list(range(27))                       # filter taps in their natural (kd, kh, kw) order
_FLIP = [26 - t for t in range(27)]          # ... flipped along all three axes (data gradients)


def _kdn_order(taps):
    """Slots [(kh, kw)][kd] of the kdn kernels from a natural-order tap list."""
    return [taps[kd * 9 + khw] for khw in range(9) for kd in range(3)]


def _pack(w, rows_dim, n_rows, taps, n_cols=None, c0=0, cols_real=None, out=None):
    """The bf16 [slot][row][col] operand of the tensor-core kernels from the layer's parameter w [d0, d1, 3, 3, 3] in ONE launch
    (mvsb200_pack_filter): rows = channel dimension `rows_dim` of w (zero rows up to n_rows), columns = the other one
    (columns c0 .. c0 + cols_real, zero columns up to n_cols), slot s = tap taps[s] (-1: an all-zero slot)."""
    import ctypes
    w = w.detach()
    if w.dtype != torch.float32 or not w.is_contiguous():
        w = w.float().contiguous()
    d0, d1 = w.shape[:2]
    rows_real, sr, sc, cols_all = (d0, 27 * d1, 27, d1) if rows_dim == 0 else (d1, 27, 27 * d1, d0)
    cols_real = cols_all - c0 if cols_real is None else cols_real
    n_cols = cols_real if n_cols is None else n_cols
    if out is None:
        out = torch.empty((len(taps), n_rows, n_cols), dtype=torch.bfloat16, device=w.device)
    _lib.call("mvsb200_pack_filter", w.data_ptr(), out.data_ptr(), len(taps), n_rows, n_cols, min(rows_real, n_rows), cols_real, c0,
              sr, sc, (ctypes.c_int * len(taps))(*taps), _stream())
    return out


def pack_filter(w: torch.Tensor) -> torch.Tensor:
    """[Cout, Cin, 3, 3, 3] -> bf16 [27, n_rows, Cin]: tap-major (kd, kh, kw), output channel (zero rows up to n_rows),
    input channel -- the K-major B operand the kernel keeps resident in shared memory."""
    return _pack(w, 0, _n_rows(w.shape[0]), _NAT)


def pack_filter_dgrad(w: torch.Tensor) -> torch.Tensor:
    """Filter of the data gradient: taps flipped, channel roles swapped ([Cin, Cout] per tap)."""
    return _pack(w, 1, _n_rows(w.shape[1]), _FLIP)


def _supported(cin, cout):
    return cin in _CIN_OK and cout % 8 == 0 and 8 <= cout <= 64


def _S1_FORM():
    """"kdn" (default): conv3d_s1_kdn_kernel, depth tap folded into N; "taps": conv3d_s1_tc_kernel, one MMA per tap
    (MVSB200_CONV_S1 selects; kept for A/B measurements and as the form the parity-class kernels derive from)."""
    import os
    form = os.environ.get("MVSB200_CONV_S1", "kdn")
    return form if form == "taps" or hasattr(_lib.load(), "mvsb200_conv3d_s1_fwd_kdn") else "taps"


def _launch(x_cl, w, role, out_dims, off):
    """Stride-1 convolution of x_cl with the layer weight w [Cout, Cin, 3, 3, 3]: role "fwd" (rows = Cout, contraction over Cin)
    or "dgrad" (x_cl is the output gradient: taps flipped, rows = Cin, contraction over Cout).  An 8-channel volume runs on the
    K = 16 kernel: the packed filter gets 8 zero columns and -- kdn form -- the kernel's TMA box reads the missing channels as
    zeros; the one-MMA-per-tap form needs the widened copy.  Algorithmic FLOPs are counted on the channels that carry data."""
    B, cin, Di, Hi, Wi = x_cl.shape
    Do, Ho, Wo = out_dims
    cout = w.shape[0] if role == "fwd" else w.shape[1]
    n_rows = _n_rows(cout)
    cin_k = max(cin, 16)
    taps = _NAT if role == "fwd" else _FLIP
    rows_dim = 0 if role == "fwd" else 1
    y = torch.empty((B, cout, Do, Ho, Wo), dtype=torch.bfloat16, device=x_cl.device, memory_format=torch.channels_last_3d)
    if _S1_FORM() == "kdn":
        # depth tap folded into the MMA N extent: filter as [(kh,kw)][kd][rows][Cin]
        wk = _pack(w, rows_dim, n_rows, _kdn_order(taps), n_cols=cin_k)
        with _timed("conv3d_s1_tc", 2.0 * 27 * cin * cout * B * Do * Ho * Wo):
            _lib.call("mvsb200_conv3d_s1_fwd_kdn", x_cl.data_ptr(), wk.data_ptr(), y.data_ptr(), B, Di, Hi, Wi, cin, Do, Ho, Wo,
                      cout, cout, n_rows, off, off, off, _stream())
        return y
    wp = _pack(w, rows_dim, n_rows, taps, n_cols=cin_k)
    if cin_k != cin:
        x16 = torch.empty((B, 16, Di, Hi, Wi), dtype=torch.bfloat16, device=x_cl.device, memory_format=torch.channels_last_3d)
        _lib.call("mvsb200_widen_rows_8to16_bf16", x_cl.data_ptr(), x16.data_ptr(), B * Di * Hi * Wi, _stream())
        x_cl = x16
    with _timed("conv3d_s1_tc", 2.0 * 27 * cin * cout * B * Do * Ho * Wo):
        _lib.call("mvsb200_conv3d_s1_fwd", x_cl.data_ptr(), wp.data_ptr(), y.data_ptr(), B, Di, Hi, Wi, cin_k, Do, Ho, Wo,
                  cout, cout, n_rows, off, off, off, _stream())
    return y


class _Conv3dS1(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, pad):
        x_cl = x.detach().contiguous(memory_format=torch.channels_last_3d)
        D, H, W = x.shape[2:]
        out_dims = (D, H, W) if pad == 1 else (D - 2, H - 2, W - 2)
        y = _launch(x_cl, w, "fwd", out_dims, -pad)
        ctx.save_for_backward(x_cl, w)
        ctx.pad = pad
        return y

    @staticmethod
    def backward(ctx, gy):
        x_cl, w = ctx.saved_tensors
        gy = gy.to(torch.bfloat16).contiguous(memory_format=torch.channels_last_3d)
        gx = _s1_dgrad(gy, w, ctx.pad, x_cl.shape) if ctx.needs_input_grad[0] else None
        gw = None
        if ctx.needs_input_grad[1]:
            with wgrad_fork(w, (x_cl, gy)) as f:
                f.result = _s1_wgrad(x_cl, gy, w, ctx.pad)
            gw = f.grad()
        return gx, gw, None


def _s1_dgrad(gy, w, pad, x_shape):
    """Data gradient of a stride-1 convolution: the same convolution of the output gradient with the flipped, transposed
    filter (gy: bf16 channel-last)."""
    cout, cin = w.shape[:2]
    off = -1 if pad == 1 else -2
    if _supported(cout, cin) or (cout == 8 and _supported(16, cin)):
        # roles swap: the gradient volume has Cout channels, the result Cin
        return _launch(gy, w, "dgrad", tuple(x_shape[2:]), off)
    return torch.nn.grad.conv3d_input(x_shape, w.to(gy.dtype), gy, padding=pad)


def _s1_wgrad(x_cl, gy, w, pad):
    """Weight gradient of a stride-1 convolution on conv3d_s1_wgrad_tc_kernel (x_cl, gy: bf16 channel-last)."""
    cout, cin = w.shape[:2]
    if cin in _CIN_OK and cout in (8, 16, 32, 64):
        B, _, Di, Hi, Wi = x_cl.shape
        Do, Ho, Wo = gy.shape[2:]
        gw27 = torch.empty((27, cin, cout), dtype=torch.float32, device=gy.device)
        with _timed("conv3d_s1_wgrad_tc", 2.0 * 27 * cin * cout * B * Do * Ho * Wo):
            _lib.call("mvsb200_conv3d_s1_wgrad", x_cl.data_ptr(), gy.data_ptr(), gw27.data_ptr(), B, Di, Hi, Wi, cin,
                      Do, Ho, Wo, cout, -pad, -pad, -pad, _stream())
        return gw27.reshape(3, 3, 3, cin, cout).permute(4, 3, 0, 1, 2).to(w.dtype)
    return torch.nn.grad.conv3d_weight(x_cl, w.shape, gy, padding=pad).to(w.dtype)


# ---- stride-2 transposed convolution as 8 output-parity classes of the stride-1 kernel -------------------------------
_CLASS_IDX = {}


def _deconv_class_tables(pads, device):
    """For ConvTranspose3d(k=3, stride=2, padding=pads): per output-parity class (pd,ph,pw) the tap mask of the
    stride-1 kernel and, per kernel tap t, the index of the original filter tap k it carries (27 = none).
    out[2j + par] = sum_{k: (par+p-k) even} W[k] . in[j + (par+p-k)/2]; with the kernel's off = -1 the tap is
    t = (par+p-k)/2 + 1 per axis."""
    key = (tuple(pads), str(device))
    hit = _CLASS_IDX.get(key)
    if hit is not None:
        return hit
    per_axis = []
    for p in pads:
        per_axis.append({par: [(k, (par + p - k) // 2 + 1) for k in range(3) if (par + p - k) % 2 == 0] for par in (0, 1)})
    idx = torch.full((8, 27), 27, dtype=torch.long)
    masks = []
    for c in range(8):
        par = (c >> 2 & 1, c >> 1 & 1, c & 1)
        mask = 0
        for kd, td in per_axis[0][par[0]]:
            for kh, th in per_axis[1][par[1]]:
                for kw, tw in per_axis[2][par[2]]:
                    if not (0 <= td < 3 and 0 <= th < 3 and 0 <= tw < 3):
                        raise ValueError(f"transposed-conv padding {pads} is outside the 3-tap window of the kernel")
                    t = (td * 3 + th) * 3 + tw
                    idx[c, t] = (kd * 3 + kh) * 3 + kw
                    mask |= 1 << t
        masks.append(mask)
    hit = (idx.to(device), masks)
    _CLASS_IDX[key] = hit
    return hit


def conv_transpose3d_s2(x, w, pads, out_dims, stats_out=None):
    """ConvTranspose3d(k=3, stride=2, padding=pads, bias=False) from the box volume x [B,Cin,md,mh,mw] to the first
    `out_dims` voxels per axis of its output, on the tcgen05 kernels.  One launch (deconv3d_s2_tc_kernel: the 8
    output-parity classes side by side in TMEM, every canvas line written once); MVSB200_DECONV=classes selects the
    earlier form, one launch of the stride-1 kernel per class.  w: [Cin, Cout, 3, 3, 3] (model.py:229-234)."""
    import ctypes
    import os
    x_cl = x.detach().contiguous(memory_format=torch.channels_last_3d)
    B, cin, md, mh, mw = x_cl.shape
    cout = w.shape[1]
    D, h, wd = out_dims
    n_rows = _n_rows(cout)
    y = torch.empty((B, cout, D, h, wd), dtype=torch.bfloat16, device=x.device, memory_format=torch.channels_last_3d)
    sB, sD, sH, sW = y.stride(0), y.stride(2), y.stride(3), y.stride(4)
    _, masks = _deconv_class_tables(pads, x.device)
    work = 0.0
    for c in range(8):
        pd_, ph_, pw_ = c >> 2 & 1, c >> 1 & 1, c & 1
        Jd, Jh, Jw = (D - pd_ + 1) // 2, (h - ph_ + 1) // 2, (wd - pw_ + 1) // 2
        if min(Jd, Jh, Jw) > 0:
            work += 2.0 * bin(masks[c]).count("1") * cin * cout * B * Jd * Jh * Jw
    if os.environ.get("MVSB200_DECONV", "fused") == "kc" and cin in (16, 32, 64):      # A/B: the K-chunk kernel with one chunk
        return conv_transpose3d_s2_kc(x_cl, (cin,), w, pads, out_dims)
    if n_rows <= 32 and os.environ.get("MVSB200_DECONV", "fused") != "classes" and hasattr(_lib.load(), "mvsb200_deconv3d_s2_fwd"):
        wp = _pack(w, 1, n_rows, _NAT + [-1])            # [k][co][ci] from [Cin, Cout, ...]; slot 27: zeros (DeconvWide, tc_common.cuh)
        ys = (ctypes.c_int64 * 4)(sB, sD, sH, sW)
        if stats_out is not None and hasattr(_lib.load(), "mvsb200_deconv3d_s2_fwd_stats"):
            # per-CTA sums of the stored values / their squares per channel, from the kernel's epilogue: the BatchNorm that follows
            # finalizes them (ops.batchnorm_relu_train(partials=...)) instead of reading the canvas again
            partials = torch.empty((_sm_count(x.device), 2, cout), dtype=torch.float32, device=x.device)
            nb = ctypes.c_int(0)
            with _timed("deconv3d_s2_tc", work):
                _lib.call("mvsb200_deconv3d_s2_fwd_stats", x_cl.data_ptr(), wp.data_ptr(), y.data_ptr(), B, md, mh, mw, cin, D, h, wd,
                          cout, n_rows, int(pads[0]), int(pads[1]), int(pads[2]), ys, partials.data_ptr(), ctypes.byref(nb), _stream())
            stats_out.append((partials, int(nb.value), (D, h, wd)))
            return y
        with _timed("deconv3d_s2_tc", work):
            _lib.call("mvsb200_deconv3d_s2_fwd", x_cl.data_ptr(), wp.data_ptr(), y.data_ptr(), B, md, mh, mw, cin, D, h, wd, cout,
                      n_rows, int(pads[0]), int(pads[1]), int(pads[2]), ys, _stream())
        return y
    idx, masks = _deconv_class_tables(pads, x.device)
    wk = w.detach().permute(2, 3, 4, 1, 0).reshape(27, cout, cin)                 # [k][co][ci]
    wz = torch.cat([wk, wk.new_zeros(1, cout, cin)], 0)
    wp = torch.zeros(8, 27, n_rows, cin, dtype=torch.bfloat16, device=x.device)
    wp[:, :, :cout] = wz[idx].to(torch.bfloat16)
    ys = (ctypes.c_int64 * 4)(sB, 2 * sD, 2 * sH, 2 * sW)
    with _timed("conv3d_s1_tc", work):
        for c in range(8):
            pd_, ph_, pw_ = c >> 2 & 1, c >> 1 & 1, c & 1
            Jd, Jh, Jw = (D - pd_ + 1) // 2, (h - ph_ + 1) // 2, (wd - pw_ + 1) // 2
            if min(Jd, Jh, Jw) <= 0:
                continue
            base = y.data_ptr() + 2 * (pd_ * sD + ph_ * sH + pw_ * sW)
            _lib.call("mvsb200_conv3d_s1_fwd_ex", x_cl.data_ptr(), wp[c].data_ptr(), base, B, md, mh, mw, cin, Jd, Jh, Jw, cout,
                      n_rows, -1, -1, -1, masks[c], ys, _stream())
    return y


def _lines_fit(cb, cs, ws):
    """Two ring stages of the line kernel (a line of the dense operand + three lines of the strided one, csrc/conv3d_s2_bwd.cu:
    launch_s2_wgrad_lines) must fit shared memory; very long lines of wide layers go to the parity-class kernel instead."""
    up = lambda v: (v + 1023) // 1024 * 1024
    ksteps = (ws + 15) // 16
    atoms = 128 // (2 * cb)
    line_a = up(max(ws + 1, 16 * ksteps + atoms) * 4 * cb)
    n_chunks, chunk = (2, 64) if cs > 64 else (1, cs)
    stage = n_chunks * up(16 * ksteps * 2 * chunk) + 3 * line_a
    return 2 * stage <= 227 * 1024 - 1024 - 8192 - 512


def _s2_wgrad_mode(big_shape, small_shape):
    """Which kernel computes the weight gradient of a stride-2 layer: "lines" (default; conv3d_s2_wgrad_lines_kernel, one
    launch, lines of the strided operand as voxel-pair rows), "classes" (the stride-1 weight-gradient kernel on the 8 parity
    sub-lattices, one launch per class and channel chunk -- slower than the library at the regulariser's shapes, kept for A/B
    and for the shapes the line kernel does not take) or "cudnn" (the library).  MVSB200_S2_WGRAD=lines|tcgen05|cudnn selects;
    "tcgen05" is the historical name of the parity-class form."""
    import os
    want = os.environ.get("MVSB200_S2_WGRAD", "lines")
    cb, cs = big_shape[1], small_shape[1]
    lib = _lib.load()
    lines_ok = (cb in (8, 16, 32) and (cs in (16, 32, 64) or (64 < cs <= 128 and cs % 16 == 0)) and big_shape[4] % 2 == 0
                and small_shape[4] <= 255 and _lines_fit(cb, cs, small_shape[4]) and hasattr(lib, "mvsb200_conv3d_s2_wgrad_lines"))
    classes_ok = cb in _CIN_OK and cs % 8 == 0 and hasattr(lib, "mvsb200_conv3d_s2_wgrad")
    if want == "lines" and lines_ok:
        return "lines"
    if want in ("lines", "tcgen05", "classes") and classes_ok:
        return "classes"
    return "cudnn"


def s2_wgrad(big, small, pads, mode="classes"):
    """gw[k][cb][cs] = sum_o big(2o - pad + k)[cb] * small(o)[cs] on the tcgen05 weight-gradient kernels -> fp32 [27, Cb, Cs].
    big: bf16 channels_last_3d [B,C,D,h,w].  small: bf16, channel-last voxel rows; mode "lines" (one launch,
    csrc/conv3d_s2_bwd.cu) also takes a box VIEW of a larger channel-last allocation (its strides go into the TMA map), mode
    "classes" (parity sub-lattices of `big` through doubled-stride TMA maps, csrc/conv3d_tc.cu) needs it dense."""
    import ctypes
    B, cb, Db, Hb, Wb = big.shape
    _, cs, Ds, Hs, Ws = small.shape
    gw = torch.empty((27, cb, cs), dtype=torch.float32, device=big.device)
    # algorithmic work: every tap once over the small volume
    with _timed("conv3d_s2_wgrad_tc", 2.0 * 27 * cb * cs * B * Ds * Hs * Ws):
        if mode == "lines":
            ss = None
            if small.stride(1) != 1 or any(st % 8 for st in (small.stride(0), small.stride(2), small.stride(3), small.stride(4))):
                small = small.contiguous(memory_format=torch.channels_last_3d)
            if not small.is_contiguous(memory_format=torch.channels_last_3d):
                ss = (ctypes.c_int64 * 4)(small.stride(0), small.stride(2), small.stride(3), small.stride(4))
            _lib.call("mvsb200_conv3d_s2_wgrad_lines", big.data_ptr(), small.data_ptr(), gw.data_ptr(), B, Db, Hb, Wb, cb, Ds, Hs, Ws,
                      cs, int(pads[0]), int(pads[1]), int(pads[2]), ss, _stream())
        else:
            small = small.contiguous(memory_format=torch.channels_last_3d)
            _lib.call("mvsb200_conv3d_s2_wgrad", big.data_ptr(), small.data_ptr(), gw.data_ptr(), B, Db, Hb, Wb, cb, Ds, Hs, Ws, cs,
                      int(pads[0]), int(pads[1]), int(pads[2]), _stream())
    return gw


class _ConvTranspose3dS2(torch.autograd.Function):
    """Forward on the one-launch tcgen05 kernel; the data gradient is a stride-2 convolution of the output gradient
    (conv3d_s2_tc_kernel), the weight gradient goes to the library (or, opt-in, to the tcgen05 strided kernel)."""

    @staticmethod
    def forward(ctx, x, w, pads, out_dims, stats_out=None):
        y = conv_transpose3d_s2(x, w, pads, out_dims, stats_out)
        ctx.save_for_backward(x.detach().contiguous(memory_format=torch.channels_last_3d), w)
        ctx.pads = tuple(pads)
        return y

    @staticmethod
    def backward(ctx, gy):
        x_cl, w = ctx.saved_tensors
        pads = ctx.pads
        gy = gy.to(torch.bfloat16).contiguous(memory_format=torch.channels_last_3d)
        gx = gw = None
        # As a convolution gy -> x: x[i] = sum_k W[k]^T gy[2i - p + k].  With padding p + 2 the library's output index is
        # i + 1 and its range covers every box row (the plain padding p stops one row short of the box).
        P2 = tuple(p + 2 for p in pads)
        m = list(x_cl.shape[2:])
        n_o = [(n + 2 * q - 3) // 2 + 1 for n, q in zip(gy.shape[2:], P2)]
        if any(1 + a > b for a, b in zip(m, n_o)):
            raise _lib.MvsB200Error(f"transposed-conv gradient: box {m} does not fit the strided window {n_o}")
        inner = (slice(None), slice(None)) + tuple(slice(1, 1 + a) for a in m)
        if ctx.needs_input_grad[0]:
            cin_t, cout_t = w.shape[:2]
            if (cout_t in _CIN_OK or (cout_t == 8 and cin_t <= 32)) and cin_t % 8 == 0:
                # x[i] = sum_k W[k]^T gy[2i - p + k]: the tcgen05 stride-2 kernel with the filter read as out = Cin, in = Cout.
                # 8-channel gradient rows (deconv_1_0) reach the K = 16 MMA through TMA's out-of-bounds zero fill: the filter
                # gets 8 zero input channels, the volume is read as it is
                B = gy.shape[0]
                n_rows = (cin_t + 15) // 16 * 16
                gx = torch.empty(x_cl.shape, dtype=torch.bfloat16, device=gy.device, memory_format=torch.channels_last_3d)
                wpk = _pack(w, 0, n_rows, _NAT, n_cols=max(cout_t, 16))
                with _timed("conv3d_s2_tc", 2.0 * 27 * cin_t * cout_t * x_cl.numel() / cin_t):
                    _lib.call("mvsb200_conv3d_s2_fwd", gy.data_ptr(), wpk.data_ptr(), gx.data_ptr(), B,
                              gy.shape[2], gy.shape[3], gy.shape[4], cout_t, m[0], m[1], m[2], cin_t, cin_t, n_rows,
                              pads[0], pads[1], pads[2], _stream())
            else:
                gx = F.conv3d(gy, w.detach().to(torch.bfloat16), None, 2, P2)[inner]   # weight [Cin, Cout, ...] read as out = Cin, in = Cout
        if ctx.needs_input_grad[1]:
            cin_t, cout_t = w.shape[:2]
            mode = _s2_wgrad_mode(gy.shape, x_cl.shape)
            if mode != "cudnn":
                # gW[ci][co][k] = sum_j x[j][ci] gy[2j - p + k][co]: the strided operand is the output gradient
                with wgrad_fork(w, (gy, x_cl)) as f:
                    g27 = s2_wgrad(gy, x_cl, pads, mode)                                 # [27, Cout, Cin]
                    f.result = g27.reshape(3, 3, 3, cout_t, cin_t).permute(4, 3, 0, 1, 2).to(w.dtype)
                gw = f.grad()
            else:
                xs = torch.zeros((x_cl.shape[0], x_cl.shape[1]) + tuple(n_o), dtype=x_cl.dtype, device=x_cl.device,
                                 ).contiguous(memory_format=torch.channels_last_3d)
                xs[inner] = x_cl
                gw = torch.nn.grad.conv3d_weight(gy, w.shape, xs, stride=2, padding=P2).to(w.dtype)
        return gx, gw, None, None, None


# ---- stride-2 convolution on the central box (the stacked branches conv_{1,2,3}_0) ----------------------------------
def pack_filter_rows(w: torch.Tensor, n_rows: int) -> torch.Tensor:
    return _pack(w, 0, n_rows, _NAT)


def _kc_chunks(widths):
    """K chunks of the multi-chunk transposed convolution for input channels grouped as `widths`: each group must be a
    swizzle span (16 / 32 / 64 channels), at most three of them."""
    if widths is None or len(widths) > 3 or any(n not in (16, 32, 64) for n in widths):
        return None
    offs, c0 = [], 0
    for n in widths:
        offs.append(c0)
        c0 += n
    return offs, list(widths)


def _s2_dgrad_own(cin, widths):
    """The data gradient of a stride-2 convolution runs on deconv3d_s2_kc_kernel when its output channels come as up to three
    groups of 16 / 32 / 64 (the stacked branches: 16 + 32 + 64) and its input has 16 / 32 / 64 channels;
    MVSB200_S2_DGRAD=cudnn sends it to the library."""
    import os
    return (os.environ.get("MVSB200_S2_DGRAD", "tcgen05") != "cudnn" and _kc_chunks(widths) is not None and cin in (16, 32, 64)
            and hasattr(_lib.load(), "mvsb200_deconv3d_s2_kc_fwd"))


def conv_transpose3d_s2_kc(x, widths, w_t, pads, out_dims, out=None, accumulate=False):
    """Stride-2 transposed convolution from the channel-stacked box volume x [B, sum(widths), md, mh, mw] (bf16, dense
    channel-last) to the canvas `out_dims`:  out[2J + par] = sum_k W[k] . x[J + (par + pad - k)/2], W[k] = w_t[:, :, k] with
    w_t: [Cin_total, Cout, 3, 3, 3] (the ConvTranspose3d layout).  One launch per 16 output channels
    (deconv3d_s2_kc_kernel).  `out`: canvas to write (dense channel-last, Cout channels); accumulate=True adds to it."""
    import ctypes
    offs, ns = _kc_chunks(widths)
    B, ctot, md, mh, mw = x.shape
    cout = w_t.shape[1]
    n_rows = (cout + 15) // 16 * 16
    D, h, wd = out_dims
    if out is None:
        out = torch.empty((B, cout, D, h, wd), dtype=torch.bfloat16, device=x.device, memory_format=torch.channels_last_3d)
        accumulate = False
    # per chunk [28][n_rows][n]: [k][co][ci] from w_t [Cin_total, Cout, ...], slot 27 = zeros (filter slots of classes a shift
    # does not serve), the chunks one after the other
    wpk = torch.empty(28 * n_rows * ctot, dtype=torch.bfloat16, device=x.device)
    pos = 0
    for o, n in zip(offs, ns):
        _pack(w_t, 1, n_rows, _NAT + [-1], c0=o, cols_real=n, out=wpk[pos:pos + 28 * n_rows * n])
        pos += 28 * n_rows * n
    ys = (ctypes.c_int64 * 4)(out.stride(0), out.stride(2), out.stride(3), out.stride(4))
    kc_off = (ctypes.c_int * 3)(*(offs + [0] * (3 - len(offs))))
    kc_n = (ctypes.c_int * 3)(*(ns + [0] * (3 - len(ns))))
    with _timed("deconv3d_s2_tc", 2.0 * 27 * ctot * cout * B * md * mh * mw):
        _lib.call("mvsb200_deconv3d_s2_kc_fwd", x.data_ptr(), ctot, wpk.data_ptr(), kc_off, kc_n, len(ns), out.data_ptr(), B, md, mh, mw,
                  D, h, wd, cout, n_rows, int(pads[0]), int(pads[1]), int(pads[2]), ys, 1 if accumulate else 0, _stream())
    return out


def _s2box_forward(x_cl, w, pads, out_dims, splits, holder):
    """Forward of the stride-2 box convolution on conv3d_s2_tc_kernel; fixes the geometry of `holder` (ops.BoxGradDest), the
    buffer the branches' gradients are collected in."""
    B, cin, Dx, Hx, Wx = x_cl.shape
    cout = w.shape[0]
    n_rows = (cout + 15) // 16 * 16
    Do, Ho, Wo = out_dims
    y = torch.empty((B, cout, Do, Ho, Wo), dtype=torch.bfloat16, device=x_cl.device, memory_format=torch.channels_last_3d)
    import os
    # train path with split outputs (the stacked branches): per-channel sums of the outputs from the kernels' epilogues -- the
    # box BatchNorm that follows reads them instead of making a statistics pass (MVSB200_S2_STATS=0: off)
    sums = None
    if holder is not None and splits is not None and cin == 32 and os.environ.get("MVSB200_S2_STATS", "1") != "0":
        sums = torch.empty((2, cout), dtype=torch.float32, device=x_cl.device)
        ws = torch.empty(_sm_count(x_cl.device) * 2 * cout, dtype=torch.float32, device=x_cl.device)
    with _timed("conv3d_s2_tc", 2.0 * 27 * cin * cout * B * Do * Ho * Wo):
        if sums is not None:
            _lib.call("mvsb200_conv3d_s2_fwd_stats", x_cl.data_ptr(), pack_filter_rows(w, n_rows).data_ptr(), y.data_ptr(), B, Dx, Hx,
                      Wx, cin, Do, Ho, Wo, cout, cout, n_rows, pads[0], pads[1], pads[2], ws.data_ptr(), sums.data_ptr(), _stream())
        else:
            _lib.call("mvsb200_conv3d_s2_fwd", x_cl.data_ptr(), pack_filter_rows(w, n_rows).data_ptr(), y.data_ptr(), B, Dx, Hx, Wx,
                      cin, Do, Ho, Wo, cout, cout, n_rows, pads[0], pads[1], pads[2], _stream())
    if holder is not None:
        # where the branches' gradients are collected: the dense box when both gradients run on this library's kernels,
        # else the padded buffer of the library's strided backward
        widths = splits if splits is not None else (cout,)
        own = _s2_dgrad_own(cin, widths) and _s2_wgrad_mode(x_cl.shape, (B, cout) + tuple(out_dims)) == "lines"
        if own:
            holder.__init__((B, cout) + tuple(out_dims), tuple(slice(0, n) for n in out_dims), splits, x_cl.device, zero=False)
        else:
            _, nat, box = _Conv3dS2Box._geometry(x_cl.shape, pads, out_dims)
            holder.__init__((B, cout) + nat, box, splits, x_cl.device)
        holder.sums = sums
    if splits is None:
        return y
    return tuple(torch.split(y, list(splits), 1))


class _Conv3dS2Box(torch.autograd.Function):
    """out(o) = sum_k W[k] x(2o - pad + k) for o in a box of `out_dims` voxels (zero outside x).  Forward on the tcgen05
    stride-2 kernel.  `splits`: the output channels are returned as that many separate tensors (the stacked branches
    conv_{1,2,3}_0); the fused box BatchNorm backward of each branch writes its gradient straight into its channel slice of
    ONE channel-stacked, channel-last box buffer (ops.BoxGradDest) -- no concatenation or layout copies of the 112-channel
    gradient -- which both gradient kernels read: the data gradient is a stride-2 transposed convolution over K chunks
    (deconv3d_s2_kc_kernel), the weight gradient the line kernel (conv3d_s2_wgrad_lines_kernel).  MVSB200_S2_DGRAD=cudnn /
    MVSB200_S2_WGRAD=cudnn send either to the library, which wants the gradient of its padded output instead."""

    @staticmethod
    def _geometry(x_shape, pads, out_dims):
        """The same convolution as the library sees it: symmetric padding P = pad (+2 if pad < 2: keeps parity), natural output
        extent `nat`, our box at offset (P - pad)/2 inside it."""
        P = tuple(q if q >= 2 else q + 2 for q in pads)
        off = tuple((a - b) // 2 for a, b in zip(P, pads))
        nat = tuple((n + 2 * a - 3) // 2 + 1 for n, a in zip(x_shape[2:], P))
        return P, nat, tuple(slice(o, o + n) for o, n in zip(off, out_dims))

    @staticmethod
    def forward(ctx, x, w, pads, out_dims, splits, holder=None):
        x_cl = x.detach().contiguous(memory_format=torch.channels_last_3d)
        outs = _s2box_forward(x_cl, w, pads, out_dims, splits, holder)
        ctx.save_for_backward(x_cl, w)
        ctx.pads, ctx.out_dims, ctx.splits, ctx.holder = tuple(pads), tuple(out_dims), splits, holder
        return outs

    @staticmethod
    def backward(ctx, *gys):
        x_cl, w = ctx.saved_tensors
        gx, gw = _s2box_backward(x_cl, w, ctx.pads, ctx.out_dims, ctx.splits, ctx.holder, gys, bool(ctx.needs_input_grad[0]),
                                 bool(ctx.needs_input_grad[1]))
        return gx, gw, None, None, None, None


def _s2box_backward(x_cl, w, pads, out_dims, splits, holder, gys, need_x, need_w, acc_into=None):
    """Gradients of the stride-2 box convolution (see _Conv3dS2Box).  acc_into: a canvas that already holds another
    contribution to the input gradient -- the data gradient is ADDED to it (in the epilogue of the transposed-convolution
    kernel) and it is returned."""
    B, cin = x_cl.shape[:2]
    cout = w.shape[0]
    out_dims = tuple(out_dims)
    widths = tuple(splits) if splits is not None else (cout,)
    P, nat, box = _Conv3dS2Box._geometry(x_cl.shape, pads, out_dims)
    wg_mode = _s2_wgrad_mode(x_cl.shape, (B, cout) + out_dims)
    own_dgrad = need_x and _s2_dgrad_own(cin, widths)
    own_wgrad = need_w and wg_mode != "cudnn"
    lib_mask = [need_x and not own_dgrad, need_w and not own_wgrad, False]
    holder = holder if holder is not None and holder.buffer is not None else None

    def assemble(shape, where):
        """The channel-stacked gradient in a buffer of `shape` with the box at `where`: the holder's buffer when it has
        this geometry (slices the fused BatchNorm backward wrote are already in place), else a fresh one + copies."""
        h = holder if holder is not None and holder.shape == shape else None
        full = shape[2:] == out_dims
        buf = h.buffer if h is not None else torch.empty(shape, dtype=torch.bfloat16, device=x_cl.device,
                                                         memory_format=torch.channels_last_3d)
        if h is None and not full:
            buf.zero_()
        c0 = 0
        for k, (g, n) in enumerate(zip(gys, widths)):
            if h is not None and h.holds(k, g):
                pass                                     # already in place
            elif g is not None:
                buf[(slice(None), slice(c0, c0 + n)) + where] = g
            elif h is not None or full:
                buf[(slice(None), slice(c0, c0 + n)) + where] = 0     # no gradient for this branch / a stale slice
            c0 += n
        return buf

    gx = gw = None
    gy_box = None
    if lib_mask[0] or lib_mask[1]:
        g_full = assemble((B, cout) + nat, box)
        gx, gw, _ = torch.ops.aten.convolution_backward(g_full, x_cl, w.detach().to(torch.bfloat16), None, [2, 2, 2], list(P),
                                                        [1, 1, 1], False, [0, 0, 0], 1, lib_mask)
        gy_box = g_full[(slice(None), slice(None)) + box]
        if gx is not None and acc_into is not None:
            gx = acc_into.add_(gx)
    if own_dgrad or own_wgrad:
        if gy_box is None:
            gy_box = assemble((B, cout) + out_dims, tuple(slice(0, n) for n in out_dims))
        if own_dgrad:
            # gx[2J + par] = sum_k W[k]^T gy[J + (par + pad - k)/2]: the forward weight [Cout, Cin, ...] IS the
            # ConvTranspose3d layout [in = Cout, out = Cin, ...] of that transposed convolution
            gx = conv_transpose3d_s2_kc(gy_box.contiguous(memory_format=torch.channels_last_3d), widths, w, pads,
                                        tuple(x_cl.shape[2:]), out=acc_into, accumulate=acc_into is not None)
        if own_wgrad:                    # after the data gradient: a forked weight gradient overlaps what follows it
            # gW[co][ci][k] = sum_o x[2o - pad + k][ci] gy[o][co]: the strided operand is the layer's input
            with wgrad_fork(w, (x_cl, gy_box)) as f:
                g27 = s2_wgrad(x_cl, gy_box, pads, wg_mode)                        # [27, Cin, Cout]; gy_box may be a view
                f.result = g27.reshape(3, 3, 3, cin, cout).permute(4, 3, 0, 1, 2).to(w.dtype)
            gw = f.grad()
    return gx, (gw.to(w.dtype) if gw is not None else None)


class _EntryConvs(torch.autograd.Function):
    """The four convolutions that read the cost volume (scripts/model.py:101-110) as ONE autograd node: conv_0_0 (stride 1,
    dense) and the stacked stride-2 branches conv_{1,2,3}_0 on the central box.  Forward = the two kernels of _Conv3dS1 and
    _Conv3dS2Box.  Backward: the cost volume's gradient is the sum of two data gradients; as separate nodes autograd adds
    them with an elementwise pass over two 1 GB canvases -- here the transposed-convolution kernel of the branches accumulates
    into the canvas conv_0_0's data gradient was written to."""

    @staticmethod
    def forward(ctx, x, w00, w_cat, pads, out_dims, splits, holder):
        x_cl = x.detach().contiguous(memory_format=torch.channels_last_3d)
        y0 = _launch(x_cl, w00, "fwd", tuple(x_cl.shape[2:]), -1)
        outs = _s2box_forward(x_cl, w_cat, pads, out_dims, splits, holder)
        ctx.save_for_backward(x_cl, w00, w_cat)
        ctx.pads, ctx.out_dims, ctx.splits, ctx.holder = tuple(pads), tuple(out_dims), splits, holder
        return (y0,) + tuple(outs)

    @staticmethod
    def backward(ctx, gy0, *gys):
        x_cl, w00, w_cat = ctx.saved_tensors
        need_x = bool(ctx.needs_input_grad[0])
        gx = gw00 = None
        if gy0 is not None:
            gy0 = gy0.to(torch.bfloat16).contiguous(memory_format=torch.channels_last_3d)
            gx = _s1_dgrad(gy0, w00, 1, x_cl.shape) if need_x else None
            if ctx.needs_input_grad[1]:
                with wgrad_fork(w00, (x_cl, gy0)) as f:
                    f.result = _s1_wgrad(x_cl, gy0, w00, 1)
                gw00 = f.grad()
        acc = gx if gx is not None and gx.is_contiguous(memory_format=torch.channels_last_3d) and gx.dtype == torch.bfloat16 else None
        g2, gw_cat = _s2box_backward(x_cl, w_cat, ctx.pads, ctx.out_dims, ctx.splits, ctx.holder, gys, need_x,
                                     bool(ctx.needs_input_grad[2]), acc_into=acc)
        if need_x:
            gx = g2 if (acc is not None or gx is None) else gx + g2
        return gx, gw00, gw_cat, None, None, None, None


def _attach_box_sums(holder, outs, splits):
    """Hand every branch its slice of the epilogue statistics of the stacked convolution (read by regulariser.py ->
    ops.box_batchnorm_relu)."""
    sums = getattr(holder, "sums", None)
    if sums is None or splits is None:
        return
    c0 = 0
    for o, n in zip(outs, splits):
        o._mvs_box_sums = (sums[0, c0:c0 + n], sums[1, c0:c0 + n])
        c0 += n


class Tcgen05ConvBackend:
    name = "tcgen05"
    fp32_weights = True      # takes the layers' fp32 parameters as they are: the filter-packing kernel does the bf16 rounding

    @staticmethod
    def conv3d_s2_box(x, w, pads, out_dims, splits=None):
        """Stride-2 convolution evaluated on a box: out(o) = sum_k W[k] x(2o - pad + k), o in [0, out_dims).  With `splits`
        (channel counts) the result is a tuple of tensors, one per group of output channels."""
        if (x.is_cuda and x.dtype == torch.bfloat16 and x.shape[1] in _CIN_OK and w.shape[0] % 8 == 0 and w.shape[0] <= 128
                and all(q in (1, 2) for q in pads) and min(x.shape[3:]) >= 2):
            from .ops import BoxGradDest
            holder = None
            if splits is not None and (x.requires_grad or w.requires_grad):
                holder = BoxGradDest.__new__(BoxGradDest)     # filled in by the forward (it knows the padded geometry)
                holder.buffer = None
            outs = _Conv3dS2Box.apply(x, w, tuple(int(q) for q in pads), tuple(int(n) for n in out_dims),
                                      None if splits is None else tuple(int(n) for n in splits), holder)
            if holder is not None:
                _attach_box_sums(holder, outs, splits)
                for k, o in enumerate(outs):
                    o._mvs_grad_dest = (holder, k)           # read by regulariser.py -> ops.box_batchnorm_relu
            return outs
        return None

    @staticmethod
    def entry_convs(x, w00, w_cat, pads, out_dims, splits):
        """conv_0_0 (stride 1, padding 1) and the stacked stride-2 branches on their box, from the same volume, as one
        autograd node (_EntryConvs): returns (y0, (S_1, S_2, S_3)) or None when the operands are not the kernels'."""
        if not (x.is_cuda and x.dtype == torch.bfloat16 and x.shape[1] in _CIN_OK and _supported(x.shape[1], w00.shape[0])
                and min(x.shape[2:]) >= 3 and w_cat.shape[0] % 8 == 0 and w_cat.shape[0] <= 128 and all(q in (1, 2) for q in pads)
                and splits is not None):
            return None
        from .ops import BoxGradDest
        holder = None
        if x.requires_grad or w_cat.requires_grad:
            holder = BoxGradDest.__new__(BoxGradDest)
            holder.buffer = None
        outs = _EntryConvs.apply(x, w00, w_cat, tuple(int(q) for q in pads), tuple(int(n) for n in out_dims),
                                 tuple(int(n) for n in splits), holder)
        if holder is not None:
            _attach_box_sums(holder, outs[1:], splits)
            for k, o in enumerate(outs[1:]):
                o._mvs_grad_dest = (holder, k)
        return outs[0], tuple(outs[1:])

    @staticmethod
    def conv3d(x, w, stride, padding):
        pad = tuple(padding) if isinstance(padding, (tuple, list)) else (padding,) * 3
        if x.is_cuda and not w.is_cuda:
            raise _lib.MvsB200Error("convolution weights live on the CPU while the volume is on the GPU; mvs_b200 has no CPU path")
        if (stride == 1 and x.is_cuda and x.dtype == torch.bfloat16 and pad in ((0, 0, 0), (1, 1, 1))
                and _supported(x.shape[1], w.shape[0]) and min(x.shape[2:]) >= 3):
            return _Conv3dS1.apply(x, w, pad[0])
        return conv_backends.TorchConvBackend.conv3d(x, w if w.dtype == x.dtype else w.to(x.dtype), stride, padding)

    @staticmethod
    def conv_transpose3d_alloc(x, w, stride, padding, out_dims):
        if (stride == 2 and x.is_cuda and x.dtype == torch.bfloat16 and x.shape[1] in _CIN_OK and w.shape[1] % 8 == 0
                and 8 <= w.shape[1] <= 64 and all(p in (1, 2) for p in padding)):
            import os
            # MVSB200_DECONV_STATS=0: no epilogue statistics (the BatchNorm that follows then reads the canvas for them, as the
            # depth-slab path does with its all-reduced sums)
            stats = [] if os.environ.get("MVSB200_DECONV_STATS", "1") != "0" else None
            y = _ConvTranspose3dS2.apply(x, w, tuple(int(p) for p in padding), tuple(int(n) for n in out_dims), stats)
            if stats:
                y._mvs_bn_partials = stats[0]            # read by regulariser._bn_dense -> ops.batchnorm_relu_train
            return y
        return conv_backends.TorchConvBackend.conv_transpose3d_alloc(x, w if w.dtype == x.dtype else w.to(x.dtype), stride, padding, out_dims)

    @classmethod
    def conv_transpose3d(cls, x, w, stride, padding, out_dims):
        D, h, w_ = out_dims
        return cls.conv_transpose3d_alloc(x, w, stride, padding, out_dims)[..., :D, :h, :w_]


def available() -> bool:
    try:
        return hasattr(_lib.load(), "mvsb200_conv3d_s1_fwd")
    except _lib.MvsB200Error:
        return False


conv_backends.register("tcgen05", Tcgen05ConvBackend)
