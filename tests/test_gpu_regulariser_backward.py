"""Backward of the default regulariser mode (bf16 operands on the tcgen05 kernels) against fp64 references.

Node level (sharp): each hand-written backward node against fp64 torch applied to the SAME bf16-rounded operands the kernels
saw, so that the only error left is the bf16 rounding of what the node stores.
  * _EntryConvs (conv_0_0 + the stacked stride-2 branches, one autograd node): the branches' data gradient is ADDED into the
    canvas conv_0_0's data gradient was written to (deconv3d_s2_kc_kernel, accumulate=1); branch gradients arrive as plain
    tensors or written in place by the box BatchNorm backward (ops.BoxGradDest).
  * the box BatchNorm of a branch with the epilogue sums of the strided convolution and a gradient destination;
  * the dense BatchNorm after a transposed convolution, with its epilogue partials, crop and skip addend, as up() calls it.
Mutations of the Python glue (accumulate dropped, sums of the wrong channels) show that these comparisons catch a lost path.

Whole module (calibrated): train-mode BatchNorm amplifies bf16 rounding to ~10 % in the gradients at random init, so a fixed
"close to fp64" bound could only catch gross faults.  The module's error is instead bounded by that of the same module on the
library's bf16 convolutions (same rounding points), and the fp64 references with one path cut must lie well outside that
bound.  The fp64 restatement of the reference network is itself pinned to the reference's goldens (the one CPU test here).
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import mvs_b200
import plane_sweep as ps
from mvs_b200 import conv3d as conv_backends
from mvs_b200 import conv3d_sm100, ops
from mvs_b200.regulariser import central_region

DEV = "cuda:0"
EPS, MOM = 1e-5, 0.1
SPLITS = (16, 32, 64)
PARAMS = [n + ".weight" for n in ps.REG_CONVS] + [n + s for n in ps.REG_BN for s in (".weight", ".bias")]
BN_USES = {"BN_0": 2, "BN_1": 3, "BN_2": 3, "BN_3": 2}


# ---------------------------------------------------------------------------------------------------------------------------
# A. fp64 restatement of CostVolumeReg.forward (oracle/plane_sweep.reg_forward: dense canvases, the reference's padding)
# ---------------------------------------------------------------------------------------------------------------------------
def reg_logits64(p, cv, detach_branches=False, detach_skip=False, frozen_stats=None, stats=None):
    """Logits of the reference network from the parameters `p` (name -> tensor, reference key names).
    detach_branches: no gradient from conv_{1,2,3}_0 into cv.  detach_skip: no gradient through y0 in y1 + y0.
    frozen_stats: name of a BatchNorm whose batch mean / variance are constants in the backward.
    stats: dict name -> list, receives (mean, biased var, voxels per channel) of every use of each BatchNorm."""
    D, h, w = cv.shape[-3:]
    pad, outpad = ps.reg_pad(D, h, w)

    def conv(name, x):
        _, _, s, tr = ps.REG_CONVS[name]
        wgt = p[name + ".weight"]
        if tr:
            return F.conv_transpose3d(x, wgt, stride=2, padding=pad, output_padding=outpad)
        return F.conv3d(x, wgt, stride=s, padding=(1 if s == 1 else pad))

    def bn_relu(name, x):
        mean, var = x.mean((0, 2, 3, 4)), x.var((0, 2, 3, 4), unbiased=False)
        if stats is not None:
            stats.setdefault(name, []).append((mean.detach(), var.detach(), x.numel() // x.shape[1]))
        if name == frozen_stats:
            mean, var = mean.detach(), var.detach()
        v = lambda t: t.view(1, -1, 1, 1, 1)
        return F.relu((x - v(mean)) * v(torch.rsqrt(var + EPS)) * v(p[name + ".weight"]) + v(p[name + ".bias"]))

    cvb = cv.detach() if detach_branches else cv
    y0 = bn_relu("BN_0", conv("conv_0_0", cv))
    y1 = bn_relu("BN_1", conv("conv_1_0", cvb))
    y2 = bn_relu("BN_2", conv("conv_2_0", cvb))
    y3 = bn_relu("BN_3", conv("conv_3_0", cvb))
    y1 = bn_relu("BN_1", conv("conv_1_1", y1))
    y2 = bn_relu("BN_2", conv("conv_2_1", y2))
    y3 = bn_relu("BN_3", conv("conv_3_1", y3))
    y3 = bn_relu("BN_2", conv("deconv_3_0", y3))
    y2 = bn_relu("BN_1", conv("deconv_2_0", y3 + y2))
    y1 = bn_relu("BN_0", conv("deconv_1_0", y2 + y1))
    return conv("conv_out", y1 + (y0.detach() if detach_skip else y0))


def running_after(stats, running):
    """torch.nn.BatchNorm's train-mode update of (running_mean, running_var), applied once per use in forward order."""
    out = {}
    for name, uses in stats.items():
        rm, rv = running[name + ".running_mean"].double(), running[name + ".running_var"].double()
        for mean, var, n in uses:
            rm = (1 - MOM) * rm + MOM * mean
            rv = (1 - MOM) * rv + MOM * var * (n / (n - 1))
        out[name + ".running_mean"], out[name + ".running_var"] = rm, rv
    return out


def _rank_depth(prob, d_batch, n_est=5):
    """scripts/depthmap.py:11-19, as tests/test_regulariser_algebra.py restates it."""
    _, order = prob.sort(dim=2, descending=True, stable=True)
    filt = prob * (order < n_est).to(prob.dtype)
    return (d_batch.unsqueeze(1) * filt).sum(2).squeeze(2) / filt.sum(2)


def test_fp64_restatement_reproduces_the_reference_gradients(golden_dir):
    """The checker of the whole-module tests, all switches off, against the gradients and running statistics the unmodified
    reference produced (tests/golden/tiny_b1v3.npz, its rank-based depth loss): agreement to 1e-4 relative (max-norm) pins the
    restatement to the reference rather than to the library it checks."""
    g = dict(np.load(os.path.join(golden_dir, "tiny_b1v3.npz")))
    w0 = dict(np.load(os.path.join(golden_dir, "reg_weights.npz")))
    p = {k: torch.from_numpy(np.asarray(w0[k])).double().requires_grad_(True) for k in PARAMS}
    cv = torch.from_numpy(g["cost"]).double().requires_grad_(True)
    stats = {}
    prob = torch.softmax(reg_logits64(p, cv, stats=stats), 2)
    depth = _rank_depth(prob, torch.from_numpy(g["d_batch"]).double())
    grads = torch.autograd.grad((depth * torch.from_numpy(g["gdepth"]).double()).sum(), [cv] + [p[k] for k in PARAMS])
    want = [g["gcv"]] + [g["gparam/" + k] for k in PARAMS]
    for name, got, ref in zip(["cv"] + PARAMS, grads, want):
        assert np.abs(got.numpy() - ref).max() <= 1e-4 * np.abs(ref).max(), name
    run = running_after(stats, {k: torch.from_numpy(np.asarray(v)) for k, v in w0.items()})
    for k, v in run.items():
        assert np.allclose(v.numpy(), g["bn_after/" + k], rtol=2e-5, atol=1e-6), k
    assert {k: len(v) for k, v in stats.items()} == BN_USES


# ---------------------------------------------------------------------------------------------------------------------------
# helpers of the GPU tests
# ---------------------------------------------------------------------------------------------------------------------------
def _err(a, ref):
    """(relative L2, relative max-norm) of a against ref, in fp64 on the host."""
    a, ref = a.detach().double().cpu(), ref.detach().double().cpu()
    d = a - ref
    return float(d.norm() / ref.norm()), float(d.abs().max() / ref.abs().max())


def _bf(t):
    """The bf16 rounding of t, as fp32 (values every path sees identically)."""
    return t.to(torch.bfloat16).float()


def _geometry(dims):
    reg = [central_region(n) for n in dims]
    pads = tuple(L for _, _, L in reg)
    C_lo = [lo for lo, _, _ in reg]
    C_hi = [hi for _, hi, _ in reg]
    m = tuple(hi - lo + 1 for lo, hi, _ in reg)
    E_lo = [max(0, lo - 1) for lo in C_lo]
    E_hi = [min(n - 1, hi + 1) for hi, n in zip(C_hi, dims)]
    F_lo = [max(0, e - 1) for e in E_lo]
    F_hi = [min(n - 1, e + 1) for e, n in zip(E_hi, dims)]
    return dict(pads=pads, m=m, C_lo=C_lo, C_hi=C_hi, F_lo=F_lo, F_dims=[b - a + 1 for a, b in zip(F_lo, F_hi)],
                box=tuple(slice(lo, hi + 1) for lo, hi in zip(C_lo, C_hi)),
                bgpad=sum(([C_lo[ax] - F_lo[ax], F_hi[ax] - C_hi[ax]] for ax in (2, 1, 0)), []))


def _entry_operands(B, dims, seed):
    """A non-negative volume (a variance cost volume is) and per-channel filter gains in [0.5, 2): the branch outputs then have
    per-channel means and spreads that differ, so statistics of the wrong channels are visibly wrong."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 32, *dims, generator=g).abs().to(torch.bfloat16).to(DEV).contiguous(memory_format=torch.channels_last_3d)
    gain = lambda c: 0.5 + 1.5 * torch.rand(c, 1, 1, 1, 1, generator=g)
    w00 = _bf(torch.randn(8, 32, 3, 3, 3, generator=g) * gain(8) / (27 * 32) ** 0.5).to(DEV)
    wcat = _bf(torch.randn(112, 32, 3, 3, 3, generator=g) * gain(112) / (27 * 32) ** 0.5).to(DEV)
    return g, x.requires_grad_(True), w00.requires_grad_(True), wcat.requires_grad_(True)


def _entry_reference(x, w00, wcat, dims, gy0, gS):
    """fp64 gradients (x, w00, wcat) of conv_0_0 (stride 1, padding 1) and of the reference's stride-2 layer (padding n//2+1)
    cropped to the central box, for output gradients gy0 and gS (the 112 stacked channels on the box)."""
    x64 = x.detach().double().cpu().requires_grad_(True)
    a64 = w00.detach().double().cpu().requires_grad_(True)
    b64 = wcat.detach().double().cpu().requires_grad_(True)
    y0 = F.conv3d(x64, a64, padding=1)
    S = F.conv3d(x64, b64, None, 2, tuple(n // 2 + 1 for n in dims))[(slice(None), slice(None)) + _geometry(dims)["box"]]
    (y0 * gy0.double().cpu()).sum().add((S * gS.double().cpu()).sum()).backward()
    return y0.detach(), S.detach(), x64.grad, a64.grad, b64.grad


# measured on a B200 (1000 W; bf16 operands, fp32 accumulation; relative max-norm): the cost volume's data gradient -- one bf16
# store by conv_0_0's data gradient, one by the accumulating transposed convolution -- up to 4.8e-3, the forward outputs up to
# 3.2e-3; the weight gradients (fp32 results of exact bf16 operands) up to 4e-6
NODE_TOL = 1e-2
WGRAD_TOL = 2e-5

ENTRY_DIMS = [(5, 12, 17), (8, 11, 14), (6, 7, 10), (13, 10, 5), (4, 6, 400)]


def _run_entry(B, dims, case, seed=0):
    """Forward of Tcgen05ConvBackend.entry_convs, then the backward with the branch gradients of `case`:
      "a" gy0 and all three branch gradients as plain tensors (the accumulate path);  "b" y0 unused;
      "c" branch 2 without a gradient;  "d" branches 0 and 2 through the box BatchNorm's in-place gradient destination.
    Returns (errors by name: (relative L2, relative max-norm), launches of the backward, weight gradient on the line kernel?)."""
    geo = _geometry(dims)
    g, x, w00, wcat = _entry_operands(B, dims, seed + sum(dims))
    n_full = B * dims[0] * dims[1] * dims[2]
    be = conv_backends.get("tcgen05")
    n0 = mvs_b200.launch_count()
    y0, S = be.entry_convs(x, w00, wcat, geo["pads"], geo["m"], SPLITS)
    assert mvs_b200.launch_count() > n0, "the tcgen05 kernels did not run"
    assert y0.dtype == torch.bfloat16 and [s.shape[1] for s in S] == list(SPLITS)
    gy0 = _bf(torch.randn(y0.shape, generator=g)).to(DEV)
    gS = [_bf(torch.randn(s.shape, generator=g)).to(DEV) for s in S]
    if case == "b":
        for t in gS:                     # the branches reach only part of the canvas: the rest of cv's gradient must be 0
            t[..., t.shape[-1] // 2:] = 0
    loss = 0 if case == "b" else (y0.float() * gy0).sum()
    inplace = (0, 2) if case == "d" else ()
    bn = {}
    for k, s in enumerate(S):
        if case == "c" and k == 2:
            continue
        if k in inplace:
            gamma = _bf(torch.rand(SPLITS[k], generator=g) + 0.5).to(DEV)
            beta = _bf(torch.randn(SPLITS[k], generator=g) * 0.3).to(DEV)
            X = ops.box_batchnorm_relu(s, gamma, beta, n_full, EPS, geo["C_lo"], geo["F_lo"], geo["F_dims"],
                                       grad_dest=s._mvs_grad_dest, sums=s._mvs_box_sums)[0]
            GX = _bf(torch.randn(X.shape, generator=g)).to(DEV)
            loss = loss + (X.float() * GX).sum()
            bn[k] = s
        else:
            loss = loss + (s.float() * gS[k]).sum()
    lines = conv3d_sm100._s2_wgrad_mode(x.shape, (B, sum(SPLITS)) + geo["m"]) == "lines"
    n1 = mvs_b200.launch_count()
    loss.backward()
    launches = mvs_b200.launch_count() - n1
    # the gradients the entry node received: what was passed, zeros for what was not, the holder's slices for in-place ones
    if case == "b":
        gy0 = torch.zeros_like(gy0)
    if case == "c":
        gS[2] = torch.zeros_like(gS[2])
    for k, s in bn.items():
        holder, kk = s._mvs_grad_dest
        assert holder.filled[kk], "the box BatchNorm backward did not write into the gradient destination"
        gS[k] = holder.dest(kk).float()
    r_y0, r_S, r_gx, r_g00, r_gcat = _entry_reference(x, w00, wcat, dims, gy0, torch.cat(gS, 1))
    errs = {"y0": _err(y0, r_y0), "S": _err(torch.cat(S, 1), r_S), "gx": _err(x.grad, r_gx), "gw_cat": _err(wcat.grad, r_gcat)}
    if case == "b":
        assert w00.grad is None or w00.grad.abs().max() == 0           # y0 unused: conv_0_0's weight gradient is exactly 0
        unreached = r_gx == 0
        assert unreached.any()
        assert x.grad.cpu()[unreached].abs().max() == 0, "canvas voxels no branch reaches are not exactly 0"
    else:
        errs["gw00"] = _err(w00.grad, r_g00)
    return errs, launches, lines


def _check_entry(errs):
    for k, v in errs.items():
        assert v[1] < (WGRAD_TOL if k.startswith("gw") else NODE_TOL), (k, v)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["a", "b", "c", "d"])
@pytest.mark.parametrize("dims", ENTRY_DIMS)
def test_entry_convs_backward(dims, case, monkeypatch):
    """B.1: conv_0_0 and the stacked branches as one node.  Per-axis sizes 4..8 (the dilated box touches the canvas border:
    regulariser.py pads X) and >= 10, odd and even; one 400-voxel line (the weight gradient then runs on the parity-class kernel,
    _lines_fit).  The branches' data gradient must be issued with accumulate=True into conv_0_0's canvas."""
    calls = []
    orig = conv3d_sm100.conv_transpose3d_s2_kc

    def recording(*a, **kw):
        calls.append((bool(kw.get("accumulate", False)), kw.get("out") is not None))
        return orig(*a, **kw)

    monkeypatch.setattr(conv3d_sm100, "conv_transpose3d_s2_kc", recording)
    monkeypatch.setattr(ops, "EVENTS", {})
    errs, launches, lines = _run_entry(2, dims, case)
    print(f"entry {dims} case {case}: " + ", ".join(f"{k} {v[0]:.1e}/{v[1]:.1e}" for k, v in errs.items()))
    _check_entry(errs)
    assert calls == [(True, True)], calls                  # one branch data gradient, added into the existing canvas
    ran = set(ops.EVENTS)
    assert {"conv3d_s1_tc", "conv3d_s1_wgrad_tc", "conv3d_s2_wgrad_tc", "deconv3d_s2_tc"} <= ran, ran
    if lines and case != "d":
        # conv_0_0: filter packing + data gradient + weight gradient; branches: weight gradient + 3 filter chunks + the
        # transposed convolution -- no library convolution
        assert launches == 8, launches


def _run_box_bn(dims, k, seed=0, wrong_sums=False):
    """B.2: box BatchNorm of branch k of the stacked convolution with the epilogue sums and the in-place gradient destination;
    gradients enter through X, scale and relu(shift)."""
    B = 2
    geo = _geometry(dims)
    g, x, w00, wcat = _entry_operands(B, dims, seed + 17 * k)
    n_full = B * dims[0] * dims[1] * dims[2]
    y0, S = conv_backends.get("tcgen05").entry_convs(x, w00, wcat, geo["pads"], geo["m"], SPLITS)
    s, n = S[k], SPLITS[k]
    sums = s._mvs_box_sums
    assert sums is not None
    if wrong_sums:                              # n channels of the stacked sums that belong to another branch
        holder = s._mvs_grad_dest[0]
        a = {0: 16, 1: 48, 2: 0}[k]
        sums = (holder.sums[0, a:a + n], holder.sums[1, a:a + n])
    gamma = _bf(torch.rand(n, generator=g) + 0.5).to(DEV).requires_grad_(True)
    beta = _bf(torch.randn(n, generator=g) * 0.3).to(DEV).requires_grad_(True)
    X, scale, shift, mean, var = ops.box_batchnorm_relu(s, gamma, beta, n_full, EPS, geo["C_lo"], geo["F_lo"], geo["F_dims"],
                                                        grad_dest=s._mvs_grad_dest, sums=sums)
    GX = _bf(torch.randn(X.shape, generator=g)).to(DEV)
    # gradients of the scale / shift outputs of the size the module's analytic outside sums give them (sums over many voxels)
    gsc, gsh = torch.randn(n, generator=g).to(DEV) * 100, torch.randn(n, generator=g).to(DEV) * 100
    ((X.float() * GX).sum() + (scale * gsc).sum() + (F.relu(shift) * gsh).sum()).backward()
    holder, kk = s._mvs_grad_dest
    assert holder.filled[kk]
    gS = holder.dest(kk)
    # fp64 torch of the regulariser's CPU path on the stored S: statistics over the canvas (zeros outside the box), X on F
    S64 = s.detach().double().cpu().requires_grad_(True)
    g64 = gamma.detach().double().cpu().requires_grad_(True)
    b64 = beta.detach().double().cpu().requires_grad_(True)
    m64 = S64.sum((0, 2, 3, 4)) / n_full
    v64 = (S64 * S64).sum((0, 2, 3, 4)) / n_full - m64 * m64
    sc64 = g64 * torch.rsqrt(v64 + EPS)
    sh64 = b64 - m64 * sc64
    X64 = F.relu(F.pad(S64, geo["bgpad"]) * sc64.view(1, -1, 1, 1, 1) + sh64.view(1, -1, 1, 1, 1))
    ((X64 * GX.double().cpu()).sum() + (sc64 * gsc.double().cpu()).sum() + (F.relu(sh64) * gsh.double().cpu()).sum()).backward()
    return {"X": _err(X, X64), "mean": _err(mean, m64), "var": _err(var, v64), "gS": _err(gS, S64.grad),
            "g_gamma": _err(gamma.grad, g64.grad), "g_beta": _err(beta.grad, b64.grad)}


# measured on a B200 (1000 W; relative max-norm): X and gS (bf16 stores) up to 5.1e-3; mean / variance (from the fp32 epilogue
# sums, the reference from the stored bf16 values) up to 6.6e-4; the gradients of gamma and beta (fp32) up to 2.7e-4
BOX_TOL = {"X": NODE_TOL, "gS": NODE_TOL, "mean": 2e-3, "var": 2e-3, "g_gamma": 1e-3, "g_beta": 1e-3}


@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 1, 2])
@pytest.mark.parametrize("dims", [(6, 7, 10), (11, 14, 20)])
def test_box_batchnorm_with_epilogue_sums_and_gradient_destination(dims, k):
    """B.2: mean and variance over the whole canvas (zeros outside the box) from the strided convolution's epilogue sums, X on F
    with relu(shift) around the data, gradients of S (written into the stacked buffer), gamma, beta -- including what enters
    through the scale / shift outputs -- against the torch expressions of the regulariser's CPU path in fp64."""
    errs = _run_box_bn(dims, k)
    print(f"box bn {dims} branch {k}: " + ", ".join(f"{n} {v[0]:.1e}/{v[1]:.1e}" for n, v in errs.items()))
    for n, tol in BOX_TOL.items():
        assert errs[n][1] < tol, (n, errs[n])


# measured on a B200 (1000 W; relative max-norm): dU (bf16 store of the BatchNorm backward) and the transposed convolution's
# input gradient up to 3.3e-3; dgamma / dbeta (fp32, statistics from the epilogue partials) up to 2e-4; the weight gradient
# up to 3.2e-7
DENSE_TOL = {"dU": NODE_TOL, "dgamma": 1e-3, "dbeta": 1e-3, "dz": NODE_TOL, "dw": WGRAD_TOL}


@pytest.mark.gpu
@pytest.mark.parametrize("cin,cout", [(64, 32), (32, 16), (16, 8)])
@pytest.mark.parametrize("dims", [(6, 7, 10), (11, 14, 20)])
def test_dense_batchnorm_after_transposed_conv_backward(cin, cout, dims):
    """B.3: conv_transpose3d_alloc -> batchnorm_relu_train(crop, canvas, add, partials) exactly as regulariser.up() calls it
    (64->32 and 32->16 cropped to the box with the branch addend, 16->8 dense with the y0 addend): gradients of the canvas over
    the whole allocation, of gamma, beta and the addend, and the transposed convolution's gradients from that canvas gradient."""
    B = 2
    geo = _geometry(dims)
    g = torch.Generator().manual_seed(cin + cout + sum(dims))
    z = torch.randn(B, cin, *geo["m"], generator=g).to(torch.bfloat16).to(DEV).contiguous(memory_format=torch.channels_last_3d)
    z.requires_grad_(True)
    w = _bf(torch.randn(cin, cout, 3, 3, 3, generator=g) / (8 * cin) ** 0.5).to(DEV).requires_grad_(True)
    gamma = _bf(torch.rand(cout, generator=g) + 0.5).to(DEV).requires_grad_(True)
    beta = _bf(torch.randn(cout, generator=g) * 0.3).to(DEV).requires_grad_(True)
    crop = geo["box"] if cout != 8 else None
    out_dims = geo["m"] if crop is not None else dims
    add = torch.randn(B, cout, *out_dims, generator=g).to(torch.bfloat16).to(DEV).contiguous(memory_format=torch.channels_last_3d)
    add.requires_grad_(True)
    U = conv_backends.get("tcgen05").conv_transpose3d_alloc(z, w, 2, geo["pads"], dims)
    U.retain_grad()
    part = getattr(U, "_mvs_bn_partials", None)
    assert part is not None and part[2] == dims
    rm, rv, nbt = torch.zeros(cout, device=DEV), torch.ones(cout, device=DEV), torch.zeros((), dtype=torch.int64, device=DEV)
    box = None if crop is None else tuple((c.start, c.stop) for c in crop)
    y, _, _ = ops.batchnorm_relu_train(U, gamma, beta, EPS, relu=True, crop=box, canvas=dims, running=(rm, rv, nbt), momentum=MOM,
                                       partials=part, add=add)
    G = _bf(torch.randn(y.shape, generator=g)).to(DEV)
    (y.float() * G).sum().backward()
    D, h, wd = dims
    U64 = U.detach().double().cpu().requires_grad_(True)
    g64 = gamma.detach().double().cpu().requires_grad_(True)
    b64 = beta.detach().double().cpu().requires_grad_(True)
    y64 = F.relu(F.batch_norm(U64[..., :D, :h, :wd], None, None, g64, b64, True, MOM, EPS))
    if crop is not None:
        y64 = y64[(slice(None), slice(None)) + crop]
    (y64 * G.double().cpu()).sum().backward()                  # over the allocation: zero gradient outside the canvas
    errs = {"dU": _err(U.grad, U64.grad), "dgamma": _err(gamma.grad, g64.grad), "dbeta": _err(beta.grad, b64.grad)}
    assert torch.equal(add.grad.float(), G)                    # the addend's gradient is the output's (a bf16 value here)
    # the transposed convolution's backward from the canvas gradient it received (fp64, the same bf16 operands)
    z64 = z.detach().double().cpu().requires_grad_(True)
    w64 = w.detach().double().cpu().requires_grad_(True)
    Ur = conv_backends.TorchConvBackend.conv_transpose3d(z64, w64, 2, geo["pads"], dims)
    (Ur * U.grad.double().cpu()).sum().backward()
    errs.update(dz=_err(z.grad, z64.grad), dw=_err(w.grad, w64.grad))
    print(f"dense bn {cin}->{cout} {dims}: " + ", ".join(f"{n} {v[0]:.1e}/{v[1]:.1e}" for n, v in errs.items()))
    for n, tol in DENSE_TOL.items():
        assert errs[n][1] < tol, (n, errs[n])


@pytest.mark.gpu
def test_mutations_are_caught(monkeypatch):
    """B.4: the node comparisons fail, by at least 10x their tolerance, when the Python glue drops a path: the branches' data
    gradient written over conv_0_0's canvas instead of added to it; the box BatchNorm fed the epilogue sums of other channels."""
    orig = conv3d_sm100.conv_transpose3d_s2_kc

    def overwrite(*a, **kw):
        kw["accumulate"] = False
        return orig(*a, **kw)

    monkeypatch.setattr(conv3d_sm100, "conv_transpose3d_s2_kc", overwrite)
    errs, _, _ = _run_entry(2, (8, 11, 14), "a")
    print(f"mutation accumulate=False: gx {errs['gx']}")
    assert errs["gx"][1] >= 10 * NODE_TOL, errs["gx"]
    monkeypatch.setattr(conv3d_sm100, "conv_transpose3d_s2_kc", orig)
    for k in range(3):
        errs = _run_box_bn((11, 14, 20), k, wrong_sums=True)
        print(f"mutation wrong sums, branch {k}: gS {errs['gS']}")
        assert errs["gS"][1] >= 10 * BOX_TOL["gS"], (k, errs["gS"])


# ---------------------------------------------------------------------------------------------------------------------------
# C. whole module in the default mode, calibrated against the same module on the library's bf16 convolutions
# ---------------------------------------------------------------------------------------------------------------------------
def _module_state(seed):
    """Reference init (plane_sweep.reg_init) with gamma in [0.5, 1.5), beta ~ 0.3 N(0, 1); every parameter rounded to bf16, so
    the fp32 parameters of the module, the bf16 copies its kernels pack and the fp64 reference all hold the same values."""
    sd = ps.reg_init(seed)
    g = torch.Generator().manual_seed(seed + 1)
    for name, c in ps.REG_BN.items():
        sd[name + ".weight"] = torch.rand(c, generator=g) + 0.5
        sd[name + ".bias"] = torch.randn(c, generator=g) * 0.3
    return {k: (_bf(v) if k in PARAMS else v) for k, v in sd.items()}


def _module_inputs(B, dims, seed):
    g = torch.Generator().manual_seed(seed + 2)
    cv = torch.randn(B, 32, *dims, generator=g).to(torch.bfloat16)
    G = torch.randn(B, 1, *dims, generator=g)
    return cv, G


def _module_run(sd, cv, G, backend):
    """One train-mode forward + backward of CostVolumeReg (default precision) with loss sum(prob * G) -> (gradients of cv and
    the 19 parameters, state after the pass)."""
    reg = mvs_b200.CostVolumeReg(device=DEV, conv_backend=backend).train()
    reg.load_state_dict(sd)
    x = cv.to(DEV).contiguous(memory_format=torch.channels_last_3d).requires_grad_(True)
    prob = reg(x)
    named = dict(reg.named_parameters())
    grads = torch.autograd.grad((prob * G.to(DEV)).sum(), [x] + [named[k] for k in PARAMS])
    torch.cuda.synchronize()
    out = dict(zip(["cv"] + PARAMS, [t.detach().float().cpu() for t in grads]))
    return out, {k: v.detach().cpu() for k, v in reg.state_dict().items()}


_REF = {}


def _module_reference(B, dims, seed, **switch):
    """fp64 gradients (and running statistics after the pass) of the restatement on the bf16-rounded cv and parameters."""
    key = (B, dims, seed, tuple(sorted(switch.items())))
    if key not in _REF:
        sd = _module_state(seed)
        cv, G = _module_inputs(B, dims, seed)
        p = {k: sd[k].double().requires_grad_(True) for k in PARAMS}
        cv64 = cv.double().requires_grad_(True)
        stats = {}
        prob = torch.softmax(reg_logits64(p, cv64, stats=stats, **switch), 2)
        leaves = [cv64] + [p[k] for k in PARAMS]
        grads = torch.autograd.grad((prob * G.double()).sum(), leaves, allow_unused=True)     # a cut can leave a leaf unused
        grads = [torch.zeros_like(t) if g is None else g for g, t in zip(grads, leaves)]
        _REF[key] = (dict(zip(["cv"] + PARAMS, grads)), running_after(stats, sd))
    return _REF[key]


# Per tensor, e_own <= LIB_FACTOR * e_lib + 0.01.  The two paths do not round at exactly the same points: the own path takes the
# branches' BatchNorm statistics from the fp32 accumulators of the strided convolution (and the decoder's from those of the
# transposed convolutions), the library path from the stored bf16 values.  Either is one bf16 rounding away from fp64, but the
# network amplifies each into a different ~5-15 % realisation: in an fp64 emulation of the storage points (8 seeds at
# B=1, 8x12x14) that change alone moves single-tensor errors by up to 1.9x, and on a B200 (1000 W) BN_1.weight at that shape
# reads 0.046 (own) against 0.023 (library).  Hence 2x, not 1.5x.
LIB_FACTOR = 2.0
# a reference with one path cut must lie at least CUT_FACTOR bounds away on the tensors that path carries.  Measured on a B200:
# cv 6.8-9x (branches, skip), conv_0_0.weight 26x (skip); BN_3.bias 2.8-4.3x (statistics; its gradient passes through the
# statistics of BN_3's second use, conv_3_1: box sums + closed-form outside sums -- the conv_3_{0,1} weights move only 0.2-2x)
CUT_FACTOR = 2.5
SENSITIVITY = {"detach_branches": ["cv"], "detach_skip": ["cv", "conv_0_0.weight"], "frozen_stats": ["BN_3.bias"]}

MODULE_CASES = [((1, (8, 12, 14)), None), ((2, (12, 33, 47)), None), ((1, (7, 24, 40)), None),
                ((1, (8, 12, 14)), "MVSB200_S2_STATS=0"), ((1, (8, 12, 14)), "MVSB200_DECONV_STATS=0"),
                ((1, (8, 12, 14)), "MVSB200_S2_DGRAD=cudnn")]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,env", MODULE_CASES, ids=lambda v: str(v))
def test_module_backward_is_as_close_to_fp64_as_the_library_path(shape, env, monkeypatch):
    """C: CostVolumeReg() in train mode, bf16 cost volume, loss sum(prob * G).  Per gradient tensor (cv and the 19 parameters)
    and per running statistic, the relative L2 error against the fp64 restatement must satisfy e_own <= 2 e_lib + 0.01, e_lib
    being that of the same module on the library's bf16 convolutions (same storage dtype, no own convolution kernel): a bound
    calibrated on an independent bf16 implementation instead of a guessed constant (train-mode BatchNorm at random init
    amplifies bf16 rounding to ~10 % in some parameter gradients).  The fp64 references with one path cut -- cv into the
    branches, y0 in y1 + y0, BN_3's batch statistics -- lie at least 2.5x that bound away, so a lost path cannot pass.
    num_batches_tracked advances by exactly the number of uses of each shared BatchNorm."""
    B, dims = shape
    seed = 5
    if env is not None:
        k, v = env.split("=")
        monkeypatch.setenv(k, v)
    sd = _module_state(seed)
    cv, G = _module_inputs(B, dims, seed)
    monkeypatch.setattr(ops, "EVENTS", {})
    own, own_state = _module_run(sd, cv, G, "auto")
    ran = set(ops.EVENTS)
    assert {"conv3d_s2_tc", "deconv3d_s2_tc", "conv3d_s2_wgrad_tc", "box_bn_relu_bwd"} <= ran, ran
    monkeypatch.setattr(ops, "EVENTS", None)
    lib, lib_state = _module_run(sd, cv, G, "cudnn")
    ref, ref_run = _module_reference(B, dims, seed)
    for name, uses in BN_USES.items():
        assert int(own_state[name + ".num_batches_tracked"]) == uses == int(lib_state[name + ".num_batches_tracked"]), name
    e, bound = {}, {}
    for name in ["cv"] + PARAMS + sorted(ref_run):
        want = ref[name] if name in ref else ref_run[name]
        got, cal = (own[name], lib[name]) if name in ref else (own_state[name], lib_state[name])
        e[name] = _err(got, want)[0], _err(cal, want)[0]
        bound[name] = LIB_FACTOR * e[name][1] + 0.01
    print(f"module B={B} {dims} {env}: e_own/e_lib " + ", ".join(f"{n} {a:.4f}/{b:.4f}" for n, (a, b) in e.items()))
    for name, (e_own, e_lib) in e.items():
        assert e_own <= bound[name], (name, e_own, e_lib)
    if env is None:
        for switch, names in SENSITIVITY.items():
            cut, _ = _module_reference(B, dims, seed, **{switch: "BN_3" if switch == "frozen_stats" else True})
            for name in names:
                d = _err(cut[name], ref[name])[0]
                print(f"  {switch}: {name} moves {d:.3f} (bound {bound[name]:.3f})")
                assert d >= CUT_FACTOR * bound[name], (switch, name, d, bound[name])
