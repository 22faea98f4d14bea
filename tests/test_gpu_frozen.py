"""FrozenMVSNet (eval-mode inference with BatchNorm folded into the tcgen05 convolution epilogues) against fp64 references.

Kernel nodes: the affine epilogues of conv3d_s1_kdn_kernel (volume and planar mode) and deconv3d_s2_tc_kernel (with / without
the skip addend, windowed output) against fp64 torch on the same bf16 operands: relative max-norm <= 1e-2 (one bf16 rounding).
Whole networks: the running statistics come from train-mode passes over the test inputs and are then perturbed per channel
(variance x U(0.25, 4), mean shifted) -- at the initial 0 / 1 statistics eval-mode BatchNorm is nearly the identity and would
hide a wrong vector.  The regulariser's bound is 1e-2 and at most 2x (+1e-3) the error of today's CostVolumeReg().eval()."""
import copy
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import mvs_b200
from mvs_b200 import _lib, harness, nets2d, refine
from mvs_b200.conv3d_sm100 import _NAT, _kdn_order, _n_rows, _pack
from mvs_b200.ops import _stream

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
CL3 = torch.channels_last_3d


def _relmax(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max())


def _bf(t):
    return t.to(torch.bfloat16).double()


def _affine(c, gen):
    """BatchNorm-like vectors with negative weights among them."""
    scale = (torch.rand(c, generator=gen) * 2 - 0.7)
    shift = torch.randn(c, generator=gen) * 0.5
    return scale.to(DEV), shift.to(DEV)


# ------------------------------------------------------------------------------------------------------------------ kdn
def _run_kdn(x, w, scale, shift, out_dims, off, planar):
    """x: bf16 [B, cin, D, H, W] channel-last; w [cout, cin, 3, 3, 3] (planar: [cout, cin, 3, 3])."""
    B, cin, Di, Hi, Wi = x.shape
    cout = w.shape[0]
    if planar:
        wk = nets2d._pack2d(w.float().contiguous(), "fwd", _n_rows(cout), max(cin, 16))
    else:
        wk = _pack(w, 0, _n_rows(cout), _kdn_order(_NAT), n_cols=max(cin, 16))
    y = torch.empty((B, cout) + tuple(out_dims), dtype=torch.bfloat16, device=DEV, memory_format=CL3)
    _lib.call("mvsb200_conv3d_s1_fwd_kdn_affine", x.data_ptr(), wk.data_ptr(), y.data_ptr(), B, Di, Hi, Wi, cin, *out_dims, cout, cout,
              _n_rows(cout), *off, int(planar), scale.data_ptr(), shift.data_ptr(), _stream())
    return y


# volume mode: every channel pair the frozen model launches (conv_0_0, conv_{1,2,3}_1); pad 1, and the E -> C offsets of conv_k_1
@pytest.mark.parametrize("cin,cout", [(32, 8), (16, 16), (32, 32), (64, 64)])
@pytest.mark.parametrize("dims,off", [((5, 13, 17), (-1, -1, -1)), ((7, 11, 21), (0, -1, 0))])
def test_kdn_affine_volume(cin, cout, dims, off):
    gen = torch.Generator().manual_seed(cin * 100 + cout)
    B = 2
    x = torch.randn((B, cin) + dims, generator=gen).to(DEV).to(torch.bfloat16).contiguous(memory_format=CL3)
    w = (torch.randn(cout, cin, 3, 3, 3, generator=gen) / (27 * cin) ** 0.5).to(DEV)
    scale, shift = _affine(cout, gen)
    out_dims = tuple(n - 2 - 2 * o for n, o in zip(dims, off))                    # padding -off per axis
    y = _run_kdn(x, w, scale, shift, out_dims, off, False)
    ref = F.conv3d(F.pad(x.double(), [-o for o in reversed(off) for _ in range(2)]), _bf(w))
    ref = torch.relu(ref * scale.double().view(1, -1, 1, 1, 1) + shift.double().view(1, -1, 1, 1, 1))
    assert y.shape == ref.shape
    assert _relmax(y, ref) <= 1e-2


# planar mode: the encoder's layers (8-channel image rows, space-to-depth inputs) and the refinement's
@pytest.mark.parametrize("cx,ci,co", [(8, 3, 8), (8, 8, 8), (32, 32, 16), (16, 16, 16), (64, 64, 32), (32, 32, 32), (16, 4, 32)])
def test_kdn_affine_planar(cx, ci, co):
    gen = torch.Generator().manual_seed(cx * 1000 + ci * 10 + co)
    N, H, W = 3, 37, 53
    x = torch.zeros(1, cx, N, H, W)
    x[:, :ci] = torch.randn(1, ci, N, H, W, generator=gen)
    x = x.to(DEV).to(torch.bfloat16).contiguous(memory_format=CL3)
    w = (torch.randn(co, ci, 3, 3, generator=gen) / (9 * ci) ** 0.5).to(DEV)
    scale, shift = _affine(co, gen)
    y = _run_kdn(x, w, scale, shift, (N, H, W), (0, -1, -1), True)
    maps = x.double()[0, :ci].permute(1, 0, 2, 3)                                   # [N, ci, H, W]
    ref = F.conv2d(maps, _bf(w), padding=1)
    ref = torch.relu(ref * scale.double().view(1, -1, 1, 1) + shift.double().view(1, -1, 1, 1))
    assert _relmax(y[0].permute(1, 0, 2, 3), ref) <= 1e-2


# ------------------------------------------------------------------------------------------------------------------ deconv
def _run_deconv(x, w, scale, shift, canvas, pads, win_lo, win_dims, add):
    B, cin = x.shape[:2]
    cout = w.shape[1]
    wp = _pack(w, 1, _n_rows(cout), _NAT + [-1])
    y = torch.empty((B, cout) + tuple(win_dims), dtype=torch.bfloat16, device=DEV, memory_format=CL3)
    ys = (ctypes.c_int64 * 4)(y.stride(0), y.stride(2), y.stride(3), y.stride(4))
    if add is not None:
        assert add.stride() == y.stride()
    _lib.call("mvsb200_deconv3d_s2_fwd_affine", x.data_ptr(), wp.data_ptr(), y.data_ptr(), B, *x.shape[2:], cin, *canvas, cout,
              _n_rows(cout), *pads, (ctypes.c_int * 6)(*win_lo, *win_dims), ys, scale.data_ptr(), shift.data_ptr(),
              None if add is None else add.data_ptr(), _stream())
    return y


@pytest.mark.parametrize("cin,cout", [(64, 32), (32, 16), (16, 8)])
@pytest.mark.parametrize("canvas", [(8, 16, 20), (7, 15, 19), (9, 13, 22)])
@pytest.mark.parametrize("with_add", [False, True])
def test_deconv_affine_window(cin, cout, canvas, with_add):
    import plane_sweep as ps
    gen = torch.Generator().manual_seed(cin + sum(canvas) + with_add)
    B = 2
    reg = [mvs_b200.central_region(n) for n in canvas]
    C_lo = tuple(lo for lo, _, _ in reg)
    C_dims = tuple(hi - lo + 1 for lo, hi, _ in reg)
    pads = tuple(L for _, _, L in reg)
    x = torch.randn((B, cin) + C_dims, generator=gen).to(DEV).to(torch.bfloat16).contiguous(memory_format=CL3)
    w = (torch.randn(cin, cout, 3, 3, 3, generator=gen) / (27 * cin / 8) ** 0.5).to(DEV)
    scale, shift = _affine(cout, gen)
    add_full = torch.randn((B, cout) + canvas, generator=gen).to(DEV).to(torch.bfloat16).contiguous(memory_format=CL3)
    box = (slice(None), slice(None)) + tuple(slice(lo, lo + n) for lo, n in zip(C_lo, C_dims))
    add_win = add_full[box].contiguous(memory_format=CL3) if with_add else None
    y_win = _run_deconv(x, w, scale, shift, canvas, pads, C_lo, C_dims, add_win)
    y_full = _run_deconv(x, w, scale, shift, canvas, pads, (0, 0, 0), canvas, add_full if with_add else None)
    # the window is computed exactly as the same window of a full-canvas launch
    assert torch.equal(y_win, y_full[box])
    # fp64: the reference's dense transposed convolution of the canvas that is zero outside C
    pad, outpad = ps.reg_pad(*canvas)
    xin = torch.zeros((B, cin) + canvas, dtype=torch.float64, device=DEV)
    xin[box] = x.double()
    ref = F.conv_transpose3d(xin, _bf(w), stride=2, padding=pad, output_padding=outpad)
    ref = torch.relu(ref * scale.double().view(1, -1, 1, 1, 1) + shift.double().view(1, -1, 1, 1, 1))
    if with_add:
        ref = ref + add_full.double()
    assert _relmax(y_full, ref) <= 1e-2
    assert _relmax(y_win, ref[box]) <= 1e-2


# ------------------------------------------------------------------------------------------------------------------ models
def _perturb_running_stats(module, seed):
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in module.modules():
            if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
                c = m.num_features
                m.running_var.mul_((0.25 * 16 ** torch.rand(c, generator=gen)).to(m.running_var.device))
                m.running_mean.add_((torch.randn(c, generator=gen) * m.running_var.cpu().sqrt()).to(m.running_mean.device))
                m.weight.copy_((torch.rand(c, generator=gen) * 2 - 0.5).to(m.weight.device))        # some negative
                m.bias.copy_((torch.randn(c, generator=gen) * 0.2).to(m.bias.device))


def _reg_eval64(sd, cv, swap12=False, drop_y0=False, unshift_dc2=False):
    """Eval-mode CostVolumeReg in fp64 on dense canvases (oracle/plane_sweep.reg_forward with train_bn=False), with switches that
    cut one path: BN_1 / BN_2 vectors exchanged between the two decoder layers, the y0 skip addition dropped, the box of
    deconv_2_0's output taken at the canvas origin instead of at C."""
    import plane_sweep as ps
    D, h, w = cv.shape[-3:]
    pad, outpad = ps.reg_pad(D, h, w)
    reg = [mvs_b200.central_region(n) for n in (D, h, w)]
    C = (slice(None), slice(None)) + tuple(slice(lo, hi + 1) for lo, hi, _ in reg)
    C0 = (slice(None), slice(None)) + tuple(slice(0, hi - lo + 1) for lo, hi, _ in reg)

    def bn(name, x, widen=None):
        rm, rv, g, b = (sd[f"{name}.{k}"] for k in ("running_mean", "running_var", "weight", "bias"))
        if widen is not None:                   # another layer's vectors cut / repeated to this layer's width
            rm, rv, g, b = (torch.cat([t] * (widen // t.numel() + 1))[:widen] for t in (rm, rv, g, b))
        return F.relu(F.batch_norm(x, rm, rv, g, b, False, 0.0, 1e-5))

    conv = lambda n, x, s: F.conv3d(x, sd[n + ".weight"], stride=s, padding=1 if s == 1 else pad)
    convT = lambda n, x: F.conv_transpose3d(x, sd[n + ".weight"], stride=2, padding=pad, output_padding=outpad)
    y0 = bn("BN_0", conv("conv_0_0", cv, 1))
    e = {k: bn(f"BN_{k}", conv(f"conv_{k}_1", bn(f"BN_{k}", conv(f"conv_{k}_0", cv, 2)), 1)) for k in (1, 2, 3)}
    c3 = bn("BN_1" if swap12 else "BN_2", convT("deconv_3_0", e[3]), 32 if swap12 else None)
    s3 = torch.zeros_like(c3)
    s3[C] = c3[C] + e[2][C]
    c2 = bn("BN_2" if swap12 else "BN_1", convT("deconv_2_0", s3), 16 if swap12 else None)
    s2 = torch.zeros_like(c2)
    s2[C] = (c2[C0] if unshift_dc2 else c2[C]) + e[1][C]
    z = bn("BN_0", convT("deconv_1_0", s2)) + (0 if drop_y0 else y0)
    return F.conv3d(z, sd["conv_out.weight"], padding=1)


def _reg_case(name, golden_dir):
    """(cost volume bf16 on the device, CostVolumeReg with trained-then-perturbed running statistics)."""
    if name == "cfg1":
        # noise on ramps along every axis: a stationary volume would hide a window shifted by tens of voxels
        gen = torch.Generator().manual_seed(7)
        ramp = sum(torch.linspace(0, 3, n).view([-1 if i == ax else 1 for i in range(3)]) for ax, n in enumerate((192, 128, 160)))
        cost = (torch.rand(1, 32, 192, 128, 160, generator=gen) * ramp).to(DEV)
    else:
        g = np.load(f"{golden_dir}/{name}.npz")
        cost = torch.from_numpy(g["cost"]).to(DEV)
    cost = cost.to(torch.bfloat16).contiguous(memory_format=CL3)
    torch.manual_seed(3)
    reg = mvs_b200.CostVolumeReg().to(DEV).train()
    with torch.no_grad():
        for _ in range(3):
            reg(cost)                                               # running statistics from the test inputs
    _perturb_running_stats(reg, 11)
    return cost, reg.eval()


def _frozen_regulariser(reg):
    holder = torch.nn.Module()
    holder.feature_encoder, holder.cost_volume_reg, holder.depthmap_refine = harness.FeatureEncoder(), reg, harness.DepthRefinement()
    holder.d_num, holder.d_scale = 8, 1.0
    return mvs_b200.FrozenMVSNet(holder.to(DEV))


@pytest.mark.parametrize("name", ["tiny_b1v3", "v7_odd", "cfg1"])
def test_regulariser_against_fp64(golden_dir, name):
    import plane_sweep as ps
    from mvs_b200 import conv3d as conv_backends
    cost, reg = _reg_case(name, golden_dir)
    fz = _frozen_regulariser(reg)
    sd = {k: v.double() if v.is_floating_point() else v for k, v in reg.state_dict().items()}
    cv = cost.double()
    ref_prob, ref_logits = ps.reg_forward(sd, cv, train_bn=False, return_logits=True)
    logits = fz.logits(cost)
    prob = fz.regularise(cost)
    with torch.no_grad():
        today_logits = reg.logits(cost, conv_backends.get(reg.conv_backend))
        today_prob = reg(cost)
    e_l, e_p = _relmax(logits, ref_logits), _relmax(prob, ref_prob)
    tol_l = min(1e-2, 2 * _relmax(today_logits, ref_logits) + 1e-3)
    tol_p = min(1e-2, 2 * _relmax(today_prob, ref_prob) + 1e-3)
    assert e_p <= tol_p, (e_p, tol_p)
    assert e_l <= tol_l, (e_l, tol_l)
    # the restatement with switches reproduces the oracle, and each cut lies far outside the tolerance
    assert _relmax(_reg_eval64(sd, cv), ref_logits) < 1e-9
    _, batch_logits = ps.reg_forward(dict(sd), cv, train_bn=True, return_logits=True)
    cuts = {"batch statistics": batch_logits, "BN_1 / BN_2 swapped": _reg_eval64(sd, cv, swap12=True),
            "y0 skip dropped": _reg_eval64(sd, cv, drop_y0=True), "deconv_2_0 window unshifted": _reg_eval64(sd, cv, unshift_dc2=True)}
    for what, cut in cuts.items():
        # at cfg1 the shifted window moves deconv_2_0's box by (48, 32, 40) voxels inside a volume 2.3x that size; through
        # deconv_1_0 and the y0 skip it reaches the logits at 2.7x the tolerance (B200): that cut is held to 2x there
        factor = 2 if (name == "cfg1" and what == "deconv_2_0 window unshifted") else 10
        assert _relmax(logits, cut) >= factor * tol_l, what


def _model_case(B, V, H, W, D, seed=0):
    torch.manual_seed(seed)
    m = harness.MVSNet(D, 480.0 / D).to(DEV)
    K, R, T = harness.synthetic_cameras(B, V, H // 4, W // 4, seed=seed)
    gen = torch.Generator().manual_seed(seed + 1)
    img = torch.randn(B * V, 3, H, W, generator=gen).to(DEV)
    d_min, d_int = torch.full((B, 1, 1, 1), 425.0), torch.ones(B, 1, 1, 1)
    m.train()
    with torch.no_grad():
        for _ in range(3):
            m(img, K, R, T, d_min, d_int, B, V)
    _perturb_running_stats(m, seed + 5)
    return m.eval(), img, K, R, T, d_min, d_int


def test_encoder_and_refinement_against_fp64():
    m, img, K, R, T, d_min, d_int = _model_case(1, 3, 96, 128, 16)
    fz = mvs_b200.FrozenMVSNet(m)
    enc64 = copy.deepcopy(m.feature_encoder).double()
    with torch.no_grad():
        ref = enc64(img.double())
        today = nets2d.encode_features(m.feature_encoder, img).double()
    err, err_today = _relmax(fz.encode(img), ref), _relmax(today, ref)
    assert err <= 2 * err_today + 0.01, (err, err_today)
    # refinement on an initial depth map inside the sweep
    B, V = 1, 3
    span = torch.full((B, 1, 1, 1), 480.0, device=DEV)
    d0 = d_min.to(DEV)
    initial = d0 + span * torch.rand(B, 1, 24, 32, device=DEV)
    ref64 = copy.deepcopy(m.depthmap_refine).double()
    with torch.no_grad():
        norm = (initial.double() - d0.double()) / span.double()
        ref_img = F.interpolate(img[::V].double(), (24, 32), mode="bilinear", align_corners=False)
        ref_r = ref64(torch.cat((norm, ref_img), 1)) * span.double() + d0.double()
        today_r = refine.refine_spans(m.depthmap_refine, initial, img, V, d0, span)
    err = float(((fz.refine(initial, img, V, d0, span) - ref_r) / span).abs().max())
    err_today = float(((today_r - ref_r) / span).abs().max())
    assert err <= 2 * err_today + 0.01, (err, err_today)


def test_whole_model_against_fp64_and_leaves_the_module_untouched(monkeypatch):
    import plane_sweep as ps
    B, V, H, W, D = 1, 3, 96, 128, 16
    m, img, K, R, T, d_min, d_int = _model_case(B, V, H, W, D)
    before = {k: v.clone() for k, v in m.state_dict().items()}
    fz = mvs_b200.FrozenMVSNet(m)
    initial, refined = fz(img, K, R, T, d_min, d_int, B, V)
    # the same chain step by step: the frozen model's probability volume and the one of today's eval path
    feats = fz.encode(img).float()
    warped, d_batch, _ = mvs_b200.homography_warping(K, R, T, d_min, d_int, feats, B, V, D, 480.0 / D)
    cost = mvs_b200.assemble_cost_volume(warped, V, torch.bfloat16)
    prob = fz.regularise(cost)
    assert torch.equal(mvs_b200.extract_depth_map(prob, d_batch), initial)
    with torch.no_grad():
        feats64 = copy.deepcopy(m.feature_encoder).double()(img.double())
        w64, _, _ = mvs_b200.homography_warping(K, R, T, d_min, d_int, feats64.float(), B, V, D, 480.0 / D)
        cost64 = mvs_b200.assemble_cost_volume(w64, V, torch.float32).double()
        t_feats = m.encode(img).float()
        t_w, _, _ = mvs_b200.homography_warping(K, R, T, d_min, d_int, t_feats, B, V, D, 480.0 / D)
        today_prob = m.cost_volume_reg(mvs_b200.assemble_cost_volume(t_w, V, torch.bfloat16))
    sd = {k: v.double() if v.is_floating_point() else v for k, v in m.cost_volume_reg.state_dict().items()}
    ref_prob = ps.reg_forward(sd, cost64, train_bn=False)
    err, err_today = _relmax(prob, ref_prob), _relmax(today_prob, ref_prob)
    assert err <= min(1e-2, 2 * err_today + 1e-3), (err, err_today)
    # depth only where the reference's kept set survives the perturbation (DESIGN §2)
    pn = ref_prob.cpu().numpy()
    ref_depth, _ = ps.extract_depth(pn, d_batch.cpu().numpy())
    stable = ps.rank_margin(pn) > 4e-2
    if stable.any():
        assert float(np.abs(initial.cpu().numpy() - ref_depth)[:, 0][stable].max()) < 0.005 * 480.0
    # the module is only read
    assert not m.training
    for k, v in m.state_dict().items():
        assert torch.equal(v, before[k]), k
    # no library convolution or BatchNorm is left
    for name in ("conv2d", "conv3d", "conv_transpose3d", "batch_norm"):
        monkeypatch.setattr(F, name, lambda *a, _n=name, **k: (_ for _ in ()).throw(AssertionError(f"F.{_n} called")))
    n0 = mvs_b200.launch_count()
    i2, r2 = fz(img, K, R, T, d_min, d_int, B, V)
    assert torch.equal(i2, initial) and torch.equal(r2, refined) and mvs_b200.launch_count() > n0


def test_zero_depth_sweep_gives_the_nonfinite_pattern_of_the_eval_path():
    B, V, H, W, D = 1, 3, 64, 80, 8
    m, img, K, R, T, _, d_int = _model_case(B, V, H, W, D)
    d_min = torch.zeros(B, 1, 1, 1)                                    # validate.py sweeps from d_min = 0, d_int = 1
    fz = mvs_b200.FrozenMVSNet(m)
    i_f, r_f = fz(img, K, R, T, d_min, d_int, B, V)
    with torch.no_grad():
        i_t, r_t = m(img, K, R, T, d_min, d_int, B, V)
    assert torch.equal(torch.isfinite(i_f), torch.isfinite(i_t))
    assert torch.equal(torch.isfinite(r_f), torch.isfinite(r_t))


def test_graph_replay_and_refresh_are_bit_exact():
    B, V, H, W, D = 1, 3, 96, 128, 16
    m, img, K, R, T, d_min, d_int = _model_case(B, V, H, W, D)
    fz = mvs_b200.FrozenMVSNet(m)
    ginf = harness.GraphedInference(fz, B, V, H, W, DEV, warmup=1)
    for seed, d0 in ((1, 425.0), (2, 500.0), (3, 425.0)):
        Kb, Rb, Tb = harness.synthetic_cameras(B, V, H // 4, W // 4, seed=seed)
        im = torch.randn(B * V, 3, H, W, generator=torch.Generator().manual_seed(seed)).to(DEV)
        dm = torch.full((B, 1, 1, 1), d0)
        gi, gr = ginf.run(im, Kb, Rb, Tb, dm, d_int)
        ei, er = fz(im, Kb, Rb, Tb, dm, d_int, B, V)
        assert torch.equal(gi, ei) and torch.equal(gr, er)
    # a train step on the bound module, refresh(), replay of the SAME graph == a freshly built frozen model
    m.train()
    opt = torch.optim.SGD(m.parameters(), lr=1e-2)
    i0, r0 = m(img, K, R, T, d_min, d_int, B, V)
    (i0.mean() + r0.mean()).backward()
    opt.step()
    m.eval()
    fz.refresh()
    gi, gr = ginf.run(img, K, R, T, d_min, d_int)
    fi, fr = mvs_b200.FrozenMVSNet(m)(img, K, R, T, d_min, d_int, B, V)
    assert torch.equal(gi, fi) and torch.equal(gr, fr)


def test_refuses_cpu_tensors_and_bad_image_sizes():
    B, V, D = 1, 3, 8
    m = harness.MVSNet(D, 60.0).to(DEV).eval()
    fz = mvs_b200.FrozenMVSNet(m)
    K, R, T = harness.synthetic_cameras(B, V, 16, 20)
    d_min, d_int = torch.full((B, 1, 1, 1), 425.0), torch.ones(B, 1, 1, 1)
    with pytest.raises(mvs_b200.MvsB200Error, match="CPU"):
        fz(torch.randn(B * V, 3, 64, 80), K, R, T, d_min, d_int, B, V)
    for H, W in ((62, 80), (8, 80)):
        with pytest.raises(mvs_b200.MvsB200Error, match="multiples of 4"):
            fz(torch.randn(B * V, 3, H, W, device=DEV), K, R, T, d_min, d_int, B, V)
