"""The drop-in boundary (SURVEY §8b): dropin/{homography,costvolume,depthmap}.py carry the reference's module names, function
names and signatures (scripts/homography.py:6-14, costvolume.py:3, depthmap.py:4) and read the host application's `config`
at call time, as `model.py:5-7` expects.  CPU: names, signatures, refusal to run without CUDA.  GPU: the call sequence of
MVSNet.forward (model.py:177-187) through the drop-in modules on the golden inputs of the unmodified reference."""
import importlib
import inspect
import os
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DROPIN = os.path.join(ROOT, "deep-multiview-depth-estimation_b200", "dropin")
REFERENCE = {   # as written in the reference (SURVEY §8b)
    "homography": ("homography_warping", ["K_batch", "R_batch", "T_batch", "d_min", "d_int", "feature_maps", "batch_size",
                                          "n_views", "d_num"]),
    "costvolume": ("assemble_cost_volume", ["warped_feature_maps", "n_views"]),
    "depthmap": ("extract_depth_map", ["prob_volume", "d_batch"]),
    "loss": ("loss_fcn", ["gt", "initial", "refined"]),                      # SURVEY §8 row f3 (scripts/loss.py:4)
}


def _import_dropins(d_num=8, d_scale=60, n_est=5):
    cfg = types.ModuleType("config")               # what the host application's scripts/config.py provides (config.py:6-9,24)
    cfg.D_NUM, cfg.D_SCALE, cfg.N_DEPTH_EST = d_num, d_scale, torch.tensor(n_est)
    cfg.DEVICE = torch.device("cuda:0" if torch.cuda.is_available() else "cpu")
    sys.modules["config"] = cfg
    if DROPIN not in sys.path:
        sys.path.insert(0, DROPIN)
    mods = {}
    for name in REFERENCE:
        sys.modules.pop(name, None)
        mods[name] = importlib.import_module(name)
        assert os.path.dirname(os.path.abspath(mods[name].__file__)) == DROPIN
    return mods


def test_names_and_signatures_match_the_reference():
    mods = _import_dropins()
    for mod, (fn, params) in REFERENCE.items():
        f = getattr(mods[mod], fn)
        assert list(inspect.signature(f).parameters) == params, (mod, fn)
    import mvs_b200
    sd = mvs_b200.CostVolumeReg(device="cpu").state_dict()
    assert {"conv_0_0.weight", "deconv_3_0.weight", "conv_out.weight", "BN_3.running_var", "BN_0.num_batches_tracked"} <= set(sd)


def test_cpu_tensors_are_refused_not_computed_on_a_fallback():
    import mvs_b200
    mods = _import_dropins()
    K = torch.eye(3).repeat(3, 1, 1); R = torch.eye(3).repeat(3, 1, 1); T = torch.zeros(3, 3, 1)
    d_min, d_int = torch.full((1, 1, 1, 1), 425.0), torch.ones(1, 1, 1, 1)
    with pytest.raises(mvs_b200.MvsB200Error):
        warped, _, _ = mods["homography"].homography_warping(K, R, T, d_min, d_int, torch.zeros(3, 32, 8, 8), 1, 3)
        mods["costvolume"].assemble_cost_volume(warped, 3)
    with pytest.raises(mvs_b200.MvsB200Error):
        mods["depthmap"].extract_depth_map(torch.zeros(1, 1, 8, 8, 8), torch.zeros(1, 8, 1, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiny_b1v3", "b2v3"])
def test_mvsnet_forward_sequence_through_the_dropins(golden_dir, name, monkeypatch):
    import mvs_b200
    import plane_sweep as ps
    g = dict(np.load(os.path.join(golden_dir, name + ".npz")))
    t = lambda a: torch.from_numpy(np.asarray(a))
    B, V, D = int(g["B"]), int(g["V"]), int(g["D"])
    mods = _import_dropins(d_num=D, d_scale=int(g["d_scale"]))
    feat = t(g["feat"]).to("cuda:0").requires_grad_(True)
    # model.py:177-187: warp -> cost volume -> regulariser -> depth, D_NUM taken from config (d_num left at its default)
    warped, d_batch, ref_idx = mods["homography"].homography_warping(t(g["K"]), t(g["R"]), t(g["T"]), t(g["d_min"]), t(g["d_int"]),
                                                                      feat, B, V)
    assert tuple(warped.shape) == (B * V, 32, D) + tuple(feat.shape[-2:]) and d_batch.is_cuda
    assert ref_idx.dtype == torch.int64 and not ref_idx.is_cuda and ref_idx.tolist() == list(range(0, B * V, V))
    cost = mods["costvolume"].assemble_cost_volume(warped, V)
    assert float((cost.detach().cpu() - t(g["cost"])).abs().max() / t(g["cost"]).abs().max()) < 1e-4
    reg = mvs_b200.CostVolumeReg(device="cuda:0", precision="fp32").train()
    w0 = np.load(os.path.join(golden_dir, "reg_weights.npz"))
    reg.load_state_dict({k: t(v).to("cuda:0") for k, v in w0.items()})
    prob = reg(cost)
    depth = mods["depthmap"].extract_depth_map(prob, d_batch)
    ok = ~ps.tie_pixels(g["prob"])
    step = float(g["d_scale"]) * float(np.asarray(g["d_int"]).reshape(-1)[0])
    assert np.abs(depth.detach().cpu().numpy()[:, 0] - g["depth"][:, 0])[ok].max() < 0.005 * step
    depth.sum().backward()
    assert feat.grad is not None and bool(torch.isfinite(feat.grad).all())
