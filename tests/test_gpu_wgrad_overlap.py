"""Weight gradients on the side stream (ops.wgrad_fork): the train step's .grads are those of the single-stream backward, they
accumulate across backward() calls, they are complete on the current stream when backward() returns, and the forked step
replays from a CUDA graph -- two replays back to back -- with the eager step's results."""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu

B, V, H, W, D = 1, 3, 96, 128, 16


def _batch(seed):
    import plane_sweep as ps
    g = torch.Generator().manual_seed(seed)
    K, R, T = ps.synthetic_cameras(B, V, H // 4, W // 4, seed=seed)
    d_min, d_int = torch.full((B, 1, 1, 1), 425.0), torch.ones(B, 1, 1, 1)
    img = torch.randn(B * V, 3, H, W, generator=g).pin_memory()
    gt = (425.0 + 480.0 * torch.rand(B, 1, H // 4, W // 4, generator=g)).pin_memory()
    return img, gt, K, R, T, d_min, d_int


@pytest.fixture(scope="module")
def model():
    from mvs_b200.harness import MVSNet
    torch.manual_seed(0)
    return MVSNet(D, 480.0 / D, precision="bf16").to("cuda:0").train()


def _forward(model, seed):
    from mvs_b200.harness import loss_fcn
    img, gt, K, R, T, d_min, d_int = _batch(seed)
    initial, refined = model(img.cuda(), K, R, T, d_min, d_int, B, V)
    return loss_fcn(gt.cuda(), initial, refined)[0]


def _grads(model):
    return {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}


def _worst(a, b):
    assert a.keys() == b.keys()
    return max(float((a[n] - b[n]).abs().max() / (b[n].abs().max() + 1e-12)) for n in a)


def test_forked_grads_equal_single_stream_and_accumulate(model, monkeypatch):
    from mvs_b200 import ops
    joined = []
    join = ops._join
    monkeypatch.setattr(ops, "_join", lambda task: (joined.append(len(ops._PENDING[task])), join(task)))
    model.zero_grad(set_to_none=True)
    loss = _forward(model, 1)                  # one forward, three backwards: only the backward differs between the runs
    monkeypatch.setattr(ops, "WGRAD_FORK", False)
    loss.backward(retain_graph=True)
    torch.cuda.synchronize()
    assert joined == []
    single = _grads(model)
    model.zero_grad(set_to_none=True)
    loss.backward(retain_graph=True)
    torch.cuda.synchronize()
    noise = _worst(_grads(model), single)      # the single-stream backward against itself: fp32 atomics' order
    model.zero_grad(set_to_none=True)
    monkeypatch.setattr(ops, "WGRAD_FORK", True)
    loss.backward(retain_graph=True)
    # the join: once the current stream reaches the point where backward() returned, the side stream has finished
    done = torch.cuda.Event()
    done.record()
    done.synchronize()
    assert ops._side_stream(torch.device("cuda:0")).query()
    # every weight gradient of the regulariser, the 2D networks and the output convolution went through the side stream
    assert len(joined) == 1 and joined[0] >= 12, joined
    forked = _grads(model)
    assert all(n in forked for n, p in model.named_parameters() if p.requires_grad)
    assert _worst(forked, single) <= max(4 * noise, 1e-3), (noise, _worst(forked, single))
    # a second backward without zero_grad adds to .grad, as AccumulateGrad does
    loss.backward()
    torch.cuda.synchronize()
    twice = _grads(model)
    assert _worst(twice, {n: 2 * g for n, g in single.items()}) <= max(4 * noise, 1e-3)
    model.zero_grad(set_to_none=True)


def test_forked_grads_with_autograd_grad_stay_returned(model):
    """torch.autograd.grad captures the weight gradients instead of accumulating them: the nodes do not fork there."""
    from mvs_b200 import ops
    model.zero_grad(set_to_none=True)
    w = model.cost_volume_reg.conv_0_0.weight
    (g,) = torch.autograd.grad(_forward(model, 2), [w])
    assert g is not None and float(g.abs().max()) > 0 and w.grad is None
    assert not ops._PENDING


def test_graphed_forked_step_equals_eager(model):
    from mvs_b200 import ops
    from mvs_b200.harness import GraphedTrainStep
    twin = copy.deepcopy(model)
    gstep = GraphedTrainStep(model, B, V, H, W, torch.device("cuda:0"))
    seeds = (3, 4)
    assert gstep.run(*_batch(seeds[0])) is not None
    first = [t.clone() for t in gstep.depth] + [gstep.loss.clone()]
    for seed in seeds:                       # two replays back to back: no host synchronisation in between
        gstep.run(*_batch(seed))
        if seed == seeds[0]:
            rerun = [t.clone() for t in gstep.depth] + [gstep.loss.clone()]
    torch.cuda.synchronize()
    assert gstep.launches > 20
    graphed = _grads(model)
    twin.load_state_dict(model.state_dict())
    twin.zero_grad(set_to_none=True)
    _forward(twin, seeds[-1]).backward()
    torch.cuda.synchronize()
    assert not ops._PENDING
    # the rank-based depth extraction can flip a rank between two forwards (reordered atomic sums): a few percent, as
    # test_gpu_graph allows between a replay and an eager step
    assert _worst(graphed, _grads(twin)) < 0.15
    for a, b in zip(first, rerun):
        assert float((a - b).abs().max()) <= 0.05 * float(b.abs().max()) + 1e-3
    gstep.release()
