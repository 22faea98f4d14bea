"""Measurement harness around the hot path: the reference's MVSNet wiring, module shells and training step so that bench.py can
time a whole forward / train step on synthetic DTU-shaped data.  FeatureEncoder / DepthRefinement are the reference's Sequentials
(/root/reference/scripts/model.py:22-65, :129-152; same state_dict keys); on the bf16 path with train-mode BatchNorm their
layers run on the library's kernels (SURVEY §8 rows f1 / f2: mvs_b200/nets2d.py, mvs_b200/refine.py), otherwise as the stock
torch modules they are.  Glue: model.py:168-207; loss: scripts/loss.py:4-41 (row f3, ops.masked_l1_loss).
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import api, nets2d, refine
from .regulariser import CostVolumeReg


class BatchNormReLU2d(nn.BatchNorm2d):
    """BatchNorm2d followed by ReLU (model.py:236-247 pairs).  Train mode on the GPU: the fused channel-last statistics /
    apply / backward kernels of libmvs_b200.so (K3b) on the [N*H*W, C] rows of the map (ATen's channels-last bf16 BatchNorm
    takes ~2x as long per pass and a separate ReLU pass); otherwise stock torch.  Same parameters and buffers as
    nn.BatchNorm2d (state_dict-compatible with the BatchNorm2d + ReLU pair of the reference)."""

    def forward(self, x):
        if x.is_cuda and self.training and self.num_features in (8, 16, 32, 64) and x.dtype in (torch.float32, torch.bfloat16):
            from . import ops
            y, _, _ = ops.batchnorm_relu_train(x.unsqueeze(2), self.weight, self.bias, self.eps, relu=True,
                                               running=(self.running_mean, self.running_var, self.num_batches_tracked),
                                               momentum=self.momentum)
            return y.squeeze(2)
        return F.relu(super().forward(x))


def _conv_bn_relu(i, o, k, s):
    # Identity keeps the module indices (state_dict keys) of the reference's Conv2d / BatchNorm2d / ReLU triples
    return [nn.Conv2d(i, o, k, stride=s, padding=k // 2, bias=False), BatchNormReLU2d(o), nn.Identity()]


class FeatureEncoder(nn.Module):
    """[N,3,H,W] -> [N,32,H/4,W/4]: 3-3-5(s2)-3-3-5(s2)-3-3 convs, 8/16/32 channels, no BN/ReLU on the last."""

    def __init__(self, in_ch=3, base=8):
        super().__init__()
        c1, c2, c3 = base, base * 2, base * 4
        layers = (_conv_bn_relu(in_ch, c1, 3, 1) + _conv_bn_relu(c1, c1, 3, 1) + _conv_bn_relu(c1, c2, 5, 2)
                  + _conv_bn_relu(c2, c2, 3, 1) + _conv_bn_relu(c2, c2, 3, 1) + _conv_bn_relu(c2, c3, 5, 2)
                  + _conv_bn_relu(c3, c3, 3, 1) + [nn.Conv2d(c3, c3, 3, padding=1, bias=False)])
        self.model = nn.Sequential(*layers)

    def forward(self, x):
        return self.model(x)


class DepthRefinement(nn.Module):
    """[B,4,h,w] (normalised depth + resized reference image) -> residual-refined normalised depth."""

    def __init__(self, in_ch=4, base=32):
        super().__init__()
        self.model = nn.Sequential(*(_conv_bn_relu(in_ch, base, 3, 1) + _conv_bn_relu(base, base, 3, 1)
                                     + _conv_bn_relu(base, base, 3, 1) + [nn.Conv2d(base, 1, 3, padding=1, bias=False)]))

    def forward(self, x):
        return self.model(x) + x[:, :1]


class MVSNet(nn.Module):
    """The reference's MVSNet wiring (model.py:168-207) around the mvs_b200 hot path."""

    def __init__(self, d_num, d_scale, precision="bf16", n_depth_est=5, conv_backend="auto"):
        super().__init__()
        self.d_num, self.d_scale, self.precision, self.n_depth_est = int(d_num), d_scale, precision, int(n_depth_est)
        self.feature_encoder = FeatureEncoder()
        self.cost_volume_reg = CostVolumeReg(precision=precision, conv_backend=conv_backend, n_depth_est=n_depth_est)
        self.depthmap_refine = DepthRefinement()

    def forward(self, nn_input, K_batch, R_batch, T_batch, d_min, d_int, batch_size, n_views, sweep=None):
        """sweep: an ops.PlaneSweep already holding this batch's geometry on the device (PlaneSweep.update); the cameras are
        then not touched here and d_min / d_int should be device tensors -- the form a captured CUDA graph replays."""
        feats = self.encode(nn_input)
        feats = feats.float()
        ev = getattr(self, "after_encoder_event", None)          # GraphedInference: where the next batch's H2D copy may start
        if ev is not None and torch.cuda.is_current_stream_capturing():
            ev.record()
        warped, d_batch, ref_views = api.homography_warping(K_batch, R_batch, T_batch, d_min, d_int, feats,
                                                            batch_size, n_views, self.d_num, self.d_scale, sweep=sweep)
        vol_dtype = torch.bfloat16 if self.precision == "bf16" else torch.float32
        cost = api.assemble_cost_volume(warped, n_views, vol_dtype)
        prob = self.cost_volume_reg(cost)
        initial = api.extract_depth_map(prob, d_batch, self.n_depth_est)
        return initial, refine.refine_depth(self.depthmap_refine, initial, nn_input, n_views, d_min, d_int, self.d_num, self.d_scale,
                                            bf16=self.precision == "bf16")

    def encode(self, nn_input):
        """model.py:20-65 -> feature maps [N, 32, H/4, W/4] (bf16 on the bf16 path).  SURVEY row f1: bf16 with train-mode BatchNorm
        (what train.py and test.py:61 run) takes the tensor-core kernels of mvs_b200/nets2d.py; MVSB200_ENCODER=torch, fp32 and
        eval-mode BatchNorm evaluate the module's stock torch layers (cuDNN)."""
        return nets2d.encode_features(self.feature_encoder, nn_input, bf16=self.precision == "bf16")

    def refine(self, initial, nn_input, n_views, d_trans, d_span):
        """model.py:190-205 on depth offsets / spans already on the device (SURVEY row f2; mvs_b200/refine.py): native on the
        bf16 path with train-mode BatchNorm (what train.py and test.py:61 run), the stock torch layers otherwise."""
        return refine.refine_spans(self.depthmap_refine, initial, nn_input, n_views, d_trans, d_span, bf16=self.precision == "bf16")


def _snapshot(tensors):
    return [t.detach().clone() for t in tensors]


def _restore(tensors, saved):
    with torch.no_grad():
        for t, s in zip(tensors, saved):
            t.copy_(s)


class GraphedTrainStep:
    """One MVSNet training step (train.py:93-108: forward, loss, backward -- and, when given, the data-parallel gradient
    all-reduce and the optimiser step) captured as ONE CUDA graph: the step is ~800 kernel launches of a few microseconds to a
    few hundred, which eager PyTorch cannot issue fast enough to keep a B200 busy.  Static device buffers hold the step's inputs
    (images, ground truth, sweep geometry); `run` copies the new batch into them (asynchronously, from pinned host memory or
    device tensors) and replays the graph.

    reducer (FlatGradAllReduce) and optimizer are optional.  With a reducer every parameter's .grad is a VIEW into the reducer's
    flat bucket (no pack / unpack copies): the graph zeroes the bucket, backward accumulates into the views, ONE all-reduce
    (NCCL work is capturable) and one scale average it, all inside the replay.  With an optimizer (torch.optim.Adam(fused=True,
    capturable=True)) its step is the last node of the graph; otherwise the caller steps after run().

    The warm-up passes that precede the capture (lazy workspaces, library plans) run on real data; BatchNorm buffers,
    parameters and optimiser state are restored afterwards, so the first replay starts from the state the caller handed in --
    an eager step and the graphed step see the same running statistics.
    Shapes are fixed per instance, as in the reference's loaders (fixed resolution, batch and view count)."""

    def __init__(self, model: "MVSNet", batch_size, n_views, H, W, device, warmup=3, reducer=None, optimizer=None):
        from . import ops, _lib
        self.model, self.B, self.V = model, batch_size, n_views
        h, w = H // 4, W // 4
        self.img = torch.zeros(batch_size * n_views, 3, H, W, device=device)
        self.gt = torch.ones(batch_size, 1, h, w, device=device)
        self.d_min = torch.zeros(batch_size, 1, 1, 1, device=device)
        self.d_int = torch.ones(batch_size, 1, 1, 1, device=device)
        self.sweep = None
        self.dims = (h, w)
        self.graph, self.loss, self.depth, self.launches = None, None, None, 0
        self.warmup, self._lib = warmup, _lib
        self.params = [p for p in model.parameters() if p.requires_grad]
        self.reducer, self.optimizer = reducer, optimizer
        # recorded INSIDE the replay, between forward and backward (an external event node of the graph): a loader stream that
        # waits on it places the next batch's host-to-device copy under the regulariser's long kernels instead of under the many
        # short launches at the start of a step, which a saturated PCIe link delays (bench.py, host-fed loop)
        try:
            self.mid_event = torch.cuda.Event(external=True)
        except TypeError:                                  # older torch: no external events
            self.mid_event = None
        if reducer is not None:
            reducer.attach_grads()                         # .grad of every parameter := view into the flat bucket

    def _load(self, img, gt, K, R, T, d_min, d_int):
        from . import ops
        if self.sweep is None:
            self.sweep = ops.PlaneSweep(K, R, T, d_min, d_int, self.B, self.V, self.model.d_num, self.model.d_scale,
                                        self.dims[0], self.dims[1], self.img.device)
        else:
            self.sweep.update(K, R, T, d_min, d_int)
        self.img.copy_(img, non_blocking=True)
        self.gt.copy_(gt, non_blocking=True)
        self.d_min.copy_(d_min, non_blocking=True)
        self.d_int.copy_(d_int, non_blocking=True)

    def _zero_grads(self):
        if self.reducer is not None:
            self.reducer.bucket.zero_()                    # one memset; the .grad views stay attached
        else:
            for p in self.params:
                p.grad = None

    def _fwd_bwd(self):
        if self.reducer is not None:
            self.reducer.bucket.zero_()
        initial, refined = self.model(self.img, None, None, None, self.d_min, self.d_int, self.B, self.V, sweep=self.sweep)
        loss, _, _ = loss_fcn(self.gt, initial, refined)
        if self.mid_event is not None and torch.cuda.is_current_stream_capturing():
            self.mid_event.record()
        loss.backward()
        if self.reducer is not None:
            self.reducer.reduce_attached()                 # all-reduce + average of the flat bucket, in place
        if self.optimizer is not None:
            self.optimizer.step()
        return loss.detach(), (initial.detach(), refined.detach())

    def _optimizer_state_tensors(self):
        out = []
        if self.optimizer is not None:
            for st in self.optimizer.state.values():
                out += [v for v in st.values() if torch.is_tensor(v)]
        return out

    def run(self, img, gt, K, R, T, d_min, d_int):
        """-> loss (device scalar, valid after the current stream reaches this point); gradients in .grad, the step's
        (initial, refined) depth maps in .depth."""
        self._load(img, gt, K, R, T, d_min, d_int)
        if self.graph is None:
            buffers = list(self.model.buffers())
            keep = _snapshot(buffers + (self.params if self.optimizer is not None else []))
            opt_fresh = self.optimizer is not None and len(self.optimizer.state) == 0
            opt_keep = _snapshot(self._optimizer_state_tensors())
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):                  # warm-up off the capture: lazy workspaces, cuDNN plans, autotune
                for _ in range(self.warmup):
                    if self.reducer is None:
                        self._zero_grads()
                    self._fwd_bwd()
                # undo what the warm-up passes did to the training state (BatchNorm running statistics, weights, moments)
                _restore(buffers + (self.params if self.optimizer is not None else []), keep)
                if opt_fresh:
                    with torch.no_grad():
                        for t in self._optimizer_state_tensors():
                            t.zero_()                      # state tensors were created by the warm-up: back to step 0, in place
                else:
                    _restore(self._optimizer_state_tensors(), opt_keep)
            torch.cuda.current_stream().wait_stream(side)
            if self.reducer is None:
                self._zero_grads()
            n0 = self._lib.launch_count()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.loss, self.depth = self._fwd_bwd()
            self.launches = self._lib.launch_count() - n0   # libmvs_b200.so launches recorded in the graph
            self.graph = g
        self.graph.replay()
        return self.loss

    def release(self):
        """Drop the captured graph (with a reducer it holds NCCL work: do this before destroy_process_group())."""
        self.graph, self.loss, self.depth = None, None, None
        torch.cuda.synchronize()


class GraphedInference:
    """MVSNet.forward under torch.no_grad() (test.py:86-92) replayed as ONE CUDA graph for a fixed input shape: static image /
    geometry buffers re-filled per call (`PlaneSweep.update`), ~250 kernel launches per depth map issued by one graph launch."""

    def __init__(self, model: "MVSNet", batch_size, n_views, H, W, device, warmup=2):
        self.model, self.B, self.V, self.warmup = model, batch_size, n_views, warmup
        self.img = torch.zeros(batch_size * n_views, 3, H, W, device=device)
        self.d_min = torch.zeros(batch_size, 1, 1, 1, device=device)
        self.d_int = torch.ones(batch_size, 1, 1, 1, device=device)
        self.dims = (H // 4, W // 4)
        self.sweep, self.graph, self.out, self.launches = None, None, None, 0
        try:        # external event recorded inside the replay after the 2D encoder (see GraphedTrainStep.mid_event)
            self.mid_event = torch.cuda.Event(external=True)
        except TypeError:
            self.mid_event = None

    @torch.no_grad()
    def _fwd(self):
        self.model.after_encoder_event = self.mid_event
        try:
            return self.model(self.img, None, None, None, self.d_min, self.d_int, self.B, self.V, sweep=self.sweep)
        finally:
            self.model.after_encoder_event = None

    @torch.no_grad()
    def run(self, img, K, R, T, d_min, d_int):
        from . import ops
        if self.sweep is None:
            self.sweep = ops.PlaneSweep(K, R, T, d_min, d_int, self.B, self.V, self.model.d_num, self.model.d_scale,
                                        self.dims[0], self.dims[1], self.img.device)
        else:
            self.sweep.update(K, R, T, d_min, d_int)
        self.img.copy_(img, non_blocking=True)
        self.d_min.copy_(d_min, non_blocking=True)
        self.d_int.copy_(d_int, non_blocking=True)
        if self.graph is None:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(self.warmup):
                    self._fwd()
            torch.cuda.current_stream().wait_stream(side)
            from . import _lib
            n0 = _lib.launch_count()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.out = self._fwd()
            self.launches = _lib.launch_count() - n0       # libmvs_b200.so launches recorded in the graph
            self.graph = g
        self.graph.replay()
        return self.out


class DepthSlabMVSNet:
    """Inference of ONE multi-view sample across the ranks of a box (BASELINE.json configs[3]): the hot path runs on depth
    slabs (mvs_b200.depth_slab), the out-of-scope 2D nets are replicated.  Each view is encoded by ONE rank
    (view v on rank v mod R) and broadcast -- every rank needs all V feature maps (75.8 MB at 5 x 400x296x32) for the sweep
    of its planes.  Wraps an MVSNet whose parameters are identical on every rank."""

    def __init__(self, model: "MVSNet", comm=None, graph=False):
        """graph: replay the rank's whole forward (2D nets, sharded hot path, NCCL exchanges) as one CUDA graph (fixed shapes);
        call release() before destroying the process group."""
        from .depth_slab import DepthSlabCostVolumeReg, TorchDistComm
        self.model = model
        self.comm = TorchDistComm() if comm is None else comm
        self.reg = DepthSlabCostVolumeReg(model.cost_volume_reg, self.comm)
        self.use_graph, self._graphed, self._sweep, self._out = bool(graph), None, None, None
        self.launches = 0
        try:
            self.mid_event = torch.cuda.Event(external=True) if graph else None
        except TypeError:
            self.mid_event = None

    def release(self):
        """Drop the captured graph (it holds NCCL work: do this before destroy_process_group())."""
        self._graphed, self._out = None, None
        torch.cuda.synchronize()

    @torch.no_grad()
    def encode(self, nn_input, by_view=None):
        """Feature maps of all views on every rank, [N,32,h,w] with channel-last memory.  by_view: view v is encoded on rank
        v mod R and broadcast; exact only when the encoder's BatchNorm uses running statistics (eval mode) -- in train mode
        (test.py:61) its batch statistics span all views, so the default then is to encode all views on every rank."""
        m, R, r = self.model, self.comm.world, self.comm.rank
        N, _, H, W = nn_input.shape
        amp = m.precision == "bf16" and nn_input.is_cuda
        if by_view is None:
            by_view = not m.feature_encoder.training
        if not by_view or R == 1:
            return m.encode(nn_input).float()
        nhwc = torch.empty((N, H // 4, W // 4, 32), dtype=torch.float32, device=nn_input.device)
        mine = [v for v in range(N) if v % R == r]
        if mine:
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
                f = m.feature_encoder(nn_input[mine].contiguous(memory_format=torch.channels_last))
            nhwc[mine] = f.float().permute(0, 2, 3, 1)
        for v in range(N):
            self.comm.broadcast(nhwc[v], v % R)
        return nhwc.permute(0, 3, 1, 2)

    def _pipeline(self, nn_input, sweep, d_trans, d_span):
        """encode -> slab sweep + slab regulariser + depth -> refinement, on geometry already resident on the device."""
        from .depth_slab import slab_cost_fn
        m = self.model
        feats = self.encode(nn_input)
        if self.mid_event is not None and torch.cuda.is_current_stream_capturing():
            self.mid_event.record()                              # where the next sample's H2D copy may start (bench.py)
        h, w = feats.shape[-2:]
        vol_dtype = torch.bfloat16 if m.precision == "bf16" else torch.float32
        initial, prob_rows, rows = self.reg.forward(slab_cost_fn(feats, sweep, vol_dtype), sweep.d_batch_dev, 1, m.d_num, h, w)
        return initial, m.refine(initial, nn_input, nn_input.shape[0], d_trans, d_span)      # replicated: 4-channel 400x296 maps

    @torch.no_grad()
    def forward(self, nn_input, K_batch, R_batch, T_batch, d_min, d_int, n_views):
        from . import ops
        m = self.model
        N, _, H, W = nn_input.shape
        h, w = H // 4, W // 4
        dev = nn_input.device
        if not self.use_graph:
            sweep = ops.PlaneSweep(K_batch, R_batch, T_batch, d_min, d_int, 1, n_views, m.d_num, m.d_scale, h, w, dev)
            return self._pipeline(nn_input, sweep, d_min.to(dev), d_int.to(dev) * m.d_num * m.d_scale)
        # the rank's WHOLE forward -- 2D nets, K1, slab regulariser, every NCCL exchange, K4 -- as one CUDA graph
        if self._sweep is None:
            self._sweep = ops.PlaneSweep(K_batch, R_batch, T_batch, d_min, d_int, 1, n_views, m.d_num, m.d_scale, h, w, dev)
            self._img = torch.zeros_like(nn_input)
            self._d_trans = torch.zeros(1, 1, 1, 1, device=dev)
            self._d_span = torch.ones(1, 1, 1, 1, device=dev)
        else:
            self._sweep.update(K_batch, R_batch, T_batch, d_min, d_int)
        self._img.copy_(nn_input, non_blocking=True)
        self._d_trans.copy_(d_min, non_blocking=True)
        self._d_span.copy_(d_int * (m.d_num * m.d_scale), non_blocking=True)
        if self._graphed is None:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):                       # lazy workspaces, NCCL connections, cuDNN plans -- outside the capture
                    self._pipeline(self._img, self._sweep, self._d_trans, self._d_span)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            from . import _lib
            g = torch.cuda.CUDAGraph()
            n0 = _lib.launch_count()
            with torch.cuda.graph(g):
                self._out = self._pipeline(self._img, self._sweep, self._d_trans, self._d_span)
            self.launches = _lib.launch_count() - n0       # libmvs_b200.so launches recorded in the graph (per replay)
            self._graphed = g
        self._graphed.replay()
        return self._out


# DTU cameras of SURVEY App. C (views = cams 0, 10, 1 of scripts/test_dataloader, K at the 160x128 feature resolution):
# the synthetic DTU-shaped geometry bench.py and the tools feed the path with.
_DTU_K = [[361.54126, 0.0, 82.90063], [0.0, 360.3975, 66.38387], [0.0, 0.0, 1.0]]
_DTU_R = [
    [[0.970263, 0.00748, 0.241939], [-0.014743, 0.999493, 0.028223], [-0.241605, -0.030951, 0.969881]],
    [[0.885052, -0.307962, 0.34906], [0.220575, 0.937798, 0.268109], [-0.409915, -0.160296, 0.897928]],
    [[0.802256, -0.439347, 0.404178], [0.427993, 0.895282, 0.123659], [-0.416183, 0.073779, 0.906283]],
]
_DTU_T = [[-191.02, 3.28832, 22.5401], [-258.497, -156.493, 71.838], [-291.419, -77.0495, 71.2762]]


def synthetic_cameras(batch_size, n_views, h=128, w=160, seed=0):
    """DTU-shaped cameras for synthetic batches: views 0..2 of a sample are the three DTU cameras above, further views and
    further batch items are small seeded perturbations of them (rotation of a few degrees about a random axis, a few
    millimetres of translation); K scaled from the 160x128 feature grid to (w, h).
    -> CPU fp32 K [N,3,3], R [N,3,3], T [N,3,1], N = batch_size * n_views, ordered b*V + v (data.py:272-274)."""
    import numpy as np
    rng = np.random.RandomState(seed)
    K = np.array(_DTU_K)
    K[0] *= w / 160.0
    K[1] *= h / 128.0
    Ks, Rs, Ts = [], [], []
    for b in range(batch_size):
        for v in range(n_views):
            R, T = np.array(_DTU_R[v % 3]), np.array(_DTU_T[v % 3])
            if v >= 3 or b > 0:
                axis = rng.randn(3)
                axis /= np.linalg.norm(axis)
                ang = 0.04 * rng.randn()
                X = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
                R = (np.eye(3) + np.sin(ang) * X + (1 - np.cos(ang)) * X @ X) @ R
                T = T + rng.randn(3) * 8.0
            Ks.append(K); Rs.append(R); Ts.append(T.reshape(3, 1))
    f = lambda a: torch.tensor(np.stack(a), dtype=torch.float32)
    return f(Ks), f(Rs), f(Ts)


def loss_fcn(gt, initial, refined):
    """Masked L1 on both depth maps (scripts/loss.py:4-41): returns (loss, initial MAE, refined MAE).  On the GPU: the fused
    kernels of libmvs_b200.so (ops.masked_l1_loss, one launch forward and one backward); the torch expression below is the
    reference's formula, kept for host tensors (the harness' CPU unit tests)."""
    if gt.is_cuda and initial.is_cuda and refined.is_cuda and gt.shape == initial.shape == refined.shape:
        from . import ops
        return ops.masked_l1_loss(gt, initial, refined)
    mask = (gt != 0).float()
    n_valid = mask.sum((1, 2, 3))
    l0 = (mask * (gt - initial).abs()).sum((1, 2, 3)) / n_valid
    l1 = (mask * (gt - refined).abs()).sum((1, 2, 3)) / n_valid
    return (l0 + l1).sum(), l0.mean(), l1.mean()


class FlatGradAllReduce:
    """Data-parallel gradient reduction for scene/batch sharding (SURVEY §8e): one flat fp32 bucket holding
    every gradient (1.53 MB for MVSNet), one all-reduce per step, averaged.  Works on any process group
    (NCCL on the GPUs, gloo in the CPU tests).  The reference has no distributed code; its parameters live in
    a plain list (model.py:164-166), so this takes a list, not a DDP-wrapped module."""

    def __init__(self, params, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.params = [p for p in params if p.requires_grad]
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        n = sum(p.numel() for p in self.params)
        dev = self.params[0].device
        self.bucket = torch.zeros(n, dtype=torch.float32, device=dev)
        self.attached = False
        self.views, o = [], 0
        for p in self.params:
            self.views.append(self.bucket[o:o + p.numel()].view_as(p))
            o += p.numel()

    def broadcast_parameters(self, buffers=()):
        if self.world == 1:
            return
        for t in list(self.params) + list(buffers):
            self.dist.broadcast(t.data if isinstance(t, nn.Parameter) else t, 0, group=self.group)

    def attach_grads(self):
        """.grad of every parameter becomes a view into the flat bucket: backward accumulates straight into it, the
        all-reduce needs no pack / unpack copies, and the whole reduction is capturable in a CUDA graph (static addresses)."""
        self.bucket.zero_()
        for p, v in zip(self.params, self.views):
            p.grad = v
        self.attached = True

    def reduce_attached(self):
        """After backward() with attached gradients: bucket <- mean over ranks, in place (one collective, one scale)."""
        if self.world == 1:
            return
        self.dist.all_reduce(self.bucket, group=self.group)
        self.bucket.mul_(1.0 / self.world)

    def reduce(self):
        """Call after backward(): grads <- mean over ranks."""
        if self.world == 1:
            return
        if self.attached and all(p.grad is v for p, v in zip(self.params, self.views)):
            return self.reduce_attached()
        for p, v in zip(self.params, self.views):
            if p.grad is None:
                v.zero_()
            else:
                v.copy_(p.grad)
        self.dist.all_reduce(self.bucket, group=self.group)
        self.bucket.div_(self.world)
        for p, v in zip(self.params, self.views):
            if p.grad is None:
                p.grad = v.clone()
            else:
                p.grad.copy_(v)
