#!/usr/bin/env python
"""bench.py -- headline measurement of the plane-sweep hot path (contract: see the task brief / DESIGN.md §5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg2|cfg1|cfg4] [--no-graph]
                    [--dump-outputs DIR]

Own arm: one "step" = one MVSNet train step (forward + loss + backward + gradient all-reduce + Adam) on one synthetic
DTU-shaped batch (BASELINE.json configs[1]: bf16, batch 4, 3 views, 640x512 input => 160x128x32 features, D = 192), replayed as
one CUDA graph (harness.GraphedTrainStep: the NCCL all-reduce of the flat gradient bucket and the fused Adam step are nodes of
the same graph; --no-graph issues it eagerly).  `value` is depth maps/s with the batch already resident in HBM;
`e2e` is the same step fed from pinned HOST buffers (H2D of the images, ground truth and sweep geometry, D2H read of the loss
inside the timed region).  `roofline` is the dominant own kernel (the stride-1 tcgen05 convolution, tensor bound),
`roofline_k1` / `roofline_k1_fp32` the fused warp+variance kernel (HBM bound), all timed live with CUDA events on the
launching stream.  Under torchrun (--gpus N): cfg2 shards by scene/batch with a flat-bucket NCCL gradient all-reduce (weak
scaling); cfg4 splits ONE sample into depth slabs across the ranks (strong scaling, mvs_b200.depth_slab).  The default line
(cfg2 at every N) carries two more measurements as extra keys so that the driver's SCALE file records them: `cfg4_depth_slab`
(BASELINE.json configs[3]: the depth-slab split over the N ranks, hot path and whole inference, graph-replayed) and, for N > 1,
`cfg3` (configs[2]: batch 8 per GPU); --no-extras skips them.

Reference arm (--impl reference): the oracle port of the reference's CPU algorithm (oracle/cpu_path.py) on the
host cores, each step a bounded sample of the same workload (stated in `cpu_baseline.sample`).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "deep-multiview-depth-estimation_b200"))

K1_NCU, K3_NCU = "r01_k1_fwd2_ncu.json", "r01_k3_kdn_ncu.json"      # committed ncu --set full captures (traffic)
_E2E_DIAG = int(os.environ.get("MVSB200_E2E_DIAG", "0"))   # diagnostics of the host-fed loop: 1 = no H2D prefetch, 2 = no loss read-back
TC_KERNELS = ("conv3d_s1_tc", "deconv3d_s2_tc", "conv3d_s2_tc", "conv3d_s1_wgrad_tc", "conv3d_s2_wgrad_tc")     # tcgen05 convolution kernels
TC2D_KERNELS = ("conv2d_tc", "conv2d_wgrad_tc")       # the same kernels on the 2D feature / refinement networks (rows f1 / f2): 2*9*Cin*Cout*pixels


def _family_2d(kern, tc_fl, tc_ms, tpeak):
    """The tcgen05 launches of the 2D networks (not part of the headline family: 3 GFLOP per view on 8..32 channels, bound by the
    count of tiny MMAs, DESIGN K6) and the figure over EVERY tcgen05 launch of the step."""
    fam2 = [n for n in TC2D_KERNELS if n in kern and "alg_flops_per_step" in kern[n]]
    if not fam2:
        return None
    ms2 = sum(kern[n]["ms_per_step"] for n in fam2)
    fl2 = sum(kern[n]["alg_flops_per_step"] for n in fam2)
    all_ms, all_fl = tc_ms + ms2, tc_fl + fl2
    return {"per_kernel": {n: {k_: kern[n][k_] for k_ in ("ms_per_step", "launches", "alg_flops_per_step", "TFLOPs", "frac")} for n in fam2},
            "alg_flops_per_step": fl2, "ms_per_step": ms2, "achieved": fl2 / (ms2 * 1e-3) / 1e12 if ms2 else None,
            "all_tcgen05_launches_of_the_step": {"alg_flops_per_step": all_fl, "ms_per_step": all_ms,
                                                 "achieved": all_fl / (all_ms * 1e-3) / 1e12 if all_ms else None,
                                                 "frac": all_fl / (all_ms * 1e-3) / 1e12 / tpeak if all_ms else None}}


WORKLOADS = {
    "cfg2": dict(B=4, V=3, H=512, W=640, D=192, train=True,
                 desc="MVSNet train step bf16, batch 4/GPU, 3 views, 640x512, D=192 (BASELINE.json configs[1])"),
    "cfg3": dict(B=8, V=3, H=512, W=640, D=192, train=True,
                 desc="MVSNet data-parallel train step bf16, batch 8/GPU, 3 views, 640x512, D=192 (BASELINE.json configs[2])"),
    "cfg1": dict(B=1, V=3, H=512, W=640, D=192, train=False,
                 desc="MVSNet forward, batch 1, 3 views, 640x512, D=192 (BASELINE.json configs[0])"),
    "cfg4": dict(B=1, V=5, H=1184, W=1600, D=256, train=False,
                 desc="MVSNet inference, 5 views, 1600x1184, D=256 on ONE GPU (BASELINE.json configs[3] without the depth-slab split)"),
}


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def _tensor_peak():
    """bf16 tensor peak for a kernel timed inside a long step: the sustained figure."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json, sustained cuBLAS bf16)"
    except Exception:
        return 1500.0, "fallback (B200_PROFILING.md)"


def _ncu_traffic(name):
    """DRAM bytes (read + write) of the committed `ncu --set full` capture of a kernel, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", name)) as f:
            m = json.load(f)["metrics"]
        return (float(m["dram__bytes_read.sum"]) + float(m["dram__bytes_write.sum"])) * 1e6
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=lambda: self.rows.extend(self.proc.stdout.readlines()), daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def run_reference(args, rank, world):
    """CPU arm: oracle port, bounded sample, all host threads.  Only rank 0 works."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch
    import cpu_path
    wl = WORKLOADS[args.workload]
    d_sample = 48
    torch.set_num_threads(os.cpu_count() or 1)
    s = cpu_path.make_sample(V=wl["V"], D=d_sample, h=wl["H"] // 4, w=wl["W"] // 4, d_total=wl["D"])
    for _ in range(args.warmup):
        cpu_path.hot_path_step(s, backward=wl["train"])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_path.hot_path_step(s, backward=wl["train"])
    dt = (time.perf_counter() - t0) / args.steps
    scale = wl["D"] / d_sample
    value = 1.0 / (dt * scale)
    sample = (f"hot path only (warp+variance+regulariser+depth, {'fwd+bwd' if wl['train'] else 'fwd'}), 1 batch item, "
              f"first {d_sample} of {wl['D']} planes at full 160x128x32; time scaled x{scale:g} linearly in D "
              f"(favours the CPU: the reference's torch.cat growth is super-linear in D)")
    line = {"impl": "reference", "metric": "depth maps/sec", "value": value, "unit": "depth maps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"]},
            "cpu_baseline": {"value": value, "unit": "depth maps/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": sample},
            "e2e": {"value": value, "unit": "depth maps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def _pin_rank_to_cores(local_rank, local_world):
    """Ranks of one box share the host: give each its own block of the cores this process may run on (torch intra-op threads,
    the fp64 geometry of every step and the H2D staging then do not fight over the same cores)."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        if local_world > 1 and len(cores) >= 2 * local_world:
            per = len(cores) // local_world
            mine = cores[local_rank * per:(local_rank + 1) * per]
            os.sched_setaffinity(0, mine)
            return len(mine)
        return len(cores)
    except (AttributeError, OSError):
        return os.cpu_count() or 1


def dump_outputs(out_dir, last, params):
    """What the last timed step handed its caller, as float32 DIR/<name>.npy: the loss, the initial and refined depth maps and,
    for a train step, the gradients (every parameter's, flattened and concatenated in model.parameters() order); at most a few
    MB at every workload.  The weights after the optimiser step are not written: Adam's first step moves each weight by about
    lr * sign(gradient), so float noise in a gradient near zero moves a weight by up to 2 lr."""
    import numpy as np
    import torch
    loss, initial, refined = last
    arrays = {"loss": loss.reshape(1), "initial_depth": initial, "refined_depth": refined}
    if params is not None:
        arrays["grads"] = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def run_b200(args, rank, world, local_rank, workload=None, light=False):
    """One workload on this rank.  light: an extra measurement riding on the default line (no per-kernel event pass, no clocks,
    no isolated K1 launches, fewer steps)."""
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the mvs_b200 path has no CPU fallback")
    import mvs_b200
    from mvs_b200 import ops
    from mvs_b200.harness import MVSNet, loss_fcn, FlatGradAllReduce, synthetic_cameras

    workload = workload or args.workload
    steps = max(3, args.steps // 2) if light else args.steps
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if os.environ.get("MVSB200_CUDNN_BENCHMARK", "1") == "1":
        torch.backends.cudnn.benchmark = True              # autotuned plans for whatever still reaches the library (MVSB200_ENCODER / _REFINE=torch A/B runs)
    wl = WORKLOADS[workload]
    B, V, H, W, D, train = wl["B"], wl["V"], wl["H"], wl["W"], wl["D"], wl["train"]
    h, w, C = H // 4, W // 4, 32
    d_scale = 480.0 / D
    torch.manual_seed(0)
    model = MVSNet(D, d_scale, precision="bf16").to(dev)
    model.train()                                          # train-mode BN also at test time (test.py:61)
    params = [p for p in model.parameters()]
    graphed = train and not args.no_graph
    # train.py:160 Adam(lr=0.005); fused = one multi-tensor kernel, capturable = its step is a node of the step's CUDA graph
    opt = torch.optim.Adam(params, lr=0.005, fused=True, capturable=graphed) if train else None
    reducer = FlatGradAllReduce(params) if (world > 1 and train) else None
    if reducer:
        reducer.broadcast_parameters(list(model.buffers()))

    gen = torch.Generator().manual_seed(1000 + rank)
    K, R, T = synthetic_cameras(B, V, h, w, seed=rank)
    d_min, d_int = torch.full((B, 1, 1, 1), 425.0), torch.ones(B, 1, 1, 1)
    img_host = torch.randn(B * V, 3, H, W, generator=gen).pin_memory()
    gt_host = (425.0 + 480.0 * torch.rand(B, 1, h, w, generator=gen))
    gt_host = (gt_host * (torch.rand(B, 1, h, w, generator=gen) > 0.3)).pin_memory()     # 30 % invalid (loss.py:8)
    img_dev, gt_dev = img_host.to(dev), gt_host.to(dev)
    loss_host = torch.zeros(1).pin_memory()

    slab = None
    if workload == "cfg4" and world > 1:                   # ONE sample across the ranks: depth-slab split (SURVEY §8e)
        from mvs_b200.harness import DepthSlabMVSNet
        K, R, T = synthetic_cameras(B, V, h, w, seed=0)     # every rank works on the same scene
        g0 = torch.Generator().manual_seed(1000)
        img_host = torch.randn(B * V, 3, H, W, generator=g0).pin_memory()
        gt_host = (425.0 + 480.0 * torch.rand(B, 1, h, w, generator=g0)).pin_memory()
        img_dev, gt_dev = img_host.to(dev), gt_host.to(dev)
        for t in list(model.parameters()) + list(model.buffers()):
            dist.broadcast(t.data, 0)
        slab = DepthSlabMVSNet(model, graph=not args.no_graph)

    # --dump-outputs: the seeded starting state of the training run, restored before the last timed step.  The float atomics of
    # the kernels make every step differ from run to run in the last bits, and the steps before would carry that into the
    # weights; from this state the last step's outputs are the same in every run up to that last-bit noise.
    start = [t.detach().clone() for t in params + list(model.buffers())] if args.dump_outputs and train and not light else None

    def restart():
        with torch.no_grad():
            for t, s in zip(params + list(model.buffers()), start):
                t.copy_(s)
            for st in opt.state.values():                 # in place: a captured graph holds these tensors
                for v in st.values():
                    if torch.is_tensor(v):
                        v.zero_()

    gstep = ginf = None
    if graphed:
        from mvs_b200.harness import GraphedTrainStep
        gstep = GraphedTrainStep(model, B, V, H, W, dev, reducer=reducer, optimizer=opt)
    elif not train and slab is None and not args.no_graph:
        from mvs_b200.harness import GraphedInference
        ginf = GraphedInference(model, B, V, H, W, dev)

    def step(img, gt):
        """-> (loss, initial depth map, refined depth map) of this step."""
        if gstep is not None:                              # forward + loss + backward + all-reduce + Adam: one CUDA graph
            return (gstep.run(img, gt, K, R, T, d_min, d_int), *gstep.depth)
        if slab is not None:
            initial, refined = slab.forward(img, K, R, T, d_min, d_int, V)
            return loss_fcn(gt, initial, refined)[0], initial, refined
        if train:
            if reducer is not None and reducer.attached:
                reducer.bucket.zero_()
            else:
                opt.zero_grad(set_to_none=True)
            initial, refined = model(img, K, R, T, d_min, d_int, B, V)
            loss, _, _ = loss_fcn(gt, initial, refined)
            loss.backward()
            if reducer:
                reducer.reduce()
            opt.step()
            return loss.detach(), initial.detach(), refined.detach()
        with torch.no_grad():
            if ginf is not None:                           # inference forward replayed as one CUDA graph
                initial, refined = ginf.run(img, K, R, T, d_min, d_int)
            else:
                initial, refined = model(img, K, R, T, d_min, d_int, B, V)
            return loss_fcn(gt, initial, refined)[0], initial, refined

    def step_resident():
        return step(img_dev, gt_dev)

    # host-fed step: every step's inputs cross PCIe from pinned host memory inside the timed region, as a prefetching loader
    # would deliver them -- double-buffered device staging, the copy of step i+1 on a side stream while step i computes
    copy_stream = torch.cuda.Stream()
    stage = [(torch.empty_like(img_dev), torch.empty_like(gt_dev)) for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    feed = {"slot": 0, "primed": False}

    def prefetch(slot_, after=None):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot_])        # the step that read this staging pair has finished with it
            if after is not None:
                copy_stream.wait_event(after)              # ... and the running step has reached its backward pass
            if _E2E_DIAG & 4:                              # diagnostics: a quarter of the image bytes
                stage[slot_][0][:3].copy_(img_host[:3], non_blocking=True)
            elif _E2E_DIAG & 8:                            # diagnostics: the images in four separate copies
                for q4 in range(4):
                    stage[slot_][0][3 * q4:3 * q4 + 3].copy_(img_host[3 * q4:3 * q4 + 3], non_blocking=True)
            else:
                stage[slot_][0].copy_(img_host, non_blocking=True)
            stage[slot_][1].copy_(gt_host, non_blocking=True)
            ready[slot_].record(copy_stream)

    loss_slots = [torch.zeros(1).pin_memory(), torch.zeros(1).pin_memory()]
    loss_done = [torch.cuda.Event(), torch.cuda.Event()]
    pending = {"n": 0}

    def step_e2e():
        """One host-fed step.  The loss of EVERY step is copied to the host and read there, one step behind the launches: the
        host waits for step i-1's loss only after step i is queued, so the GPU never idles on the host's read-back."""
        cur = feed["slot"]
        if not feed["primed"]:
            consumed[0].record(); consumed[1].record()
            prefetch(cur)
            feed["primed"] = True
        torch.cuda.current_stream().wait_event(ready[cur])
        loss = step(stage[cur][0], stage[cur][1])[0]
        consumed[cur].record()
        # the next step's 47 MB H2D copy is issued AFTER this step's launches: the step's own small H2D copies (sweep geometry,
        # on the compute stream) share the host-to-device copy engine with it and would otherwise queue behind it -- the whole
        # copy (0.86 ms at PCIe 5 rate) then sat in front of every step instead of under it (measured: MVSB200_E2E_DIAG=1)
        if not (_E2E_DIAG & 1):
            runner = gstep if gstep is not None else (ginf if ginf is not None else slab)
            prefetch(cur ^ 1, getattr(runner, "mid_event", None) if not (_E2E_DIAG & 16) else None)
        else:
            ready[cur ^ 1].record()
        i = pending["n"]
        loss_slots[i & 1].copy_(loss.reshape(1), non_blocking=True)
        loss_done[i & 1].record()
        if i > 0 and not (_E2E_DIAG & 2):
            loss_done[(i - 1) & 1].synchronize()           # the user reads the previous step's loss
            loss_host.copy_(loss_slots[(i - 1) & 1])
        pending["n"] = i + 1
        feed["slot"] = cur ^ 1
        return loss_host

    def timed(fn, n):
        """-> (ms for n calls of fn, what the last call returned)"""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    graph_note = None
    if gstep is not None:
        try:
            step_resident()
            torch.cuda.synchronize()
        except Exception as e:                             # capture refused: say so and measure the eager step
            graph_note = f"capture failed, eager step measured: {type(e).__name__}: {str(e)[:200]}"
            sys.stderr.write("bench.py: " + graph_note + "\n")
            if world > 1:
                raise                                      # ranks must not diverge between a graphed and an eager step
            gstep = None
            opt = torch.optim.Adam(params, lr=0.005, fused=True)
            opt.zero_grad(set_to_none=True)
    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0 and not light:
        sampler.start()
    if gstep is None and ginf is None and not light:
        ops.EVENTS = {}
    n0 = mvs_b200.launch_count()
    if start is None:
        ms, last = timed(step_resident, steps)
    else:                                                  # two timed windows; the restart between them is not timed
        ms = timed(step_resident, steps - 1)[0] if steps > 1 else 0.0
        restart()
        ms_last, last = timed(step_resident, 1)
        ms += ms_last
    if args.dump_outputs and rank == 0 and not light:
        dump_outputs(args.dump_outputs, last, params if train else None)
    launches = ((gstep.launches * steps) if gstep is not None else
                (ginf.launches * steps) if ginf is not None else
                (slab.launches * steps) if slab is not None and getattr(slab, "launches", 0) else mvs_b200.launch_count() - n0)
    events, ops.EVENTS = ops.EVENTS, None
    clocks = sampler.stop() if (rank == 0 and not light) else None
    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, steps)
    maps = B * (1 if slab is not None else world) * steps
    value, e2e_value = maps / (ms * 1e-3), maps / (ms_e2e * 1e-3)

    def cleanup():
        if gstep is not None:
            gstep.release()
        if slab is not None:
            slab.release()

    if light:
        out = {"workload": wl["desc"], "value": value, "unit": "depth maps/s", "ms_per_step": ms / steps, "steps": steps,
               "per_gpu_batch": B, "n_gpus": world,
               "e2e": {"value": e2e_value, "unit": "depth maps/s", "ms_per_step": ms_e2e / steps,
                       "h2d_bytes_per_step": img_host.numel() * 4 + gt_host.numel() * 4, "d2h_bytes_per_step": 4},
               "gpu_launches": launches}
        cleanup()
        return out if rank == 0 else None

    if gstep is not None or ginf is not None:
        # per-kernel durations cannot be bracketed inside a graph replay: the same step, issued eagerly right after the
        # timed region with every libmvs_b200.so launch between two CUDA events on its launching stream
        graphed_step, gstep, graphed_inf, ginf = gstep, None, ginf, None
        if train and graphed_step is not None:
            opt_graph, opt = opt, torch.optim.Adam(params, lr=0.005, fused=True)      # eager twin of the captured optimiser
        step_resident()
        ops.EVENTS = {}
        for _ in range(steps):
            step_resident()
        torch.cuda.synchronize()
        events, ops.EVENTS = ops.EVENTS, None
        gstep, ginf = graphed_step, graphed_inf            # (reporting only from here on)

    # per-kernel live timings -> rooflines
    peak, peak_src = _peaks()
    tpeak, tpeak_src = _tensor_peak()
    vox = B * D * h * w
    if slab is not None:                                   # K1 of this rank: its own planes + halo
        k0, k1_ = slab.reg.plan(D).cost_planes(rank)
        vox = B * (k1_ - k0) * h * w
    alg = {"warp_variance_fwd": 4 * B * V * C * h * w + 2 * vox * C,            # fp32 features in, bf16 volume out
           "warp_variance_bwd": 2 * vox * C + 2 * 4 * B * V * C * h * w,        # bf16 gcost + features in, gfeat out
           "softmax_ranks_fwd": 2 * 4 * vox + 4 * 5 * B * h * w}
    kern = {}
    for name, evs in events.items():
        tot = sum(a.elapsed_time(b) for a, b, _ in evs)
        kern[name] = {"ms": tot / len(evs), "launches": len(evs), "ms_per_step": tot / steps}
        if name in alg:
            t = tot / len(evs)
            kern[name].update({"alg_bytes": alg[name], "GBps": alg[name] / (t * 1e-3) / 1e9,
                               "frac_hbm": alg[name] / (t * 1e-3) / 1e9 / peak})
        work = [w_ for _, _, w_ in evs if w_ is not None]
        if work and (name in TC_KERNELS or name in TC2D_KERNELS):
            kern[name].update({"alg_flops_per_step": sum(work) / steps, "TFLOPs": sum(work) / (tot * 1e-3) / 1e12,
                               "frac": sum(work) / (tot * 1e-3) / 1e12 / tpeak})
    k1 = kern.get("warp_variance_fwd", {})
    k2 = kern.get("warp_variance_bwd", {})
    roofline_k1 = {"kernel": "warp_variance_fwd kernel<V=%d, bf16 volume> inside the step (as used by the bf16 regulariser)" % V,
                   "bound": "hbm", "achieved": k1.get("GBps"),
                   "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": k1.get("frac_hbm"),
                   "traffic": None, "alg_bytes_per_launch": alg["warp_variance_fwd"], "ms_per_launch": k1.get("ms"),
                   "voxels_per_s": vox / (k1["ms"] * 1e-3) if k1 else None,
                   "note": "algorithmic bytes = 4*B*V*C*h*w (fp32 features) + 2*B*C*D*h*w (bf16 volume)"}
    roofline_k2 = {"kernel": "warp_variance_bwd kernel<V=%d, bf16 upstream gradient> inside the step" % V, "bound": "hbm",
                   "achieved": k2.get("GBps"), "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": k2.get("frac_hbm"),
                   "traffic": None, "alg_bytes_per_launch": alg["warp_variance_bwd"], "ms_per_launch": k2.get("ms")} if k2 else None
    # the same kernel with the fp32 volume the reference produces (SURVEY §8d quotes the HBM roofline on these bytes:
    # 4*V*C*h*w in + 4*C*D*h*w out per sample), timed live on this batch's geometry: L2 flushed between launches, CUDA events
    roofline_k1_fp32 = None
    if slab is None:
        with torch.no_grad():
            sweep = ops.PlaneSweep(K, R, T, d_min, d_int, B, V, D, d_scale, h, w, dev)
            feat = torch.randn(B * V, h, w, C, device=dev).permute(0, 3, 1, 2)
            flush = torch.empty(160 * 1024 * 1024, dtype=torch.float32, device=dev)       # 640 MB > L2
            ts = []
            for i in range(3 + 5):
                flush.zero_()
                a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                cv32 = ops.warp_variance(feat, sweep, torch.float32)
                b_.record()
                torch.cuda.synchronize()
                if i >= 3:
                    ts.append(a.elapsed_time(b_))
                del cv32
            del flush
        t32 = sorted(ts)[len(ts) // 2]
        bytes32 = 4 * B * V * C * h * w + 4 * B * D * h * w * C
        roofline_k1_fp32 = {"kernel": "warp_variance_fwd kernel<V=%d, fp32 volume>" % V, "bound": "hbm",
                            "achieved": bytes32 / (t32 * 1e-3) / 1e9, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                            "frac": bytes32 / (t32 * 1e-3) / 1e9 / peak, "alg_bytes_per_launch": bytes32, "ms_per_launch": t32,
                            "voxels_per_s": B * D * h * w / (t32 * 1e-3),
                            "traffic": _ncu_traffic(K1_NCU),
                            "note": "isolated launches on the step's shapes (B=%d), median of 5, L2 flushed" % B}
    # headline roofline: the tcgen05 convolution family (every tensor-core launch of the step), per-kernel entries beside it
    fam = [n for n in TC_KERNELS if n in kern and "alg_flops_per_step" in kern[n]]
    tc_ms = sum(kern[n]["ms_per_step"] for n in fam)
    tc_fl = sum(kern[n]["alg_flops_per_step"] for n in fam)
    k3 = kern.get("conv3d_s1_tc", {})
    roofline = {"kernel": "tcgen05 convolution family of the regulariser (tcgen05.mma / TMEM / TMA implicit-GEMM 3x3x3 convolutions: "
                          + ", ".join(fam) + "), all launches of the step together",
                "bound": "tensor", "achieved": tc_fl / (tc_ms * 1e-3) / 1e12 if tc_ms else None, "peak": tpeak,
                "peak_source": tpeak_src, "unit": "TFLOP/s", "frac": tc_fl / (tc_ms * 1e-3) / 1e12 / tpeak if tc_ms else None,
                "alg_flops_per_step": tc_fl, "ms_per_step": tc_ms,
                "flops_counted": "algorithmic: 2*27*Cin*Cout*voxels on the channels that carry data (zero-padded channels of the "
                                 "widened 8->16 gradient are not counted)",
                "per_kernel": {n: {k_: kern[n][k_] for k_ in ("ms_per_step", "launches", "alg_flops_per_step", "TFLOPs", "frac")} for n in fam},
                "dominant_kernel": {"kernel": "conv3d_s1_kdn_kernel<CIN,NOUT,MB> (%d launches/step: forward and data gradient of conv_0_0 "
                                              "and conv_{1,2,3}_1)" % (k3.get("launches", 0) // max(steps, 1)),
                                    "achieved": k3.get("TFLOPs"), "frac": k3.get("frac"), "ms_per_step": k3.get("ms_per_step"),
                                    "alg_flops_per_step": k3.get("alg_flops_per_step")},
                "networks_2d": _family_2d(kern, tc_fl, tc_ms, tpeak),
                "traffic": _ncu_traffic(K3_NCU),
                "traffic_case": "ncu --set full capture of the 32->32 dense canvas launch (252 MB in + 252 MB out algorithmic)"}

    line = None
    if rank == 0:
        line = {"metric": "depth maps/sec", "value": value, "unit": "depth maps/s", "n_gpus": world, "steps": steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True,
                "scaling": "strong" if slab is not None else "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": wl["desc"], "per_gpu_batch": B, "views": V, "D": D, "features": [C, h, w],
                           "l2": "inputs_exceed_l2 (cost volume %.0f MB per step > 126 MB L2)" % (2 * vox * C / 1e6),
                           "parallelism": (f"depth-slab x{world} (one sample; K1 on own planes + halo, halo/box exchanges and BatchNorm-sum "
                                           f"all-reduces over NCCL, logits re-sharded to rows for K4; hot path "
                                           f"{'replayed as one CUDA graph per rank' if not args.no_graph else 'issued eagerly'})"
                                           if slab is not None else
                                           f"dp{world} (scene/batch sharding; gradients are views into one flat fp32 bucket, one NCCL "
                                           f"all-reduce per step inside the step's CUDA graph)" if world > 1 else "single GPU"),
                           "regulariser_convs": model.cost_volume_reg.conv_backend,
                           "cudnn_benchmark": bool(torch.backends.cudnn.benchmark),
                           "cuda_graph": (f"forward+loss+backward{'+all-reduce' if reducer else ''}+Adam replayed as one CUDA graph "
                                          f"({gstep.launches} libmvs_b200.so launches per replay); per-kernel timings from {steps} "
                                          f"eager steps run right after the timed region") if gstep is not None else
                                         (f"inference forward replayed as one CUDA graph ({ginf.launches} libmvs_b200.so launches per "
                                          f"replay)" if ginf is not None else (graph_note or "off"))},
                "e2e": {"value": e2e_value, "unit": "depth maps/s", "ms_per_step": ms_e2e / steps,
                        "h2d_bytes_per_step": img_host.numel() * 4 + gt_host.numel() * 4, "d2h_bytes_per_step": 4,
                        "input_pipeline": "pinned host buffers, double-buffered device staging: the H2D copy of step i+1 runs on a "
                                          "side stream while step i computes -- it starts when step i reaches its backward pass (an external "
                                          "event recorded inside the step's CUDA graph), under the regulariser's long kernels: under the short "
                                          "launches at the start of a step the saturated PCIe link cost 0.6 ms per step; "
                                          "the loss of every step is copied to the host and read there one step "
                                          "behind the launches (the final read falls inside the timed region's closing synchronize)"},
                "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_k1": roofline_k1,
                "roofline_k1_fp32": roofline_k1_fp32, "roofline_k2": roofline_k2, "kernels": kern,
                "cost_volume_voxels_per_s": roofline_k1["voxels_per_s"]}
    cleanup()
    return line


def cfg4_hot_path(args, rank, world, local_rank):
    """BASELINE.json configs[3] hot path only (K1 -> regulariser -> softmax/depth on given feature maps; no 2D nets): ONE sample,
    5 views, 400x296x32 features, D = 256, split into depth slabs over the ranks (world == 1: the unsharded path), each rank's
    pass replayed as one CUDA graph.  -> ms per depth map, max over ranks."""
    import torch
    import torch.distributed as dist
    import mvs_b200
    from mvs_b200 import ops
    from mvs_b200.harness import synthetic_cameras
    wl = WORKLOADS["cfg4"]
    V, D, h, w = wl["V"], wl["D"], wl["H"] // 4, wl["W"] // 4
    dev = torch.device("cuda", local_rank)
    torch.manual_seed(0)
    K, R, T = synthetic_cameras(1, V, h, w)
    d_min, d_int = torch.full((1, 1, 1, 1), 425.0), torch.ones(1, 1, 1, 1)
    feat = torch.randn(V, h, w, 32, device=dev).permute(0, 3, 1, 2)
    reg = mvs_b200.CostVolumeReg(device=dev).train()
    sweep = ops.PlaneSweep(K, R, T, d_min, d_int, 1, V, D, 480.0 / D, h, w, dev)
    reps = max(3, args.steps // 2)
    with torch.no_grad():
        if world > 1:
            from mvs_b200.depth_slab import DepthSlabCostVolumeReg, GraphedSlabForward
            for t in list(reg.parameters()) + list(reg.buffers()):
                dist.broadcast(t.data, 0)
            dist.broadcast(feat, 0)
            fwd = GraphedSlabForward(DepthSlabCostVolumeReg(reg), sweep, feat.shape, dev)
            run = lambda: fwd(feat)
        else:
            def single():
                cost = ops.warp_variance(feat, sweep, torch.bfloat16)
                return ops.softmax_depth(reg.logits(cost, mvs_b200.conv3d.get(reg.conv_backend)), sweep.d_batch_dev, 5)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    single()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                held = single()
            run = g.replay
        for _ in range(2):
            run()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            run()
        e1.record()
        torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / reps], device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        fwd.release()
    return float(ms.item())


def cpu_baseline(workload):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import cpu_path
    wl = WORKLOADS[workload]
    # cfg1/cfg2: the whole D = 192 sweep of one batch item (~13 s on 16 cores, nothing extrapolated); cfg4: 24 of 256 planes
    # (the reference materialises 19 GB of warped volumes at cfg4)
    d_sample = wl["D"] if wl["H"] * wl["W"] <= 512 * 640 else 24
    torch.set_num_threads(os.cpu_count() or 1)
    s = cpu_path.make_sample(V=wl["V"], D=d_sample, h=wl["H"] // 4, w=wl["W"] // 4, d_total=wl["D"])
    dt, _ = cpu_path.hot_path_step(s, backward=wl["train"])
    scale = wl["D"] / d_sample
    return {"value": 1.0 / (dt * scale), "unit": "depth maps/s", "cores": torch.get_num_threads(), "kind": "port",
            "seconds_sample": dt,
            "sample": (f"oracle port (oracle/cpu_path.py), hot path {'fwd+bwd' if wl['train'] else 'fwd'}, 1 batch item, first "
                       f"{d_sample} of {wl['D']} planes at 160x128x32, one un-warmed pass; time scaled x{scale:g} linearly in D")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg4 depth-slab / cfg3 measurements riding on the default line")
    ap.add_argument("--no-graph", action="store_true", help="issue the train step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (loss, depth maps, gradients) as DIR/<name>.npy; a train "
                         "step's last timed step then starts from the seeded initial weights")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    cores = _pin_rank_to_cores(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    torch.set_num_threads(max(1, min(cores, 16)))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    line = run_b200(args, rank, world, local_rank)
    extras = {}
    if args.workload == "cfg2" and not args.no_extras:
        # riding on the default line so that the driver's BENCH / SCALE files record them (BASELINE.json configs[3] and [2])
        def attempt(name, fn):
            try:
                torch.cuda.empty_cache()
                extras[name] = fn()
            except Exception as e:                          # an extra must never cost the headline line
                extras[name] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
                if world > 1:
                    raise

        def cfg4():
            hot = cfg4_hot_path(args, rank, world, local_rank)
            torch.cuda.empty_cache()
            whole = run_b200(args, rank, world, local_rank, workload="cfg4", light=True)
            out = {"workload": WORKLOADS["cfg4"]["desc"].replace(" on ONE GPU", "").replace(" without the depth-slab split", "")
                               + (f", depth-slab split over {world} GPUs" if world > 1 else ", one GPU (unsharded)"),
                   "n_gpus": world, "scaling": "strong", "hot_path_ms_per_depth_map": hot,
                   "hot_path": "K1 -> regulariser -> softmax/depth on resident feature maps, one CUDA graph per rank, max over ranks"}
            if whole:
                out.update({"whole_inference_ms_per_depth_map": whole["ms_per_step"], "value": whole["value"], "unit": whole["unit"],
                            "e2e": whole["e2e"], "gpu_launches": whole["gpu_launches"]})
            return out

        attempt("cfg4_depth_slab", cfg4)
        if world > 1:
            attempt("cfg3", lambda: run_b200(args, rank, world, local_rank, workload="cfg3", light=True))
    if rank == 0:
        line.update({k: v for k, v in extras.items() if v is not None})
        line["config"]["scale_line_workload"] = ("cfg2 (batch 4 per GPU) at every N; BASELINE.json configs[2] (batch 8 per GPU) is the "
                                                 "`cfg3` key of the N > 1 lines, configs[3] the `cfg4_depth_slab` key")
        line["host_cores_per_rank"] = cores
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.workload)
        print(json.dumps(line), flush=True)
    if world > 1:
        # replayed graphs that held NCCL work were released above; drain and leave without the collective teardown (observed:
        # destroy_process_group() after a captured collective may not return)
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
