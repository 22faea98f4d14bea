#!/usr/bin/env python
"""Which kernels do the side-stream weight gradients (ops.wgrad_fork) run under?  One eager cfg2 train step under torch.profiler
(CUDA activities), after warm-up steps; for every kernel on the side stream: its time, the kernels of the launching stream it
overlapped and for how long.  Writes <out>/wgrad_overlap.json and <out>/wgrad_overlap.md."""
import argparse
import collections
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "deep-multiview-depth-estimation_b200"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import torch  # noqa: E402
from torch.profiler import profile, ProfilerActivity  # noqa: E402
from mvs_b200.harness import MVSNet, loss_fcn  # noqa: E402
import plane_sweep as ps  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--B", type=int, default=4)
ap.add_argument("--D", type=int, default=192)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--out", required=True, help="directory for the two reports")
a = ap.parse_args()
dev = torch.device("cuda:0")
B, V, H, W, D = a.B, 3, 512, 640, a.D
torch.manual_seed(0)
model = MVSNet(D, 480.0 / D, precision="bf16").to(dev).train()
K, R, T = ps.synthetic_cameras(B, V, H // 4, W // 4)
d_min, d_int = torch.full((B, 1, 1, 1), 425.0), torch.ones(B, 1, 1, 1)
g = torch.Generator().manual_seed(1000)
img = torch.randn(B * V, 3, H, W, generator=g).to(dev)
gt = (425.0 + 480.0 * torch.rand(B, 1, H // 4, W // 4, generator=g)).to(dev)


def step():
    model.zero_grad(set_to_none=True)
    initial, refined = model(img, K, R, T, d_min, d_int, B, V)
    loss_fcn(gt, initial, refined)[0].backward()


for _ in range(a.warmup):
    step()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    step()
    torch.cuda.synchronize()

kern = []
for e in prof.profiler.kineto_results.events():
    if e.device_type() == torch.autograd.DeviceType.CUDA and e.duration_ns() > 0 and not e.name().startswith("Memset") \
            and not e.name().startswith("Memcpy"):
        kern.append((e.start_ns(), e.start_ns() + e.duration_ns(), e.device_resource_id(), e.name()))
streams = sorted({k[2] for k in kern})
main_id = max(streams, key=lambda s: sum(1 for k in kern if k[2] == s))   # the launching stream issues most kernels
side_k = [k for k in kern if k[2] != main_id]
main_k = [k for k in kern if k[2] == main_id]


def short(name):
    name = name.replace("(anonymous namespace)::", "")
    return name.split("(")[0][:90]


rows = []
for s0, s1, sid, name in side_k:
    over = collections.defaultdict(float)
    for m0, m1, _, mname in main_k:
        o = min(s1, m1) - max(s0, m0)
        if o > 0:
            over[short(mname)] += o / 1e6
    rows.append({"kernel": short(name), "stream": sid, "ms": (s1 - s0) / 1e6, "overlap_ms": sum(over.values()),
                 "overlapped": sorted(([k, v] for k, v in over.items()), key=lambda kv: -kv[1])})
t0 = min(k[0] for k in kern)
t1 = max(k[1] for k in kern)
busy_main = sum(k[1] - k[0] for k in main_k) / 1e6
res = {"device": torch.cuda.get_device_name(dev), "shape": dict(B=B, V=V, H=H, W=W, D=D), "launching_stream": main_id,
       "side_streams": sorted({k[2] for k in side_k}), "step_kernel_span_ms": (t1 - t0) / 1e6,
       "launching_stream_kernel_ms": busy_main, "side_kernel_ms": sum(r["ms"] for r in rows),
       "side_overlap_ms": sum(r["overlap_ms"] for r in rows), "side_kernels": rows}
os.makedirs(a.out, exist_ok=True)
with open(os.path.join(a.out, "wgrad_overlap.json"), "w") as f:
    json.dump(res, f, indent=1)
lines = [f"# Side-stream weight gradients of one eager cfg2 step ({res['device']})", "",
         f"step kernel span {res['step_kernel_span_ms']:.2f} ms; launching-stream kernels {busy_main:.2f} ms; side-stream kernels "
         f"{res['side_kernel_ms']:.2f} ms, of which {res['side_overlap_ms']:.2f} ms under launching-stream kernels", "",
         "| side kernel | ms | overlapped ms | launching-stream kernels it ran under (ms) |", "|---|---|---|---|"]
for r in rows:
    top = ", ".join(f"{k} {v:.3f}" for k, v in r["overlapped"][:4]) or "none"
    lines.append(f"| {r['kernel']} | {r['ms']:.3f} | {r['overlap_ms']:.3f} | {top} |")
with open(os.path.join(a.out, "wgrad_overlap.md"), "w") as f:
    f.write("\n".join(lines) + "\n")
print("\n".join(lines[:3]))
