#!/usr/bin/env python
"""Eval-mode inference, graph-replayed: FrozenMVSNet against today's two no-grad paths, plus the new epilogue kernels against the
kernel + BatchNorm pass they replace.

Variants (each a harness.GraphedInference, one CUDA graph per forward; warm-up and capture outside the timed window):
  (a) eval     model.eval()                 encoder / refinement on the modules' torch layers, regulariser eval branch
  (b) train    model.train()                test.py:61's mode (batch statistics), the native train-path kernels
  (c) frozen   FrozenMVSNet(model.eval())   BatchNorm in the convolution epilogues, deconv_3_0 / deconv_2_0 on C only
Workloads: cfg1 (B=1, V=3, 640x512, D=192), cfg2-shaped batch (B=4), cfg4 size on one GPU (V=5, 1600x1184, D=256).
The variants alternate within every round (>= 3 rounds); per variant the median and the spread (min..max) over rounds of the
per-forward time.  The input working set of cfg2 / cfg4 exceeds the L2; cfg1's is re-filled by every forward's own passes.

  python tools/bench_frozen.py --out DIR [--rounds 3] [--iters 10] [--configs cfg1,cfg2,cfg4]
"""
import argparse
import copy
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "deep-multiview-depth-estimation_b200"))
import torch  # noqa: E402

import mvs_b200  # noqa: E402
from mvs_b200 import _lib, harness, ops  # noqa: E402
from mvs_b200.conv3d_sm100 import _NAT, _kdn_order, _n_rows, _pack  # noqa: E402

DEV = torch.device("cuda:0")
CL3 = torch.channels_last_3d
CONFIGS = {"cfg1": (1, 3, 512, 640, 192), "cfg2": (4, 3, 512, 640, 192), "cfg4": (1, 5, 1184, 1600, 256)}


def card():
    out = {"name": torch.cuda.get_device_name(DEV)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power = [s.strip() for s in r.stdout.strip().split(",")]
        out.update(name=name, power_limit=power)
    except Exception as e:                      # the numbers stay valid, the power limit is then unknown
        out["power_limit"] = f"unavailable ({e})"
    return out


def events_ms(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def stats(xs):
    xs = sorted(xs)
    return {"median_ms": xs[len(xs) // 2], "min_ms": xs[0], "max_ms": xs[-1], "rounds": xs}


def bench_model(name, rounds, iters):
    B, V, H, W, D = CONFIGS[name]
    torch.manual_seed(0)
    model = harness.MVSNet(D, 480.0 / D).to(DEV)
    K, R, T = harness.synthetic_cameras(B, V, H // 4, W // 4)
    img = torch.randn(B * V, 3, H, W).pin_memory()
    d_min, d_int = torch.full((B, 1, 1, 1), 425.0), torch.ones(B, 1, 1, 1)
    variants = {"eval": GraphedVariant(copy.deepcopy(model).eval(), B, V, H, W),
                "train": GraphedVariant(copy.deepcopy(model).train(), B, V, H, W),
                "frozen": GraphedVariant(mvs_b200.FrozenMVSNet(copy.deepcopy(model).eval()), B, V, H, W)}
    for v in variants.values():                 # capture + warm replays, outside the timed window
        for _ in range(3):
            v.run(img, K, R, T, d_min, d_int)
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for k, v in variants.items():
            times[k].append(events_ms(lambda: v.replay(), iters))
    res = {"B": B, "V": V, "H": H, "W": W, "D": D, "iters_per_round": iters, "launches": {k: v.g.launches for k, v in variants.items()}}
    res.update({k: stats(t) for k, t in times.items()})
    res["frozen_vs_eval"] = res["eval"]["median_ms"] / res["frozen"]["median_ms"]
    res["frozen_vs_train"] = res["train"]["median_ms"] / res["frozen"]["median_ms"]
    del variants
    torch.cuda.empty_cache()
    return res


class GraphedVariant:
    def __init__(self, model, B, V, H, W):
        self.g = harness.GraphedInference(model, B, V, H, W, DEV, warmup=2)

    def run(self, *batch):
        return self.g.run(*batch)

    def replay(self):
        self.g.graph.replay()


# ---------------------------------------------------------------------------------------------------------------- kernels
def kdn(x, wk, cout, out_dims, off, aff=None):
    B, cin = x.shape[:2]
    y = torch.empty((B, cout) + tuple(out_dims), dtype=torch.bfloat16, device=DEV, memory_format=CL3)
    if aff is None:
        _lib.call("mvsb200_conv3d_s1_fwd_kdn", x.data_ptr(), wk.data_ptr(), y.data_ptr(), B, *x.shape[2:], cin, *out_dims, cout, cout,
                  _n_rows(cout), *off, ops._stream())
    else:
        _lib.call("mvsb200_conv3d_s1_fwd_kdn_affine", x.data_ptr(), wk.data_ptr(), y.data_ptr(), B, *x.shape[2:], cin, *out_dims, cout,
                  cout, _n_rows(cout), *off, 0, aff[0].data_ptr(), aff[1].data_ptr(), ops._stream())
    return y


def deconv(x, wp, cout, canvas, pads, win=None, aff=None, add=None):
    B, cin = x.shape[:2]
    dims = canvas if win is None else win[1]
    y = torch.empty((B, cout) + tuple(dims), dtype=torch.bfloat16, device=DEV, memory_format=CL3)
    ys = (ctypes.c_int64 * 4)(y.stride(0), y.stride(2), y.stride(3), y.stride(4))
    if aff is None:
        _lib.call("mvsb200_deconv3d_s2_fwd", x.data_ptr(), wp.data_ptr(), y.data_ptr(), B, *x.shape[2:], cin, *canvas, cout, _n_rows(cout),
                  *pads, ys, ops._stream())
    else:
        _lib.call("mvsb200_deconv3d_s2_fwd_affine", x.data_ptr(), wp.data_ptr(), y.data_ptr(), B, *x.shape[2:], cin, *canvas, cout,
                  _n_rows(cout), *pads, (ctypes.c_int * 6)(*win[0], *win[1]), ys, aff[0].data_ptr(), aff[1].data_ptr(),
                  None if add is None else add.data_ptr(), ops._stream())
    return y


def bench_kernels(rounds, iters):
    """At cfg1's regulariser sizes (B=1, D=192, 128x160): each new epilogue form next to the old kernel + the eval-mode BatchNorm
    pass it replaces (ops.affine_relu, the pass CostVolumeReg's eval branch runs), on the same outputs."""
    B, D, h, w = 1, 192, 128, 160
    canvas = (D, h, w)
    reg = [mvs_b200.central_region(n) for n in canvas]
    C_lo = tuple(lo for lo, _, _ in reg)
    C_dims = tuple(hi - lo + 1 for lo, hi, _ in reg)
    pads = tuple(L for _, _, L in reg)
    box = (slice(None), slice(None)) + tuple(slice(lo, lo + n) for lo, n in zip(C_lo, C_dims))
    g = torch.Generator(device=DEV).manual_seed(0)
    rnd = lambda *s: torch.randn(*s, device=DEV, generator=g)
    aff = lambda c: (rnd(c).abs() + 0.5, rnd(c) * 0.2)
    out = {}
    cases = []
    # conv_0_0: 32 -> 8 on the canvas; conv_3_1: 64 -> 64 on C (input over E)
    x0 = rnd(B, 32, *canvas).to(torch.bfloat16).contiguous(memory_format=CL3)
    w0 = _pack(rnd(8, 32, 3, 3, 3) * 0.05, 0, 16, _kdn_order(_NAT))
    a0 = aff(8)
    cases.append(("kdn conv_0_0 32->8 canvas", lambda: kdn(x0, w0, 8, canvas, (-1, -1, -1), a0),
                  lambda: ops.affine_relu(kdn(x0, w0, 8, canvas, (-1, -1, -1)), *a0)))
    E_dims = tuple(n + 2 for n in C_dims)
    x3 = rnd(B, 64, *E_dims).to(torch.bfloat16).contiguous(memory_format=CL3)
    w3 = _pack(rnd(64, 64, 3, 3, 3) * 0.02, 0, 64, _kdn_order(_NAT))
    a3 = aff(64)
    cases.append(("kdn conv_3_1 64->64 box C", lambda: kdn(x3, w3, 64, C_dims, (0, 0, 0), a3),
                  lambda: ops.affine_relu(kdn(x3, w3, 64, C_dims, (0, 0, 0)), *a3)))
    # transposed convolutions: the old form writes the canvas, normalises it and adds the skip on C (deconv_3_0 / deconv_2_0)
    for name, cin, cout, win in (("deconv_3_0 64->32", 64, 32, True), ("deconv_2_0 32->16", 32, 16, True), ("deconv_1_0 16->8", 16, 8, False)):
        xin = rnd(B, cin, *C_dims).to(torch.bfloat16).contiguous(memory_format=CL3)
        wp = _pack(rnd(cin, cout, 3, 3, 3) * 0.05, 1, _n_rows(cout), _NAT + [-1])
        a = aff(cout)
        wdims = C_dims if win else canvas
        wlo = C_lo if win else (0, 0, 0)
        add = rnd(B, cout, *wdims).to(torch.bfloat16).contiguous(memory_format=CL3)
        crop = box if win else (slice(None),) * 5

        def old(xin=xin, wp=wp, cout=cout, a=a, add=add, crop=crop):
            return ops.affine_relu(deconv(xin, wp, cout, canvas, pads), *a)[crop] + add

        cases.append((f"{name} {'window C' if win else 'canvas'}", lambda xin=xin, wp=wp, cout=cout, a=a, add=add, wlo=wlo, wdims=wdims:
                      deconv(xin, wp, cout, canvas, pads, (wlo, wdims), a, add), old))
    for name, new, old in cases:
        yn, yo = new(), old()
        torch.cuda.synchronize()
        diff = float((yn.float() - yo.float()).abs().max() / yo.float().abs().max())
        for f in (new, old):
            for _ in range(3):
                f()
        tn, to = [], []
        for _ in range(rounds):
            tn.append(events_ms(new, iters))
            to.append(events_ms(old, iters))
        out[name] = {"new": stats([1e3 * t for t in tn]), "old_plus_bn_pass": stats([1e3 * t for t in to]),
                     "unit": "us", "rel_max_diff_new_vs_old": diff}
        for k in ("new", "old_plus_bn_pass"):
            out[name][k] = {kk.replace("_ms", "_us"): v for kk, v in out[name][k].items()}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="directory for bench_frozen.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--configs", default="cfg1,cfg2,cfg4")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_frozen: no CUDA device")
    if a.rounds < 3:
        sys.exit("bench_frozen: at least 3 rounds")
    os.makedirs(a.out, exist_ok=True)
    res = {"card": card(), "timing": "CUDA events around graph replays / kernel launches, warm-up outside the window"}
    res["kernels_cfg1"] = bench_kernels(a.rounds, 20)
    print(json.dumps({"kernels_cfg1": res["kernels_cfg1"]}, indent=1), flush=True)
    for name in a.configs.split(","):
        res[name] = bench_model(name, a.rounds, a.iters if name != "cfg4" else max(3, a.iters // 2))
        print(name, json.dumps(res[name]), flush=True)
    res["card_after"] = card()
    with open(os.path.join(a.out, "bench_frozen.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"], **{k: {v: res[k][v]["median_ms"] for v in ("eval", "train", "frozen")}
                                                 for k in a.configs.split(",")}}))


if __name__ == "__main__":
    main()
