"""The tcgen05 convolution entry points refuse bad arguments before any CUDA call (no GPU needed).

Each entry point starts from a call whose only fault is the one its last check before any CUDA call refuses (an unsupported
channel count, a bad cout, a bad pad or bad strides), so that no case reaches the GPU even if an earlier check went missing.
A case changes arguments of that call and checks the return code, the entry point named at the start of the error message
and a fragment of the message that names the refused argument.
"""
import ctypes

import pytest

import mvs_b200

BADARG, UNSUPPORTED = -1, -3
A, M = 0x10000, 0x10008          # a 16-byte aligned and a misaligned device address (never dereferenced)


def _i64(*v):
    return (ctypes.c_int64 * len(v))(*v)


def _i32(*v):
    return (ctypes.c_int * len(v))(*v)


_S1 = dict(x=A, w=A, y=A, B=1, Di=4, Hi=4, Wi=4, Cin=128, Do=4, Ho=4, Wo=4, cout=16, y_cs=16, n_rows=16,
           off_d=-1, off_h=-1, off_w=-1)
_S1_EX = {k: v for k, v in _S1.items() if k != "y_cs"}
_S1_WG = dict(x=A, gy=A, gw=A, B=1, Di=4, Hi=4, Wi=4, Cin=16, Do=4, Ho=4, Wo=4, cout=24, off_d=-1, off_h=-1, off_w=-1)
_S2 = dict(x=A, w=A, y=A, B=1, Dx=8, Hx=8, Wx=8, Cin=128, Do=4, Ho=4, Wo=4, cout=16, y_cs=16, n_rows=16,
           pad_d=1, pad_h=1, pad_w=1)
_S2_WG = dict(big=A, small=A, gw=A, B=1, Db=8, Hb=8, Wb=8, Cb=16, Ds=4, Hs=4, Ws=4, Cs=16, pad_d=1, pad_h=1, pad_w=3)
_DC = dict(x=A, w=A, y=A, B=1, Di=4, Hi=4, Wi=4, Cin=8, Do=8, Ho=8, Wo=8, cout=16, n_rows=16, pad_d=1, pad_h=1, pad_w=1,
           ys=_i64(8192, 1024, 128, 16))

# entry point -> (error-message prefix, arguments of the starting call in ABI order; the stream is appended)
ENTRY = {
    "conv3d_s1_fwd": ("conv3d_s1_fwd", _S1),
    "conv3d_s1_fwd_ex": ("conv3d_s1_fwd_ex", dict(_S1_EX, Cin=48, tap_mask=0x7ffffff, ys=_i64(1024, 256, 64, 16))),
    "conv3d_s1_wgrad": ("conv3d_s1_wgrad", _S1_WG),
    "conv3d_s1_wgrad_ex": ("conv3d_s1_wgrad", dict(_S1_WG, kd_mask=7)),
    "conv3d_s1_fwd_kdn": ("conv3d_s1_fwd_kdn", _S1),
    "conv3d_s1_fwd_kdn_affine": ("conv3d_s1_fwd_kdn_affine", dict(_S1, planar=0, scale=A, shift=A)),
    "conv2d_rows_fwd": ("conv3d_s1_fwd_kdn", dict(x=A, w=A, y=A, N=4, H=4, W=4, Cin=128, cout=16, y_cs=16, n_rows=16)),
    "conv3d_s2_fwd": ("conv3d_s2_fwd", _S2),
    "conv3d_s2_fwd_stats": ("conv3d_s2_fwd_stats", dict(_S2, workspace=A, sums=A)),
    "conv3d_s2_wgrad": ("conv3d_s2_wgrad", _S2_WG),
    "conv3d_s2_wgrad_lines": ("conv3d_s2_wgrad_lines", dict(_S2_WG, pad_w=1, ss=_i64(1024, 256, 64, 12))),
    "deconv3d_s2_fwd": ("deconv3d_s2_fwd", _DC),
    "deconv3d_s2_fwd_stats": ("deconv3d_s2_fwd", dict(_DC, stats=A, n_blocks=_i32(0))),
    "deconv3d_s2_fwd_affine": ("deconv3d_s2_fwd_affine",
                               dict({k: v for k, v in _DC.items() if k != "ys"}, window=_i32(0, 0, 0, 8, 8, 8),
                                    ys=_DC["ys"], scale=A, shift=A, add=None)),
    "deconv3d_s2_kc_fwd": ("deconv3d_s2_kc_fwd",
                           dict(x=A, x_cs=112, w=A, kc_off=_i32(0, 16, 48), kc_n=_i32(16, 32, 64), n_kc=3, y=A, B=1, Di=4,
                                Hi=4, Wi=4, Do=8, Ho=8, Wo=8, cout=32, n_rows=32, pad_d=1, pad_h=1, pad_w=1,
                                ys=_i64(16384, 2048, 256, 36), accumulate=0)),
}

# fragments of the expected messages: "unsupported channels" comes with MVSB200_E_UNSUPPORTED, every other one with
# MVSB200_E_BADARG.  A case whose check went missing fails on its fragment even where the starting call's fault returns
# the same code.
NULL, ALIGN, SHAPE, PAD = "null", "16-byte aligned", "bad shape", "pad must be 1 or 2 per axis"
COUT, YCS, STRIDES, UNSUP = "n_rows", "output channel stride", "multiples of 8 elements", "unsupported channels"


def _c(fragment, *overs):
    return [(o, fragment) for o in overs]


_COUT = _c(COUT, dict(cout=12), dict(n_rows=24), dict(cout=32, n_rows=16))
_PAD = _c(PAD, dict(pad_d=0), dict(pad_h=3), dict(pad_w=2, pad_d=3))
_SHAPE = _c(SHAPE, dict(B=0), dict(B=65536), dict(Wi=0), dict(Ho=0))

CASES = {
    "conv3d_s1_fwd": [*_c(UNSUP, dict(), dict(Cin=8)), *_c(NULL, dict(x=None), dict(y=None)), *_c(ALIGN, dict(w=M), dict(y=M)),
                      *_SHAPE, *_COUT, *_c(COUT, dict(n_rows=80, cout=80)), *_c(YCS, dict(y_cs=12), dict(y_cs=8))],
    "conv3d_s1_fwd_ex": [*_c(UNSUP, dict(), dict(Cin=48)), *_c(NULL, dict(w=None), dict(ys=None)), *_c(ALIGN, dict(x=M)),
                         *_SHAPE, *_COUT, *_c(STRIDES, dict(ys=_i64(1024, 256, 64, 12)), dict(ys=_i64(1028, 256, 64, 16))),
                         *_c("empty tap mask", dict(tap_mask=0), dict(tap_mask=0xf8000000))],
    "conv3d_s1_wgrad": [*_c("cout must be 8, 16, 32 or 64", dict(), dict(cout=128)), *_c(NULL, dict(gw=None)),
                        *_c(ALIGN, dict(gy=M)), *_c(SHAPE, dict(B=0), dict(Wo=0))],
    "conv3d_s1_wgrad_ex": [*_c("cout must be 8, 16, 32 or 64", dict(), dict(cout=4)), *_c(NULL, dict(x=None)),
                           *_c(ALIGN, dict(gw=M)), *_c(SHAPE, dict(Hi=0)), *_c("depth-tap mask", dict(kd_mask=0), dict(kd_mask=8))],
    "conv3d_s1_fwd_kdn": [*_c(UNSUP, dict(), dict(Cin=24)), *_c(NULL, dict(y=None)), *_c(ALIGN, dict(x=M)), *_SHAPE, *_COUT,
                          *_c(YCS, dict(y_cs=20))],
    "conv3d_s1_fwd_kdn_affine": [*_c(UNSUP, dict(), dict(Cin=24)), *_c("null scale / shift", dict(scale=None), dict(shift=None)),
                                 *_c("planar mode", dict(planar=2), dict(planar=1, B=2), dict(planar=1, off_d=-1),
                                     dict(planar=1, off_d=0, Do=3)),
                                 *_c(NULL, dict(x=None)), *_c(ALIGN, dict(w=M)), *_c(SHAPE, dict(Ho=0)), *_COUT,
                                 *_c(YCS, dict(y_cs=4))],
    "conv2d_rows_fwd": [*_c(UNSUP, dict(), dict(Cin=24)), *_c(NULL, dict(x=None)), *_c(ALIGN, dict(y=M)),
                        *_c(SHAPE, dict(N=0), dict(H=0), dict(W=0)), *_c(COUT, dict(cout=12), dict(n_rows=80, cout=80)),
                        *_c(YCS, dict(y_cs=12))],
    "conv3d_s2_fwd": [*_c(UNSUP, dict(), dict(Cin=24), dict(Cin=8, n_rows=48, cout=48, y_cs=48)), *_c(NULL, dict(x=None)),
                      *_c(ALIGN, dict(w=M)), *_c(SHAPE, dict(Hx=1), dict(Wx=1), dict(B=0), dict(Do=0)), *_COUT,
                      *_c(COUT, dict(n_rows=144, cout=144, y_cs=144)), *_c(YCS, dict(y_cs=12)), *_PAD],
    "conv3d_s2_fwd_stats": _c("null statistics buffers", dict(workspace=None), dict(sums=None)),
    "conv3d_s2_wgrad": [*_c(PAD, dict()), *_c(NULL, dict(big=None)), *_c(ALIGN, dict(small=M)), *_c(SHAPE, dict(Db=0), dict(Ws=0)),
                        *_c("strided operand", dict(Cb=8), dict(Cb=128)), *_c("dense operand", dict(Cs=12), dict(Cs=0)), *_PAD],
    "conv3d_s2_wgrad_lines": [*_c(STRIDES, dict(), dict(ss=_i64(0, 256, 64, 16)), dict(ss=_i64(1024, 256, 60, 16))),
                              *_c(NULL, dict(gw=None)), *_c(ALIGN, dict(big=M)),
                              *_c(SHAPE, dict(B=65536), dict(Wb=1), dict(Hs=0)), *_c("even number", dict(Wb=7)),
                              *_c("limited to 255", dict(Ws=256)), *_c("strided operand", dict(Cb=64)),
                              *_c("dense operand needs", dict(Cs=48), dict(Cs=136)), *_PAD],
    "deconv3d_s2_fwd": [*_c(UNSUP, dict(), dict(Cin=128)), *_c(NULL, dict(x=None), dict(ys=None)), *_c(ALIGN, dict(y=M)), *_SHAPE,
                        *_COUT, *_c(COUT, dict(n_rows=64, cout=64)), *_PAD, *_c(STRIDES, dict(ys=_i64(8192, 1024, 128, 20)))],
    "deconv3d_s2_fwd_stats": [*_c(UNSUP, dict(), dict(Cin=48)), *_c(NULL, dict(w=None)), *_c(ALIGN, dict(x=M)),
                              *_c(SHAPE, dict(Di=0)), *_c(COUT, dict(cout=20)), *_PAD,
                              *_c(STRIDES, dict(ys=_i64(8196, 1024, 128, 16)))],
    "deconv3d_s2_fwd_affine": [*_c(UNSUP, dict(), dict(Cin=24)),
                               *_c(NULL, dict(window=None), dict(scale=None), dict(shift=None), dict(ys=None)),
                               *_c(ALIGN, dict(add=M), dict(w=M)), *_SHAPE, *_COUT, *_PAD,
                               *_c("outside the canvas", dict(window=_i32(-1, 0, 0, 8, 8, 8)), dict(window=_i32(0, 0, 0, 8, 0, 8)),
                                   dict(window=_i32(0, 0, 4, 8, 8, 5))),
                               *_c(STRIDES, dict(ys=_i64(8192, 1024, 124, 16)))],
    "deconv3d_s2_kc_fwd": [*_c(STRIDES, dict(), dict(ys=_i64(16384, 2048, 256, 31))),
                           *_c(NULL, dict(kc_off=None), dict(kc_n=None), dict(y=None)), *_c(ALIGN, dict(x=M)),
                           *_c(SHAPE, dict(B=0), dict(Wo=0)), *_c("K chunks", dict(n_kc=0), dict(n_kc=4), dict(x_cs=116)),
                           *_c("a K chunk has", dict(kc_n=_i32(16, 32, 48))),
                           *_c("outside the voxel row", dict(kc_off=_i32(0, 16, 52)), dict(kc_off=_i32(0, 16, 56))),
                           *_c(COUT, dict(cout=36), dict(n_rows=80, cout=80)), *_PAD],
}


def _params():
    for entry, cases in CASES.items():
        for i, (over, fragment) in enumerate(cases):
            yield pytest.param(entry, over, fragment, id=f"{entry}-{i}")


@pytest.mark.parametrize("entry,over,fragment", list(_params()))
def test_conv_entry_point_refuses_bad_arguments(entry, over, fragment):
    prefix, start = ENTRY[entry]
    assert set(over) <= set(start)
    lib = mvs_b200.load_library()
    args = list(dict(start, **over).values()) + [None]
    assert getattr(lib, "mvsb200_" + entry)(*args) == (UNSUPPORTED if fragment == UNSUP else BADARG)
    msg = lib.mvsb200_last_error().decode()
    assert msg.startswith(prefix + ": ") and fragment in msg, msg
