"""ctypes binding of libmvs_b200.so (C ABI declared in include/mvs_b200.h).

There is no CPU or PyTorch fallback: if the shared library is missing, or a call fails, this raises.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MVSB200_LIB") or os.path.normpath(os.path.join(_HERE, "..", "csrc", "libmvs_b200.so"))   # env: A/B builds
ABI_VERSION = 1
F32, BF16 = 0, 1
VIEW_PARAM_FLOATS = 16
FUSION_CAM_FLOATS, FUSION_BLOCK_PIXELS, FUSION_MAX_SOURCES = 32, 128, 16     # MVSB200_FUSION_* of include/mvs_b200.h
PC_MAX_CELLS = 1 << 28                                                       # MVSB200_PC_MAX_CELLS
PC_ICP_BLOCKS, PC_ICP_SUMS = 1024, 18                                        # MVSB200_PC_ICP_*
PC_RANSAC_MAX_SAMPLE, PC_RANSAC_RECORD = 64, 80                             # MVSB200_PC_RANSAC_*
PC_KNN_MAX = 32                                                              # MVSB200_PC_KNN_MAX

_c = ctypes
_P, _I = _c.c_void_p, _c.c_int

_SIGNATURES = {
    "mvsb200_abi_version": (_I, []),
    "mvsb200_last_error": (_c.c_char_p, []),
    "mvsb200_launch_count": (_c.c_uint64, []),
    "mvsb200_nchw_to_nhwc_f32": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "mvsb200_nhwc_to_nchw_f32": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "mvsb200_pack_filter": (_I, [_P, _P] + [_I] * 8 + [_P, _P]),
    "mvsb200_widen_rows_8to16_bf16": (_I, [_P, _P, _c.c_int64, _P]),
    "mvsb200_warp_variance_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "mvsb200_warp_variance_bwd": (_I, [_P, _P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _I, _P]),
    "mvsb200_warp_materialize": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "mvsb200_softmax_depth_fwd": (_I, [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "mvsb200_softmax_depth_conf_fwd": (_I, [_P, _I, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "mvsb200_depth_confidence": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "mvsb200_depth_from_ranks": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "mvsb200_depth_bwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "mvsb200_softmax_bwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "mvsb200_variance_views_fwd": (_I, [_P, _P, _I, _I, _c.c_int64, _P]),
    "mvsb200_variance_views_bwd": (_I, [_P, _P, _P, _I, _I, _c.c_int64, _P]),
    "mvsb200_conv3d_s1_fwd": (_I, [_P, _P, _P] + [_I] * 14 + [_P]),
    "mvsb200_conv3d_s1_fwd_kdn": (_I, [_P, _P, _P] + [_I] * 14 + [_P]),
    "mvsb200_conv3d_s1_fwd_kdn_affine": (_I, [_P, _P, _P] + [_I] * 15 + [_P, _P, _P]),
    "mvsb200_conv3d_s1_fwd_ex": (_I, [_P, _P, _P] + [_I] * 13 + [_c.c_uint, _P, _P]),
    "mvsb200_conv3d_s2_fwd": (_I, [_P, _P, _P] + [_I] * 14 + [_P]),
    "mvsb200_conv3d_s2_fwd_stats": (_I, [_P, _P, _P] + [_I] * 14 + [_P, _P, _P]),
    "mvsb200_conv3d_s2_wgrad": (_I, [_P, _P, _P] + [_I] * 12 + [_P]),
    "mvsb200_conv3d_s2_wgrad_lines": (_I, [_P, _P, _P] + [_I] * 12 + [_P, _P]),
    "mvsb200_deconv3d_s2_fwd": (_I, [_P, _P, _P] + [_I] * 13 + [_P, _P]),
    "mvsb200_deconv3d_s2_fwd_stats": (_I, [_P, _P, _P] + [_I] * 13 + [_P, _P, _P, _P]),
    "mvsb200_deconv3d_s2_fwd_affine": (_I, [_P, _P, _P] + [_I] * 13 + [_P, _P, _P, _P, _P, _P]),
    "mvsb200_deconv3d_s2_kc_fwd": (_I, [_P, _I, _P, _P, _P, _I, _P] + [_I] * 12 + [_P, _I, _P]),
    "mvsb200_conv3d_s1_wgrad": (_I, [_P, _P, _P] + [_I] * 12 + [_P]),
    "mvsb200_conv3d_s1_wgrad_ex": (_I, [_P, _P, _P] + [_I] * 12 + [_c.c_uint, _P]),
    "mvsb200_image_to_rows8": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "mvsb200_conv2d_rows_fwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "mvsb200_s2d_rows_bf16": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "mvsb200_conv_out_workspace_floats": (_c.c_int64, []),
    "mvsb200_conv_out_fwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "mvsb200_conv_out_dgrad": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "mvsb200_conv_out_wgrad": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "mvsb200_affine_workspace_floats": (_c.c_int64, []),
    "mvsb200_channel_sums": (_I, [_P, _I, _P, _P, _I, _P, _P, _P, _P]),
    "mvsb200_channel_sums_bwd": (_I, [_P, _I, _P, _P, _I, _P, _P, _P, _P]),
    "mvsb200_affine_relu_geo_fwd": (_I, [_P, _I, _P, _P, _I, _P, _P, _P, _I, _P]),
    "mvsb200_affine_relu_geo_bwd": (_I, [_P, _I, _P, _P, _I, _P, _P, _P, _I, _P, _P, _P, _P, _I, _P]),
    "mvsb200_box_bn_algebra_fwd": (_I, [_P, _P, _P, _P, _I, _c.c_double, _P, _P, _c.c_double, _c.c_double, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mvsb200_outside_sums_fwd": (_I, [_P, _P, _P, _I, _I, _P, _P, _P, _P]),
    "mvsb200_outside_sums_bwd": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P]),
    "mvsb200_box_bn_algebra_bwd": (_I, [_P, _P, _P, _P, _P, _P, _I, _c.c_double, _P, _P, _P, _P, _P]),
    "mvsb200_box_bn_relu_bwd_reduce": (_I, [_P, _I, _P, _P, _I, _P, _P, _P, _I, _P, _P, _P, _I, _P]),
    "mvsb200_box_bn_relu_bwd_apply": (_I, [_P, _I, _P, _P, _I, _P, _P, _P, _P, _P, _I, _P, _P, _I, _P]),
    "mvsb200_masked_l1_workspace_floats": (_c.c_int64, [_I]),
    "mvsb200_masked_l1_fwd": (_I, [_P, _P, _P, _I, _I, _P, _P, _P]),
    "mvsb200_masked_l1_bwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _P, _P]),
    "mvsb200_refine_input_fwd": (_I, [_P, _P, _P, _I, _I, _I, _P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "mvsb200_refine_input_bwd": (_I, [_P, _I, _P, _P, _I, _I, _P, _P]),
    "mvsb200_refine_output_fwd": (_I, [_P, _I, _P, _P, _P, _I, _I, _P, _P]),
    "mvsb200_refine_output_bwd": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "mvsb200_bn_workspace_floats": (_c.c_int64, []),
    "mvsb200_bn_stats": (_I, [_P, _I, _c.c_int64, _I, _P, _P, _P, _P]),
    "mvsb200_bn_relu_fwd": (_I, [_P, _I, _P, _P, _P, _I, _c.c_int64, _I, _P]),
    "mvsb200_bn_relu_fwd_s2d": (_I, [_P, _I, _P, _P, _P, _I, _c.c_int64, _I, _I, _I, _P]),
    "mvsb200_bn_relu_bwd_s2d": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _c.c_int64, _I, _I, _I, _P]),
    "mvsb200_bn_stats_affine": (_I, [_P, _I, _c.c_int64, _I, _P, _P, _P, _P, _c.c_double, _c.c_double, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mvsb200_bn_finalize_affine": (_I, [_P, _I, _c.c_int64, _I, _P, _P, _c.c_double, _c.c_double, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mvsb200_bn_stats_geo": (_I, [_P, _I, _c.c_int64, _I, _P, _P, _P, _P, _P]),
    "mvsb200_bn_relu_fwd_crop": (_I, [_P, _I, _P, _P, _P, _I, _c.c_int64, _I, _P, _P]),
    "mvsb200_bn_relu_add_apply": (_I, [_P, _I, _P, _P, _P, _P, _I, _c.c_int64, _I, _P, _P]),
    "mvsb200_bn_relu_bwd_crop": (_I, [_P, _I, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _c.c_int64, _I, _P, _P]),
    "mvsb200_bn_relu_bwd": (_I, [_P, _I, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _c.c_int64, _I, _P]),
    "mvsb200_fusion_check": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _c.c_float, _c.c_float, _c.c_float, _I, _P, _P, _P, _P, _P]),
    "mvsb200_fusion_visibility": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _c.c_float, _c.c_float, _c.c_float, _I, _I, _P, _P, _P, _P, _P,
                                       _P]),
    "mvsb200_fusion_emit": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _P, _P, _P]),
    "mvsb200_resize_rgb": (_I, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "mvsb200_pc_grid_keys": (_I, [_P, _I] + [_c.c_float] * 4 + [_I, _I, _I, _P, _P]),
    "mvsb200_pc_grid_cells": (_I, [_P, _P, _P, _I, _P, _P, _P, _P]),
    "mvsb200_pc_nearest": (_I, [_P, _I, _P, _P, _P] + [_c.c_float] * 4 + [_I, _I, _I, _c.c_float, _c.c_float, _P, _P]),
    "mvsb200_pc_nearest_index": (_I, [_P, _I, _P, _P, _P] + [_c.c_float] * 4 + [_I, _I, _I, _c.c_float, _c.c_float, _P, _P, _P]),
    "mvsb200_pc_thin_neighbours": (_I, [_P, _P, _P, _I] + [_c.c_float] * 4 + [_I, _I, _I, _c.c_double, _P, _P, _P, _P]),
    "mvsb200_pc_thin_round": (_I, [_P, _P, _P, _P, _I, _P, _P]),
    "mvsb200_pc_transform_crop": (_I, [_P, _I, _P, _P, _I, _I, _c.c_double, _c.c_double, _P, _P, _P]),
    "mvsb200_pc_voxel_keys": (_I, [_P, _I] + [_c.c_double] * 4 + [_c.c_int64] * 3 + [_P, _P]),
    "mvsb200_pc_voxel_mean": (_I, [_P, _P, _P, _I, _P, _P, _P]),
    "mvsb200_pc_icp_sums": (_I, [_P, _P, _I, _P, _P, _P, _P, _P]),
    "mvsb200_pc_transform64": (_I, [_P, _I, _P, _P, _P]),
    "mvsb200_pc_ransac_align": (_I, [_P, _P, _I, _I, _I, _c.c_double, _I, _c.c_uint64, _P, _P, _P, _P, _P, _P]),
    "mvsb200_pc_knn": (_I, [_P, _I, _P, _P, _P] + [_c.c_float] * 4 + [_I, _I, _I, _c.c_float, _c.c_float, _I, _P, _P, _P]),
    "mvsb200_pc_normals": (_I, [_P, _I, _P, _P, _P] + [_c.c_float] * 4 + [_I, _I, _I, _c.c_float, _c.c_float, _I, _P, _I, _P, _P]),
}

_lib = None


class MvsB200Error(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises MvsB200Error when it is missing or has the wrong ABI."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MvsB200Error(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            f"or `make -C {os.path.dirname(LIB_PATH)}`.  There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise MvsB200Error(f"{LIB_PATH} does not export {name}; rebuild it") from e
        fn.restype, fn.argtypes = res, args
    if lib.mvsb200_abi_version() != ABI_VERSION:
        raise MvsB200Error(f"ABI mismatch: library {lib.mvsb200_abi_version()}, binding {ABI_VERSION}")
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGNATURES)


def call(name, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise MvsB200Error(f"{name} failed ({rc}): {lib.mvsb200_last_error().decode(errors='replace')}")


def launch_count() -> int:
    return int(load().mvsb200_launch_count())
