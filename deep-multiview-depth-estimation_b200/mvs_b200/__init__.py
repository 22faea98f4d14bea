"""mvs_b200 -- B200-native (sm_100a) plane-sweep path of MVSNet behind the reference's Python interfaces.

    from mvs_b200 import homography_warping, assemble_cost_volume, extract_depth_map, CostVolumeReg

Everything computes in libmvs_b200.so (C ABI: include/mvs_b200.h); importing this package without the built
library raises at first use -- there is no CPU or pure-PyTorch fallback for the ops.
"""
from ._lib import MvsB200Error, LIB_PATH, launch_count, load as load_library  # noqa: F401
from .api import homography_warping, assemble_cost_volume, extract_depth_map  # noqa: F401
from .handle import WarpedFeatureVolumes  # noqa: F401
from .ops import PlaneSweep, warp_variance, warp_materialize, softmax_depth, softmax_over_depth, depth_from_prob  # noqa: F401
from .regulariser import CostVolumeReg, central_region  # noqa: F401
from . import conv3d_sm100  # noqa: F401  (registers the tcgen05 convolution backend)
from .refine import refine_depth  # noqa: F401
from .nets2d import encode_features  # noqa: F401
from .frozen import FrozenMVSNet  # noqa: F401
from .ops import depth_confidence  # noqa: F401
from .fusion import fuse_depth_maps, visibility_fusion, infer_scene, write_ply, read_ply  # noqa: F401
from .evaluation import thin_points, nearest_distance, evaluate_point_cloud, load_dtu_eval  # noqa: F401

__all__ = ["homography_warping", "assemble_cost_volume", "extract_depth_map", "CostVolumeReg",
           "WarpedFeatureVolumes", "PlaneSweep", "warp_variance", "warp_materialize", "softmax_depth",
           "softmax_over_depth", "depth_from_prob", "refine_depth", "encode_features", "FrozenMVSNet", "depth_confidence",
           "fuse_depth_maps", "visibility_fusion", "infer_scene", "write_ply", "read_ply", "thin_points", "nearest_distance",
           "evaluate_point_cloud", "load_dtu_eval", "MvsB200Error", "launch_count", "load_library"]
