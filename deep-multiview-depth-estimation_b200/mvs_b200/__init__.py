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
from .fusion import fuse_depth_maps, visibility_fusion, infer_scene, write_ply, read_ply, point_viewpoints  # noqa: F401
from .evaluation import thin_points, nearest_distance, nearest_neighbour, k_nearest, evaluate_point_cloud, load_dtu_eval  # noqa: F401
from .normals import estimate_normals  # noqa: F401
from .tanks import (CropVolume, read_crop_volume, crop_points, voxel_down_sample, evaluate_tanks_and_temples,  # noqa: F401
                    load_tnt_eval, Mapping, read_trajectory, write_trajectory, read_mapping, load_tnt_trajectory, camera_poses,
                    write_evaluation_files)
from .registration import (uniform_down_sample, icp_point_to_point, register_tanks_and_temples,  # noqa: F401
                           trajectory_points, align_trajectory)

__all__ = ["homography_warping", "assemble_cost_volume", "extract_depth_map", "CostVolumeReg",
           "WarpedFeatureVolumes", "PlaneSweep", "warp_variance", "warp_materialize", "softmax_depth",
           "softmax_over_depth", "depth_from_prob", "refine_depth", "encode_features", "FrozenMVSNet", "depth_confidence",
           "fuse_depth_maps", "visibility_fusion", "infer_scene", "write_ply", "read_ply", "thin_points", "nearest_distance",
           "nearest_neighbour", "evaluate_point_cloud", "load_dtu_eval", "CropVolume", "read_crop_volume", "crop_points",
           "voxel_down_sample",
           "evaluate_tanks_and_temples", "load_tnt_eval", "uniform_down_sample", "icp_point_to_point", "register_tanks_and_temples",
           "Mapping", "read_trajectory", "write_trajectory", "read_mapping", "load_tnt_trajectory", "camera_poses",
           "trajectory_points", "align_trajectory", "k_nearest", "estimate_normals", "point_viewpoints", "write_evaluation_files",
           "MvsB200Error", "launch_count", "load_library"]
