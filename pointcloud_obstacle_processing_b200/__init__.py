"""B200-native per-frame perception hot path of stateSpaceRobotics/pointcloud_obstacle_processing.

Package contents: csrc/ (hand-written sm_100a kernels + the C ABI of include/pcop.h), api.py (host-side
mirror of the reference's stage wrappers over that ABI), synth/ (synthetic frames for the BASELINE configs).
"""
from ._ctypes_abi import (DepthImageC, FrameFootprints, FrameResult, Params, PointCloud2Frame, OUT_ALL, OUT_CLUSTERS, OUT_CROP, OUT_DEFAULT, OUT_FOOTPRINTS, OUT_OBSTACLES,
                          OUT_PLANE, OUT_REMAINING, OUT_SOR, OUT_VOXEL, WARN_PLANE_BREAK,
                          WARN_RNG_TABLE_EXHAUSTED, WARN_SOR_TOO_FEW_POINTS, WARN_VOXEL_OVERFLOW_FALLBACK)
from .api import (DEPTH_ENCODINGS, DepthImage, ObstacleProcessor, PcopError, PointCloud2Message, load_library, node_windows, params_code_defaults,
                  params_yaml)
from .result import Frame

__all__ = ["ObstacleProcessor", "PcopError", "Frame", "Params", "FrameResult", "PointCloud2Frame",
           "PointCloud2Message", "DepthImage", "DepthImageC", "DEPTH_ENCODINGS", "load_library", "node_windows", "params_yaml",
           "params_code_defaults"]
