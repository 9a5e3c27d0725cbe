"""ctypes mirror of include/pcop.h (POD structs only; no logic)."""
import ctypes as C

MAX_PASSES = 16  # PCOP_MAX_PLANE_PASSES_RECORDED

OK, ERR_BAD_PARAM, ERR_CAPACITY, ERR_CUDA, ERR_INTERNAL = 0, 1, 2, 3, 4
WARN_VOXEL_OVERFLOW_FALLBACK, WARN_SOR_TOO_FEW_POINTS, WARN_PLANE_BREAK, WARN_RNG_TABLE_EXHAUSTED = 1, 2, 4, 8
WARN_SHADOW_DEGENERATE = 16
OCC_BATCH_MAX_CELLS = 1 << 20  # PCOP_OCC_BATCH_MAX_CELLS
OUT_CROP, OUT_VOXEL, OUT_SOR, OUT_PLANE, OUT_REMAINING, OUT_CLUSTERS, OUT_OBSTACLES = 1, 2, 4, 8, 16, 32, 64
OUT_DEFAULT, OUT_ALL = 16 | 32 | 64, 127
OUT_FOOTPRINTS = 128  # per-cluster box + ground-plane convex hull (pcop_last_footprints); not part of OUT_ALL
OUT_DEVICE = 256  # modifier: result arrays stay in device memory (pointers are device pointers)
STAGE_NAMES = ["h2d", "crop", "voxel", "sor", "plane", "cluster", "centroid", "d2h"]


class Params(C.Structure):
    """pcop_params: field names are the params.yaml keys (reference params.yaml:1-31, od.cpp:940-975)."""
    _fields_ = [
        ("x_min", C.c_float), ("x_max", C.c_float), ("y_min", C.c_float), ("y_max", C.c_float),
        ("z_min", C.c_float), ("z_max", C.c_float),
        ("downsample_size", C.c_float),
        ("statistical_outlier_meanK", C.c_int32), ("statistical_outlier_stdDevThres", C.c_float),
        ("plane_segment_dist_thres", C.c_float), ("plane_segment_angle", C.c_int32),
        ("euc_cluster_tolerance", C.c_float), ("euc_min_cluster_size", C.c_int32),
        ("euc_max_cluster_size", C.c_int32),
        ("plane_axis", C.c_float * 3), ("plane_keep_fraction", C.c_double),
        ("plane_max_iterations", C.c_int32), ("plane_probability", C.c_double),
        ("ransac_seed", C.c_uint32), ("optimize_coefficients", C.c_int32),
        ("enable_crop", C.c_int32), ("enable_voxel", C.c_int32), ("enable_sor", C.c_int32),
        ("enable_plane", C.c_int32), ("enable_cluster", C.c_int32),
        ("publish_point_clouds", C.c_int32), ("outputs", C.c_uint32),
        ("accumulate_count", C.c_int32), ("block_size", C.c_float), ("dev_percent", C.c_float),
        ("grid_opacity", C.c_int32), ("downsample_input_data", C.c_int32),
        ("passthrough_filter_enable", C.c_int32), ("convex_hull_alpha", C.c_float),
    ]

    def copy(self):
        other = Params()
        C.memmove(C.byref(other), C.byref(self), C.sizeof(Params))
        return other


class PointCloud2Frame(C.Structure):
    """pcop_pointcloud2_frame: one sensor_msgs/PointCloud2 message (data = host or device address)."""
    _fields_ = [
        ("data", C.c_void_p), ("n_points", C.c_int32), ("point_step", C.c_int32),
        ("off_x", C.c_int32), ("off_y", C.c_int32), ("off_z", C.c_int32), ("is_dense", C.c_int32),
    ]


DEPTH_16UC1, DEPTH_32FC1 = 1, 2  # PCOP_DEPTH_*


class DepthImageC(C.Structure):
    """pcop_depth_image: one sensor_msgs/Image depth image + its pinhole model (data = host or device address)."""
    _fields_ = [
        ("data", C.c_void_p), ("width", C.c_int32), ("height", C.c_int32), ("step", C.c_int32),
        ("encoding", C.c_int32), ("fx", C.c_double), ("fy", C.c_double), ("cx", C.c_double), ("cy", C.c_double),
    ]


class FrameResult(C.Structure):
    """pcop_frame_result."""
    _fields_ = [
        ("status", C.c_int32), ("warnings", C.c_uint32),
        ("n_input", C.c_int32), ("n_crop", C.c_int32), ("n_voxel", C.c_int32), ("n_sor", C.c_int32),
        ("n_remaining", C.c_int32), ("n_clusters", C.c_int32), ("n_cluster_points", C.c_int32),
        ("n_plane_passes", C.c_int32),
        ("plane_pass_points", C.c_int32 * MAX_PASSES), ("plane_pass_inliers", C.c_int32 * MAX_PASSES),
        ("plane_pass_coeff", (C.c_float * 4) * MAX_PASSES),
        ("plane_coeff", C.c_float * 4), ("n_plane_inliers", C.c_int32),
        ("crop_kept_idx", C.POINTER(C.c_int32)),
        ("voxel_keys", C.POINTER(C.c_uint32)),
        ("voxel_centroids", C.POINTER(C.c_float)),
        ("sor_kept_idx", C.POINTER(C.c_int32)),
        ("plane_inlier_idx", C.POINTER(C.c_int32)),
        ("remaining_cloud", C.POINTER(C.c_float)),
        ("remaining_src_idx", C.POINTER(C.c_int32)),
        ("cluster_offsets", C.POINTER(C.c_int32)),
        ("cluster_indices", C.POINTER(C.c_int32)),
        ("obstacles", C.POINTER(C.c_float)),
    ]


class FrameFootprints(C.Structure):
    """pcop_frame_footprints: boxes [C][8], hull CSR over remaining-cloud indices."""
    _fields_ = [
        ("n_clusters", C.c_int32), ("n_hull_vertices", C.c_int32),
        ("boxes", C.POINTER(C.c_float)),
        ("hull_offsets", C.POINTER(C.c_int32)),
        ("hull_indices", C.POINTER(C.c_int32)),
    ]
