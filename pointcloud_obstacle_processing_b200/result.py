"""numpy view of a pcop_frame_result (copies out of the handle-owned pinned buffers)."""
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

from ._ctypes_abi import FrameFootprints, FrameResult, MAX_PASSES


def _arr(ptr, n, dtype, cols=None):
    if not ptr or n < 0:
        return None
    count = n * (cols or 1)
    if count == 0:
        a = np.zeros((0,), dtype=dtype)
    else:
        a = np.ctypeslib.as_array(ptr, shape=(count,)).astype(dtype, copy=True)
    return a.reshape(n, cols) if cols else a


@dataclass
class Frame:
    """One frame's outputs: counts N,M,V,S,P,C,L plus the arrays that were requested.

    `clusters` is the std::vector<pcl::PointIndices> of od.cpp:793 (indices into
    `remaining_cloud` = planar_cloud_y, od.cpp:765); `obstacles` is the
    PointIndicesArray.points payload (msg/PointWithRad.msg:1-4).  With outputs | OUT_FOOTPRINTS, `boxes` (C, 8) holds
    every cluster's {min x, min y, min z, 0, max x, max y, max z, 0} and `hull_offsets` / `hull_indices` the CSR of its
    ground-plane convex hull (counter-clockwise, indices into `remaining_cloud`); None otherwise.
    """
    status: int = 0
    warnings: int = 0
    n_input: int = 0
    n_crop: int = 0
    n_voxel: int = 0
    n_sor: int = 0
    n_remaining: int = 0
    n_clusters: int = 0
    n_cluster_points: int = 0
    n_plane_passes: int = 0
    plane_pass_points: List[int] = field(default_factory=list)
    plane_pass_inliers: List[int] = field(default_factory=list)
    plane_pass_coeff: Optional[np.ndarray] = None
    plane_coeff: Optional[np.ndarray] = None
    n_plane_inliers: int = 0
    crop_kept_idx: Optional[np.ndarray] = None
    voxel_keys: Optional[np.ndarray] = None
    voxel_centroids: Optional[np.ndarray] = None
    sor_kept_idx: Optional[np.ndarray] = None
    plane_inlier_idx: Optional[np.ndarray] = None
    remaining_cloud: Optional[np.ndarray] = None
    remaining_src_idx: Optional[np.ndarray] = None
    cluster_offsets: Optional[np.ndarray] = None
    cluster_indices: Optional[np.ndarray] = None
    obstacles: Optional[np.ndarray] = None
    boxes: Optional[np.ndarray] = None
    hull_offsets: Optional[np.ndarray] = None
    hull_indices: Optional[np.ndarray] = None

    @property
    def hulls(self):
        """one index array per cluster: its hull vertices, counter-clockwise (None without OUT_FOOTPRINTS)"""
        if self.hull_offsets is None or self.hull_indices is None:
            return None
        o = self.hull_offsets
        return [self.hull_indices[o[k]:o[k + 1]] for k in range(len(o) - 1)]

    def set_footprints(self, fp: FrameFootprints):
        """copies the footprint arrays of a (host) pcop_frame_footprints; NULL pointers leave them None"""
        self.boxes = _arr(fp.boxes, fp.n_clusters, np.float32, 8)
        self.hull_offsets = _arr(fp.hull_offsets, fp.n_clusters + 1, np.int32)
        self.hull_indices = _arr(fp.hull_indices, fp.n_hull_vertices, np.int32)
        return self

    @property
    def clusters(self):
        if self.cluster_offsets is None or self.cluster_indices is None:
            return None
        o = self.cluster_offsets
        return [self.cluster_indices[o[k]:o[k + 1]] for k in range(self.n_clusters)]

    @staticmethod
    def from_c(r: FrameResult) -> "Frame":
        npass = min(r.n_plane_passes, MAX_PASSES)
        return Frame(
            status=r.status, warnings=r.warnings, n_input=r.n_input, n_crop=r.n_crop, n_voxel=r.n_voxel,
            n_sor=r.n_sor, n_remaining=r.n_remaining, n_clusters=r.n_clusters,
            n_cluster_points=r.n_cluster_points, n_plane_passes=r.n_plane_passes,
            plane_pass_points=list(r.plane_pass_points)[:npass],
            plane_pass_inliers=list(r.plane_pass_inliers)[:npass],
            plane_pass_coeff=np.array([list(r.plane_pass_coeff[k]) for k in range(npass)],
                                      dtype=np.float32).reshape(npass, 4),
            plane_coeff=np.array(list(r.plane_coeff), dtype=np.float32),
            n_plane_inliers=r.n_plane_inliers,
            crop_kept_idx=_arr(r.crop_kept_idx, r.n_crop, np.int32),
            voxel_keys=_arr(r.voxel_keys, r.n_voxel, np.uint32),
            voxel_centroids=_arr(r.voxel_centroids, r.n_voxel, np.float32, 4),
            sor_kept_idx=_arr(r.sor_kept_idx, r.n_sor, np.int32),
            plane_inlier_idx=_arr(r.plane_inlier_idx, r.n_plane_inliers, np.int32),
            remaining_cloud=_arr(r.remaining_cloud, r.n_remaining, np.float32, 4),
            remaining_src_idx=_arr(r.remaining_src_idx, r.n_remaining, np.int32),
            cluster_offsets=_arr(r.cluster_offsets, r.n_clusters + 1, np.int32),
            cluster_indices=_arr(r.cluster_indices, r.n_cluster_points, np.int32),
            obstacles=_arr(r.obstacles, r.n_clusters, np.float32, 4),
        )
