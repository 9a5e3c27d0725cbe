"""GPU: every output bit on its own, and two mixes, over a call of several waves on two lanes.

Each requested array, footprints included, equals byte for byte the same array of an OUT_ALL | OUT_FOOTPRINTS call on
the same frames, with results on the host and with OUT_DEVICE; every array not requested is NULL; counts and plane
records do not depend on the mask."""
import ctypes as C

import numpy as np
import pytest

from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi

pytestmark = pytest.mark.gpu

# (field, output bit, elements, element bytes): r is the frame's result, fp its footprints
ARRAYS = [
    ("crop_kept_idx", abi.OUT_CROP, lambda r, fp: r.n_crop, 4),
    ("voxel_keys", abi.OUT_VOXEL, lambda r, fp: r.n_voxel, 4),
    ("voxel_centroids", abi.OUT_VOXEL, lambda r, fp: r.n_voxel, 16),
    ("sor_kept_idx", abi.OUT_SOR, lambda r, fp: r.n_sor, 4),
    ("plane_inlier_idx", abi.OUT_PLANE, lambda r, fp: r.n_plane_inliers, 4),
    ("remaining_cloud", abi.OUT_REMAINING, lambda r, fp: r.n_remaining, 16),
    ("remaining_src_idx", abi.OUT_REMAINING, lambda r, fp: r.n_remaining, 4),
    ("cluster_offsets", abi.OUT_CLUSTERS, lambda r, fp: r.n_clusters + 1, 4),
    ("cluster_indices", abi.OUT_CLUSTERS, lambda r, fp: r.n_cluster_points, 4),
    ("obstacles", abi.OUT_OBSTACLES, lambda r, fp: r.n_clusters, 16),
    ("boxes", abi.OUT_FOOTPRINTS, lambda r, fp: fp.n_clusters, 32),
    ("hull_offsets", abi.OUT_FOOTPRINTS, lambda r, fp: fp.n_clusters + 1, 4),
    ("hull_indices", abi.OUT_FOOTPRINTS, lambda r, fp: fp.n_hull_vertices, 4),
]
MASKS = [abi.OUT_CROP, abi.OUT_VOXEL, abi.OUT_SOR, abi.OUT_PLANE, abi.OUT_REMAINING, abi.OUT_CLUSTERS,
         abi.OUT_OBSTACLES, abi.OUT_FOOTPRINTS, abi.OUT_VOXEL | abi.OUT_FOOTPRINTS, abi.OUT_CROP | abi.OUT_OBSTACLES]
FRAMES = 40


@pytest.fixture
def two_lanes(monkeypatch):
    monkeypatch.setenv("PCOP_LANES", "2")
    monkeypatch.setenv("PCOP_WAVE_FRAMES", "8")


def params(outputs):
    p = synth.params(2)
    p.publish_point_clouds = 0  # (1 would request OUT_ALL whatever the mask)
    p.enable_sor = 1
    p.outputs = outputs
    return p


def frames():
    clouds = synth.frames(2, 11, FRAMES)
    n = clouds.shape[1]
    counts = np.random.default_rng(3).integers(n // 4, n + 1, FRAMES).astype(np.int32)
    counts[5] = 0
    counts[17] = n
    return clouds, counts


def collect(op, res, device):
    """per frame: (the counts and plane records, the footprint counts, {field: bytes, or None for a NULL pointer})"""
    head = abi.FrameResult.crop_kept_idx.offset  # (every count and plane record lies before the first pointer)
    out = []
    for f, r in enumerate(res):
        fp = op.last_footprints(f)
        arrays = {}
        for field, bit, count, size in ARRAYS:
            ptr = C.cast(getattr(fp if bit == abi.OUT_FOOTPRINTS else r, field), C.c_void_p).value
            nbytes = count(r, fp) * size
            if ptr is None:
                arrays[field] = None
            elif device:
                arrays[field] = op.download(ptr, nbytes, np.uint8).tobytes()
            else:
                arrays[field] = C.string_at(ptr, nbytes)
        out.append((C.string_at(C.addressof(r), head), (fp.n_clusters, fp.n_hull_vertices), arrays))
    return out


@pytest.mark.parametrize("mask", MASKS, ids=lambda m: f"outputs_{m}")
def test_requested_arrays_equal_the_full_call(two_lanes, mask):
    clouds, counts = frames()
    n = clouds.shape[1]
    with ObstacleProcessor(params(abi.OUT_ALL | abi.OUT_FOOTPRINTS), n, max_batch=16) as op:
        want = collect(op, op.process_batch_raw(clouds.ctypes.data, n, counts), False)
        assert all(a is not None for _, _, arrays in want for a in arrays.values())
        assert sum(fc[0] for _, fc, _ in want) > 0 and want[5][2]["remaining_cloud"] == b""
        for device in (False, True):
            what = f"outputs {mask}" + (" | OUT_DEVICE" if device else "")
            op.set_params(params(mask | (abi.OUT_DEVICE if device else 0)))
            got = collect(op, op.process_batch_raw(clouds.ctypes.data, n, counts), device)
            for f, ((g_head, g_fp, g_arrays), (w_head, w_fp, w_arrays)) in enumerate(zip(got, want)):
                assert g_head == w_head, f"{what} frame {f}: counts or plane records differ"
                assert g_fp == (w_fp if mask & abi.OUT_FOOTPRINTS else (w_fp[0], 0)), f"{what} frame {f}: footprint counts"
                for field, bit, _, _ in ARRAYS:
                    if mask & bit:
                        assert g_arrays[field] == w_arrays[field], f"{what} frame {f}: {field} differs"
                    else:
                        assert g_arrays[field] is None, f"{what} frame {f}: {field} not requested but not NULL"
