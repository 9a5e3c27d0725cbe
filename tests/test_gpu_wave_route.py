"""GPU: the route of a batched wave (which crop + voxel, plane and clustering kernels it launches) and its repeats.

A wave's first route is a guess from what the lane's earlier waves needed; once the wave's counts are back, each part
a wrong guess left undone runs again.  Kernel timing runs every wave on one lane, and its launch counts per kernel
show the route that ran and how often: every run of a wave's back half ends with one k_pack_scan."""
import numpy as np
import pytest

import oracle_lib as O
from parity_util import compare_frames
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
from test_gpu_occupancy_batch import _frames_needing_repeats, assert_same_frame

pytestmark = pytest.mark.gpu

PLANE_SMALL_TIER_MAX = 65536  # plane-stage inputs the small tier of the plane kernel takes
ECE_SMALL_MAX = 8960          # remaining clouds the fused clustering kernel takes


def launches(op):
    return {k: n for k, (_, n) in op.kernel_times().items()}


@pytest.mark.parametrize("kind,kernel", [("plane", "k_plane_loop_large"), ("cluster", "k_ece_route"),
                                         ("plane_windows", "k_plane_loop_windows")])
def test_history_carries_over_to_the_next_call(kind, kernel, monkeypatch):
    """a call whose one wave repeats its plane stage (its clustering) leaves that in the lane's history: the same call
    again launches the large plane tier (the generic clustering kernels) up front and repeats nothing.  plane_windows:
    BASELINE configs[2] frame 1 reaches the plane stage with 132404 points, above 8 slices of the large tier (its
    remaining cloud of 26224 points repeats the clustering too, its dense voxel buckets may repeat the voxel stage)"""
    if kind == "plane_windows":
        p = synth.params(3)
        clouds = synth.frames(3, 1, 1)
        counts = np.full(1, clouds.shape[1], np.int32)
    else:
        p, clouds, counts, _ = _frames_needing_repeats(kind, monkeypatch)
    B = len(counts)
    with ObstacleProcessor(p, clouds.shape[1], max_batch=B) as op:  # (one wave per call: the history is its last wave's)
        op.enable_kernel_timing(True)
        first = op.process_batch(clouds, counts)
        guessed = launches(op)
        op.enable_kernel_timing(True)  # (starts the totals over)
        second = op.process_batch(clouds, counts)
        learned = launches(op)
    assert kernel in guessed and guessed["k_pack_scan"] > 1, guessed
    assert kernel in learned and learned["k_pack_scan"] == 1, learned
    plane_kernels = {k for k in guessed.keys() | learned.keys() if k.startswith("k_plane")}
    assert plane_kernels <= {"k_plane_gen0", "k_plane_loop", "k_plane_loop_large", "k_plane_loop_windows",
                             "k_plane_record"}, plane_kernels  # (every pass inside the cluster kernels)
    for f in range(B):
        assert_same_frame(second[f], first[f], 0, f"{kind} frame {f}")


def test_one_wave_repeated_from_its_upload_and_from_its_plane_stage():
    """a crop survivor with a NaN y (the fused voxel path declines its frame) in the same wave as plane-stage inputs
    above the small resident tier: the wave runs again from its upload with the generic crop + voxel kernels, then
    again from the plane stage with the large tier, and every frame equals the oracle's"""
    p = synth.params(2)
    p.downsample_size = 0.04  # (about 89 000 points reach the plane stage; the fused voxel paths still apply)
    clouds = synth.frames(2, 20, 2).copy()
    clouds[1, O.crop(p, clouds[1])[1][100], 1] = np.nan
    counts = np.full(2, clouds.shape[1], np.int32)
    with ObstacleProcessor(p, clouds.shape[1], max_batch=2) as op:
        op.enable_kernel_timing(True)
        got = op.process_batch(clouds, counts)
        n = launches(op)
    # (the premises: a plane-stage input above the small tier, no remaining cloud above the fused clustering limit)
    assert PLANE_SMALL_TIER_MAX < max(r.n_sor for r in got)
    assert max(r.n_remaining for r in got) <= ECE_SMALL_MAX
    assert any(k.startswith(("k_vp_", "k_vf_")) for k in n), n  # first run: a fused voxel path
    assert n["k_voxel_keys"] == 1, n                            # repeat from the upload: the generic voxel kernels
    assert n["k_plane_loop_large"] == 1, n                      # repeat from the plane stage: the large tier
    assert n["k_pack_scan"] == 3, n
    for f in range(2):
        compare_frames(got[f], O.process(p, clouds[f, :counts[f]]), p, f"frame {f}: ")
