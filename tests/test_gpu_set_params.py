"""GPU: pcop_set_params on a handle with several lanes.  Every lane must run the new parameters, and the partition
voxel path's buffers must follow the plan of the new parameters (they were sized at create before)."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle_lib as O
from parity_util import compare_frames
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, params_yaml

pytestmark = pytest.mark.gpu

B = 20  # three waves of about 8 frames: every lane of a 2- or 3-lane handle runs one


@pytest.fixture(params=[2, 3])
def lanes(request, monkeypatch):
    """waves of about 8 frames dealt to 2 or 3 lanes (read when the handle is created)"""
    monkeypatch.setenv("PCOP_LANES", str(request.param))
    monkeypatch.setenv("PCOP_WAVE_FRAMES", "8")
    return request.param


@pytest.fixture
def three_lanes(monkeypatch):
    monkeypatch.setenv("PCOP_LANES", "3")
    monkeypatch.setenv("PCOP_WAVE_FRAMES", "8")


def box_frames(p, n, seed):
    """B frames of n points uniform in the crop box, 30 % of them on a noisy ground plane"""
    rng = np.random.default_rng(seed)
    lo = np.array([p.x_min, p.y_min, p.z_min], np.float32)
    hi = np.array([p.x_max, p.y_max, p.z_max], np.float32)
    clouds = np.ones((B, n, 4), np.float32)
    clouds[:, :, :3] = rng.uniform(lo, hi, size=(B, n, 3))
    m = int(0.3 * n)
    clouds[:, :m, 2] = -0.3 + rng.normal(0.0, 0.002, size=(B, m))
    return clouds


def check(op, clouds, what):
    p = op.params.copy()
    res = op.process_batch(clouds)
    with ThreadPoolExecutor(8) as ex:
        oracle = list(ex.map(lambda f: O.process(p, clouds[f]), range(B)))
    for f in range(B):
        compare_frames(res[f], oracle[f], p, f"{what} frame {f}: ")


def test_voxel_enabled_after_create(lanes):
    """created without the voxel stage (no partition-path buffers), then set to the partition plan"""
    p = params_yaml()
    off = p.copy()
    off.enable_voxel = 0
    clouds = box_frames(p, 30000, 1)
    with ObstacleProcessor(off, 30000, max_batch=24) as op:
        op.set_params(p)
        check(op, clouds, "voxel on")


def test_leaf_shrunk_after_create(lanes):
    """leaf 0.05 at create (at most 133 reduce groups per frame), then 0.005: about 390 groups per frame"""
    p = params_yaml()
    coarse = p.copy()
    coarse.downsample_size = 0.05
    fine = p.copy()
    fine.downsample_size = 0.005
    clouds = box_frames(p, 100000, 2)
    with ObstacleProcessor(coarse, 100000, max_batch=24) as op:
        op.set_params(fine)
        check(op, clouds, "leaf 0.005")


def test_leaf_changed_between_calls(three_lanes):
    p = params_yaml()
    clouds = box_frames(p, 20000, 3)
    with ObstacleProcessor(p, 20000, max_batch=24) as op:
        check(op, clouds, "leaf 0.015")
        q = p.copy()
        q.downsample_size = 0.03
        op.set_params(q)
        check(op, clouds, "leaf 0.03")


def test_ransac_seed_changed_between_calls(three_lanes):
    p = params_yaml()
    clouds = box_frames(p, 20000, 4)
    with ObstacleProcessor(p, 20000, max_batch=24) as op:
        check(op, clouds, "seed 12345")
        q = p.copy()
        q.ransac_seed = 987654321
        op.set_params(q)
        check(op, clouds, "seed 987654321")
