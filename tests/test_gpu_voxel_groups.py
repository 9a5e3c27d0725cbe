"""Partition voxel path: groups of the reduce kernel at its limits -- up to 128 buckets (the bitmap's 262 144 keys at
S = 11) and exactly 2048 elements -- bit for bit against the oracle, with the partition kernels doing the work."""
import numpy as np
import pytest

import oracle_lib as O
from parity_util import assert_bits_equal
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
from test_gpu_parity import _voxel_only

pytestmark = pytest.mark.gpu

N = 120000                      # points per frame: 2^14 buckets of 2^11 keys for the 25-bit config-2 keys
NX, NY, NZ = 801, 801, 41       # cells of the config-2 crop box at 0.1 m
B0 = np.array([-400, -400, -25])
S, K, EMAX = 11, 128, 2048


def _points(keys, rng, jitter=(0.2, 0.8)):
    """one point inside each voxel of `keys` (composite key of the crop box's cells)"""
    keys = np.asarray(keys, np.int64)
    c = np.stack([keys % NX, keys // NX % NY, keys // (NX * NY)], axis=1) + B0
    return ((c + rng.uniform(*jitter, size=c.shape)) * 0.1).astype(np.float32)


def _layer_keys(rng, n, cz0, cz1):
    return rng.integers(0, NX * NY, size=n) + NX * NY * rng.integers(cz0, cz1, size=n)


def _frame(rng, *parts):
    """the parts, then points outside the crop box up to N, in random order (original index order != key order)"""
    xyz = np.concatenate(parts)
    fill = np.full((N - len(xyz), 3), 100.0, np.float32)
    xyz = np.concatenate([xyz, fill])[rng.permutation(N)]
    return np.concatenate([xyz, np.ones((N, 1), np.float32)], axis=1)


def _groups(cloud):
    """(buckets, elements, bucket id span) of every group of k_vp_scan's greedy rule, from the survivors' keys"""
    x = cloud[:, :3]
    keep = (x[:, 0] >= -40) & (x[:, 0] <= 40) & (x[:, 1] >= -40) & (x[:, 1] <= 40) & (x[:, 2] >= -2.5) & (x[:, 2] <= 1.5)
    c = np.floor(x[keep] * np.float32(10.0)).astype(np.int64) - B0
    cnt = np.bincount((c[:, 0] + NX * (c[:, 1] + NY * c[:, 2])) >> S)
    out, kb, e, b0 = [], 0, 0, 0
    for b in np.flatnonzero(cnt):
        if kb and (e + cnt[b] > EMAX or kb >= K):
            out.append((kb, e, b_last - b0))
            kb, e = 0, 0
        if not kb:
            b0 = b
        kb, e, b_last = kb + 1, e + cnt[b], b
    return out + [(kb, e, b_last - b0)]


def _runs(rng, keys, lo, hi):
    """lo .. hi - 1 points in each voxel of `keys`"""
    return np.repeat(np.asarray(keys), rng.integers(lo, hi, size=len(keys)))


def test_voxel_partition_groups_at_the_bucket_and_element_limits():
    p = _voxel_only(synth.params(2))
    rng = np.random.default_rng(125)
    bg = _layer_keys(rng, 20000, 0, 10)  # background below z = -1.5 m: a few points per bucket
    frames = []
    # sparse buckets of one z layer: groups of 128 buckets (direct bucket table), runs of 3-7 points
    layer = _layer_keys(rng, 3000, 20, 21)
    frames.append(_frame(rng, _points(layer, rng), _points(_runs(rng, layer[:80], 3, 8), rng)))
    # 250 buckets over the whole box: groups of 128 buckets whose ids span more than the direct table (binary search)
    wide = _layer_keys(rng, 250, 0, NZ)
    frames.append(_frame(rng, _points(wide, rng), _points(_runs(rng, wide[:25], 3, 6), rng)))
    # one bucket of exactly 2048 points over ~1300 voxels
    b = (25 * NX * NY >> S) + 10
    keys = rng.integers(b << S, (b + 1) << S, size=2 * EMAX)
    keys = keys[(keys % NX != NX - 1) & (keys // NX % NY != NY - 1)][:EMAX]  # (the last cell of x / y is cropped)
    frames.append(_frame(rng, _points(keys, rng), _points(bg, rng)))
    # one voxel holding a whole 2048-point bucket
    frames.append(_frame(rng, _points(np.full(EMAX, 30 * NX * NY + 123 * NX + 456), rng, (0.05, 0.95)), _points(bg, rng)))

    groups = [_groups(f) for f in frames]
    assert groups[0][0][0] == K and groups[0][0][2] < 4096       # (the table spans 4096 bucket ids)
    assert groups[1][0][0] == K and groups[1][0][2] >= 4096
    assert (1, EMAX, 0) in groups[2] and (1, EMAX, 0) in groups[3]

    clouds = np.stack(frames)
    with ObstacleProcessor(p, N, max_batch=len(frames)) as op:
        op.enable_kernel_timing(True)
        res = op.process_batch(clouds, np.full(len(frames), N, np.int32))
        names = op.kernel_times()
    assert "k_vp_reduce" in names and "k_vf_reduce" not in names, sorted(names)
    for f in range(len(frames)):
        o = O.process(p, clouds[f])
        assert res[f].n_crop == o.n_crop and res[f].n_voxel == o.n_voxel, (f, res[f].n_crop, o.n_crop, res[f].n_voxel, o.n_voxel)
        assert_bits_equal(res[f].voxel_keys, o.voxel_keys, f"frame {f} voxel keys")
        assert_bits_equal(res[f].voxel_centroids, o.voxel_centroids, f"frame {f} voxel centroids")
