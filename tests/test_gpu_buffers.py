"""GPU: a handle gives back every buffer it grew.

One handle on two lanes is taken through every buffer that grows after pcop_create: the batched grid scratch, the
single-frame grid and shadow scratch, the PointCloud2 staging and decode descriptors, the partition voxel path's group
buffers and the device pack buffer.  Every result is checked against the oracle.  After the handle is destroyed, a
second run of the same cycle must leave the free device memory exactly where the first run left it."""
import numpy as np
import pytest

import oracle_lib as O
from parity_util import assert_bits_equal, compare_frames
from pc2_util import LAYOUTS, pack, sensor_poses, to_sensor
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi
from test_gpu_occupancy_batch import _download_frame, check_batch, poses
from test_gpu_pointcloud2_windows import Stream

pytestmark = pytest.mark.gpu

B = 12  # two waves (8 + 4 frames), one per lane


@pytest.fixture
def two_lanes(monkeypatch):
    """waves of about 8 frames dealt to two lanes (read when the handle is created)"""
    monkeypatch.setenv("PCOP_LANES", "2")
    monkeypatch.setenv("PCOP_WAVE_FRAMES", "8")


def check_frames(got, p, clouds, what):
    assert len(got) == len(clouds), what
    for f, g in enumerate(got):
        compare_frames(g, O.process(p, clouds[f]), p, f"{what} frame {f}: ")


def windows(p, world, per, points, seed):
    """B windows of `per` posed messages each, cut from the first `points` points of the world frames"""
    names = list(LAYOUTS)
    sw, ws = sensor_poses(p, B * per, seed)
    payloads, counts, layouts = [], [], []
    for f in range(B):
        cuts = np.linspace(0, points, per + 1).astype(int)
        for j in range(per):
            m = len(counts)
            layouts.append(names[m % len(names)])
            counts.append(int(cuts[j + 1] - cuts[j]))
            payloads.append(pack(to_sensor(world[f, cuts[j]:cuts[j + 1]], ws[m]), layouts[m], seed + m))
    return Stream(payloads, counts, layouts, [False] * len(counts), sw, np.arange(B + 1) * per)


def grow_every_buffer():
    """create a handle, grow every buffer that grows, check every result, destroy the handle"""
    p = synth.params(1)
    p.publish_point_clouds = 0  # (otherwise every output is requested from the start)
    p.outputs = abi.OUT_DEFAULT
    n = synth.points_per_frame(1)
    clouds = synth.frames(1, 300, B)
    counts = np.full(B, n, np.int32)
    ws, sw = poses(p, B, 301)
    with ObstacleProcessor(p, n, max_batch=16) as op:
        q = p.copy()
        # grid scratch: a smaller block size gives more cells per frame; the shadows get more clusters as well
        for rnd, block in enumerate((0.1, 0.05)):
            q.block_size = block
            op.set_params(q)
            frames, grids = op.process_batch_occupancy(clouds, ws, sw)
            plain = op.process_batch(clouds)
            check_batch(q, clouds, counts, ws, sw, frames, grids, plain, f"block {block}")
            check_frames(plain, q, clouds, f"block {block}")
            f0 = int(np.argmax([fr.n_clusters for fr in plain]))
            o = O.process(q, clouds[f0])
            assert o.n_clusters >= 2
            k = o.n_clusters // 2 if rnd == 0 else o.n_clusters
            off, idx = o.cluster_offsets[:k + 1], o.cluster_indices[:o.cluster_offsets[k]]
            grid, cells, row_avg = op.occupancy_grid(clouds[f0])
            og, oc, oa = O.occupancy_grid(q, clouds[f0])
            assert_bits_equal(grid, og, f"block {block}: single-frame grid")
            assert_bits_equal(cells, oc, f"block {block}: single-frame counts")
            assert_bits_equal(row_avg, oa, f"block {block}: single-frame row averages")
            sg, rec, w = op.handle_shadow_casting(grid, o.remaining_cloud, off, idx, ws[f0], sw[f0])
            osg, orec, ow = O.occupancy_shadows(q, og, o.remaining_cloud, off, idx, ws[f0], sw[f0])
            assert_bits_equal(sg, osg, f"block {block}, {k} clusters: shadow grid")
            assert_bits_equal(rec, orec, f"block {block}, {k} clusters: shadow records")
            assert w == ow
        # PointCloud2 staging and decode descriptors: 4x the host payload bytes and 3x the messages per wave
        for per, points in ((1, n // 4), (3, n)):
            s = windows(q, clouds, per, points, 400 + per)
            got = op.process_batch_pointcloud2_windows(s.messages(), s.first, s.transforms)
            check_frames(got, q, [s.concat(f) for f in range(B)], f"{per} messages per window")
        # partition voxel path: a smaller leaf allows about 9x the reduce groups per frame
        q.downsample_size = 0.005
        op.set_params(q)
        check_frames(op.process_batch(clouds), q, clouds, "leaf 0.005")
        # device pack buffer: every output requested, then the results left on the device
        q.outputs = abi.OUT_ALL
        op.set_params(q)
        check_frames(op.process_batch(clouds), q, clouds, "all outputs")
        q.outputs = abi.OUT_ALL | abi.OUT_DEVICE
        op.set_params(q)
        res = op.process_batch_raw(clouds.ctypes.data, n, counts)
        check_frames([_download_frame(op, r) for r in res], q, clouds, "device results")


def test_a_handle_gives_back_every_buffer_it_grew(two_lanes):
    """(the first cycle also loads the modules, which the context keeps: the baseline is taken after it)"""
    torch = pytest.importorskip("torch")
    grow_every_buffer()
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    grow_every_buffer()
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    assert free1 == free0, (free0, free1)
