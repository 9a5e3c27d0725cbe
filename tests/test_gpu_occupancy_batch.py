"""GPU: pcop_process_batch_occupancy, the pipeline and the occupancy grid the node publishes for every frame of a batch.

Every grid is checked byte for byte against the oracle chain occupancy_grid -> process -> occupancy_shadows with the
frame's own pose; every frame result against a pcop_process_batch call on the same frames."""
import ctypes as C
import dataclasses
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle_lib as O
from parity_util import assert_bits_equal, compare_frames
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, PcopError, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi
from pointcloud_obstacle_processing_b200.result import Frame
from shadow_util import rigid

pytestmark = pytest.mark.gpu


@pytest.fixture
def two_lanes(monkeypatch):
    """waves of about 8 frames dealt to two lanes (read when the handle is created)"""
    monkeypatch.setenv("PCOP_LANES", "2")
    monkeypatch.setenv("PCOP_WAVE_FRAMES", "8")


def poses(p, B, seed):
    """one sensor pose per frame, looking back into the crop box: (world_to_sensor [B, 4, 4], sensor_to_world [B, 4, 4])"""
    rng = np.random.default_rng(seed)
    ws, sw = [], []
    for _ in range(B):
        m, inv = rigid(rng.uniform(-0.3, 0.3), rng.uniform(0.3, 0.6), 0.0,
                       [p.x_max + rng.uniform(0.2, 1.5), 0.5 * (p.y_min + p.y_max) + rng.uniform(-1.0, 1.0),
                        rng.uniform(0.8, 1.6)])
        sw.append(m)
        ws.append(inv)
    return np.stack(ws), np.stack(sw)


def oracle_grids(p, clouds, counts, ws, sw):
    """[(grid, warnings)] of the oracle chain, per frame"""
    def one(f):
        cloud = clouds[f, :counts[f]]
        g0, _, _ = O.occupancy_grid(p, cloud)
        o = O.process(p, cloud)
        g, _, w = O.occupancy_shadows(p, g0, o.remaining_cloud, o.cluster_offsets, o.cluster_indices, ws[f], sw[f])
        return g, w
    with ThreadPoolExecutor(8) as ex:
        return list(ex.map(one, range(len(counts))))


def assert_same_frame(g, want, shadow_warning, what):
    """every field of g equals want's; warnings: want's plus the shadow bit where the oracle skipped a fan"""
    assert g.warnings == want.warnings | (abi.WARN_SHADOW_DEGENERATE if shadow_warning else 0), what
    for fld in dataclasses.fields(Frame):
        if fld.name == "warnings":
            continue
        a, b = getattr(g, fld.name), getattr(want, fld.name)
        if isinstance(b, np.ndarray) or isinstance(a, np.ndarray):
            assert a is not None and b is not None, f"{what}: {fld.name}"
            assert_bits_equal(a, b, f"{what}: {fld.name}")
        else:
            assert a == b, f"{what}: {fld.name}: {a} != {b}"


def check_batch(p, clouds, counts, ws, sw, frames, grids, plain, what):
    oracle = oracle_grids(p, clouds, counts, ws, sw)
    for f in range(len(counts)):
        og, ow = oracle[f]
        assert_same_frame(frames[f], plain[f], ow, f"{what} frame {f}")
        assert_bits_equal(grids[f], og, f"{what} frame {f}: grid")
    return oracle


@pytest.mark.parametrize("block_size,count_kernel", [(0.25, "k_occ_count_wave_s16"), (0.1, "k_occ_count_wave_g")])
def test_config2_frames_over_waves_and_lanes(block_size, count_kernel, two_lanes):
    """64 distinct HDL-64 frames, each with its own pose, over several waves on two lanes; grids into numpy, pinned
    and device memory.  320 x 320 cells count in 16-bit shared-memory counters, 800 x 800 in global memory."""
    torch = pytest.importorskip("torch")
    p = synth.params(2)
    p.block_size = block_size
    p.grid_opacity = 40
    n = synth.points_per_frame(2)
    B = 64
    clouds = synth.frames(2, 3000, B)
    counts = np.full(B, n, np.int32)
    ws, sw = poses(p, B, 1)
    with ObstacleProcessor(p, n, max_batch=16) as op:
        W, H = op.occupancy_dims()
        plain = op.process_batch(clouds)
        d2h_plain = op.last_d2h_bytes
        frames, grids = op.process_batch_occupancy(clouds, ws, sw)
        d2h_host = op.last_d2h_bytes
        pinned = torch.empty((B, H, W), dtype=torch.int8).pin_memory()
        res = op.process_batch_occupancy_raw(clouds.ctypes.data, n, counts, ws, sw, pinned.data_ptr())
        pinned_frames = [Frame.from_c(r) for r in res]
        dev = torch.full((B, H, W), 7, dtype=torch.int8, device="cuda")
        op.process_batch_occupancy_raw(clouds.ctypes.data, n, counts, ws, sw, dev.data_ptr())
        d2h_dev = op.last_d2h_bytes
        g_dev = dev.cpu().numpy()
        op.enable_kernel_timing(True)
        op.process_batch_occupancy(clouds[:2], ws[:2], sw[:2])
        names = op.kernel_times()
    assert count_kernel in names and "k_occ_threshold_wave" in names and "k_occ_mark" in names, sorted(names)
    assert d2h_host - d2h_dev == B * W * H and d2h_dev == d2h_plain
    oracle = check_batch(p, clouds, counts, ws, sw, frames, grids, plain, "numpy")
    for f in range(B):
        assert_same_frame(pinned_frames[f], plain[f], oracle[f][1], f"pinned frame {f}")
        assert_bits_equal(pinned.numpy()[f], oracle[f][0], f"pinned frame {f}: grid")
        assert_bits_equal(g_dev[f], oracle[f][0], f"device frame {f}: grid")
    assert sum(int((g == 40).sum()) for g, _ in oracle) > 0 and sum(int((g == 100).sum()) for g, _ in oracle) > 0


def test_config1_ragged_batch():
    """params.yaml (101 x 120 cells: 32-bit shared-memory counters); frames of different sizes, an empty one and a
    3-point one"""
    p = synth.params(1)
    p.outputs = abi.OUT_ALL
    p.grid_opacity = 25
    n = synth.points_per_frame(1)
    clouds = synth.frames(1, 50, 7)
    counts = np.array([n, n - 1777, 20000, 0, 3, n, 12345], np.int32)
    ws, sw = poses(p, 7, 2)
    with ObstacleProcessor(p, n, max_batch=3) as op:
        plain = op.process_batch(clouds, counts)
        frames, grids = op.process_batch_occupancy(clouds, ws, sw, counts)
        op.enable_kernel_timing(True)
        op.process_batch_occupancy(clouds[:1], ws[:1], sw[:1])
        assert "k_occ_count_wave_s32" in op.kernel_times()
    check_batch(p, clouds, counts, ws, sw, frames, grids, plain, "config 1")


def _frames_needing_repeats(kind, monkeypatch):
    """(params, clouds, counts, max_batch) of a batch whose first pass is repeated inside the wave"""
    if kind == "cluster":  # remaining clouds on both sides of the fused clustering kernel's limit
        monkeypatch.setenv("PCOP_ECE_SMALL_MAX", "4500")
        p = synth.params(2)
        n = synth.points_per_frame(2)
        return p, synth.frames(2, 10, 5), np.array([n, n - 1777, 50000, 0, 3], np.int32), 2
    if kind == "voxel":  # a crop survivor with a NaN y: the fused voxel path declines the frame
        p = synth.params(2)
        n = synth.points_per_frame(2)
        clouds = synth.frames(2, 200, 3).copy()
        kept = O.crop(p, clouds[1])[1]
        clouds[1, kept[100], 1] = np.nan
        clouds[1, kept[5000], 2] = np.nan
        return p, clouds, np.full(3, n, np.int32), 3
    # plane: HDL-64 frames with a 2 cm voxel leaf reach the plane stage with about 100 000 points, above the resident
    # plane kernel's small tier (the first wave of a handle speculates on that tier)
    p = synth.params(2)
    p.downsample_size = 0.02
    clouds = synth.frames(2, 20, 3)
    return p, clouds, np.full(3, clouds.shape[1], np.int32), 3


@pytest.mark.parametrize("kind", ["cluster", "voxel", "plane"])
def test_speculation_repeats_rebuild_the_grids(kind, monkeypatch):
    """the wave engine repeats a wave's back half (clustering, plane stage) or the whole wave (voxel decline) when a
    frame outgrew the path it guessed; the kernel launches show that the repeat happened, and the grids of the repeated
    waves still match"""
    p, clouds, counts, max_batch = _frames_needing_repeats(kind, monkeypatch)
    p.grid_opacity = 60
    p.block_size = 0.25
    B = len(counts)
    ws, sw = poses(p, B, 3)
    with ObstacleProcessor(p, clouds.shape[1], max_batch=max_batch) as op:
        op.enable_kernel_timing(True)  # (launch counts per kernel; timing runs every wave on one lane)
        frames, grids = op.process_batch_occupancy(clouds, ws, sw, counts)  # (fresh handle: the first call speculates)
        launches = {k: n for k, (_, n) in op.kernel_times().items()}
    waves = -(-B // max_batch)
    counted = sum(n for k, n in launches.items() if k.startswith("k_occ_count_wave"))
    assert counted >= waves, launches
    if kind == "voxel":  # the declined wave ran again from its upload on, counts included
        assert counted > waves, launches
    else:  # the back half ran again without new counts
        assert launches["k_occ_threshold_wave"] > counted, launches
        assert ("k_ece_route" if kind == "cluster" else "k_plane_loop_large") in launches, launches
    with ObstacleProcessor(p, clouds.shape[1], max_batch=max_batch) as op:
        plain = op.process_batch(clouds, counts)
    check_batch(p, clouds, counts, ws, sw, frames, grids, plain, kind)
    for f in range(B):
        compare_frames(frames[f], O.process(p, clouds[f, :counts[f]]), p, f"{kind} frame {f}: ")


def _skipped_fan_scene():
    """a params.yaml frame with a member at sensor x = 1e-6 below a sensor shifted 2 m along y: its shadow line runs
    to the 2^20-cell cap of the cell search and the fan is skipped (PCOP_WARN_SHADOW_DEGENERATE)"""
    rng = np.random.default_rng(0)
    blob = np.stack([rng.uniform(0.02, 0.1, 60), rng.uniform(1.0, 1.08, 60), rng.uniform(0.12, 0.2, 60),
                     np.ones(60)], 1).astype(np.float32)
    blob[0, :3] = [1e-6, 1.04, 0.2]  # alone in its voxel, so it survives the voxel stage unchanged
    sw = np.eye(4, dtype=np.float32)
    sw[1, 3] = 2.0
    ws = np.eye(4, dtype=np.float32)
    ws[1, 3] = -2.0
    return np.concatenate([synth.frame(1, 3), blob]).astype(np.float32), ws, sw


def test_device_results_and_a_skipped_fan_in_one_frame():
    """outputs | OUT_DEVICE: the downloaded arrays equal pcop_process_batch's; the frame whose fan is skipped is the
    only one with the warning bit"""
    p = synth.params(1)
    p.outputs = abi.OUT_ALL
    p.grid_opacity = 40
    pd = p.copy()
    pd.outputs = abi.OUT_ALL | abi.OUT_DEVICE
    n = synth.points_per_frame(1)
    B, bad = 6, 3
    scene, s_ws, s_sw = _skipped_fan_scene()
    clouds = np.zeros((B, len(scene), 4), np.float32)
    clouds[:, :n] = synth.frames(1, 70, B)
    clouds[bad] = scene
    counts = np.full(B, n, np.int32)
    counts[bad] = len(scene)
    ws, sw = poses(p, B, 4)
    ws[bad], sw[bad] = s_ws, s_sw
    with ObstacleProcessor(p, len(scene), max_batch=4) as op:
        plain = op.process_batch(clouds, counts)
    with ObstacleProcessor(pd, len(scene), max_batch=4) as op:
        W, H = op.occupancy_dims()
        grids = np.zeros((B, H, W), np.int8)
        res = op.process_batch_occupancy_raw(clouds.ctypes.data, clouds.shape[1], counts, ws, sw, grids.ctypes.data)
        frames = [_download_frame(op, r) for r in res]
    oracle = check_batch(p, clouds, counts, ws, sw, frames, grids, plain, "device results")
    assert [w for _, w in oracle] == [abi.WARN_SHADOW_DEGENERATE if f == bad else 0 for f in range(B)]
    assert [fr.warnings & abi.WARN_SHADOW_DEGENERATE for fr in frames] == [w for _, w in oracle]


def _download_frame(op, r):
    """a Frame of an OUT_DEVICE result: counts and plane record from r, arrays downloaded from its device pointers"""
    c = abi.FrameResult()
    C.memmove(C.byref(c), C.byref(r), C.sizeof(abi.FrameResult))
    arrays = dict(crop_kept_idx=(r.n_crop, np.int32, None), voxel_keys=(r.n_voxel, np.uint32, None),
                  voxel_centroids=(r.n_voxel, np.float32, 4), sor_kept_idx=(r.n_sor, np.int32, None),
                  plane_inlier_idx=(r.n_plane_inliers, np.int32, None), remaining_cloud=(r.n_remaining, np.float32, 4),
                  remaining_src_idx=(r.n_remaining, np.int32, None), cluster_offsets=(r.n_clusters + 1, np.int32, None),
                  cluster_indices=(r.n_cluster_points, np.int32, None), obstacles=(r.n_clusters, np.float32, 4))
    for name in arrays:
        setattr(c, name, None)
    fr = Frame.from_c(c)
    for name, (count, dtype, cols) in arrays.items():
        a = op.download(getattr(r, name), count * (cols or 1), dtype)
        setattr(fr, name, a.reshape(count, cols) if cols else a)
    return fr


def test_position_independence():
    """200 frames drawn from 12 sources in a pseudo-random order (three lanes, uneven waves): every grid equals its
    source frame's grid, itself checked against the oracle"""
    p = synth.params(2)
    p.block_size = 0.25
    p.grid_opacity = 40
    n = synth.points_per_frame(2)
    D, B = 12, 200
    src = synth.frames(2, 5000, D)
    ws, sw = poses(p, D, 5)
    with ObstacleProcessor(p, n, max_batch=D) as op:
        plain = op.process_batch(src)
        small, small_grids = op.process_batch_occupancy(src, ws, sw)
    check_batch(p, src, np.full(D, n, np.int32), ws, sw, small, small_grids, plain, "source")
    order = np.random.default_rng(78).integers(0, D, B)
    with ObstacleProcessor(p, n, max_batch=B) as op:
        for rep in range(2):  # the second call reuses every lane's buffers
            frames, grids = op.process_batch_occupancy(np.ascontiguousarray(src[order]), ws[order], sw[order])
            bad = [f for f in range(B) if not np.array_equal(grids[f], small_grids[order[f]]) or
                   frames[f].warnings != small[order[f]].warnings or frames[f].n_clusters != small[order[f]].n_clusters]
            assert not bad, f"call {rep}: {len(bad)} of {B} frames differ from their source frame, first {bad[:5]}"


def test_accumulated_cloud_and_no_allocation_after_the_first_call():
    """xyzw = NULL takes the accumulated cloud and empties the accumulator; repeated calls of one shape allocate
    nothing on the device"""
    torch = pytest.importorskip("torch")
    p = synth.params(1)
    p.outputs = abi.OUT_ALL
    p.grid_opacity = 30
    n = synth.points_per_frame(1)
    cloud = synth.frame(1, 9)
    ws, sw = poses(p, 1, 6)
    clouds = synth.frames(1, 90, 24)
    ws24, sw24 = poses(p, 24, 7)
    with ObstacleProcessor(p, n, max_batch=24) as op:
        fr, grid = op.process_batch_occupancy(cloud[None], ws, sw)
        op.accumulate(cloud[:n // 3])
        op.accumulate(cloud[n // 3:])
        afr, agrid = op.process_batch_occupancy(None, ws, sw)
        assert op.accumulated_count == 0
        assert_same_frame(afr[0], fr[0], 0, "accumulated")
        assert_bits_equal(agrid, grid, "accumulated grid")
        op.process_batch_occupancy(clouds, ws24, sw24)
        torch.cuda.synchronize()
        free0, _ = torch.cuda.mem_get_info()
        for _ in range(3):
            op.process_batch_occupancy(clouds, ws24, sw24)
            op.process_batch_occupancy(clouds[:1], ws24[:1], sw24[:1])
        torch.cuda.synchronize()
        free1, _ = torch.cuda.mem_get_info()
    assert free1 == free0, (free0, free1)
    og, ow = oracle_grids(p, cloud[None], [n], ws, sw)[0]
    assert_bits_equal(grid[0], og, "grid")


def test_bad_arguments_and_oversize_grid_leave_the_handle_usable():
    p = synth.params(1)
    n = synth.points_per_frame(1)
    clouds = synth.frames(1, 40, 2)
    counts = np.full(2, n, np.int32)
    ws, sw = poses(p, 2, 8)
    with ObstacleProcessor(p, n, max_batch=2) as op:
        W, H = op.occupancy_dims()
        grids = np.zeros((2, H, W), np.int8)
        res = (abi.FrameResult * 2)()
        st = op._lib.pcop_process_batch_occupancy(op._h, C.c_void_p(clouds.ctypes.data), n, counts.ctypes.data_as(C.c_void_p),
                                                  2, None, sw.ctypes.data_as(C.c_void_p),
                                                  grids.ctypes.data_as(C.c_void_p), res)
        assert st == abi.ERR_BAD_PARAM
        big = p.copy()
        big.block_size = 0.003  # 1500 x 1260 cells
        op.set_params(big)
        with pytest.raises(PcopError) as e:
            op.process_batch_occupancy(clouds, ws, sw)
        assert e.value.status == abi.ERR_CAPACITY
        op.set_params(p)
        frames, grids = op.process_batch_occupancy(clouds, ws, sw)
        plain = op.process_batch(clouds)
    check_batch(p, clouds, counts, ws, sw, frames, grids, plain, "after errors")
