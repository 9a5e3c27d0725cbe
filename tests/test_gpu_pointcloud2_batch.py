"""pcop_process_batch_pointcloud2: a batch of raw sensor-frame PointCloud2 messages, each with its own pose and layout,
through the batched pipeline (and the grid product).

Every frame is compared bit for bit against pcop_process_batch (or pcop_process_batch_occupancy) on the clouds the
reference chain decodes (oracle fromPCLPointCloud2 -> transformPointCloud); selected frames also against the oracle
pipeline and against the single-frame chain pcop_accumulate_pointcloud2 + pcop_process_accumulated."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from parity_util import assert_bits_equal, compare_frames
from pc2_util import LAYOUTS, decode_batch, pack, sensor_poses, to_sensor
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, PcopError, PointCloud2Message, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi
from pointcloud_obstacle_processing_b200.result import Frame
from test_gpu_occupancy_batch import _download_frame, _frames_needing_repeats, assert_same_frame, oracle_grids

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def two_lanes(monkeypatch):
    """waves of about 8 frames dealt to two lanes (read when the handle is created)"""
    monkeypatch.setenv("PCOP_LANES", "2")
    monkeypatch.setenv("PCOP_WAVE_FRAMES", "8")


def desc(addr, n, layout, is_dense=False):
    """the pcop_pointcloud2_frame of a payload at a raw host or device address"""
    return abi.PointCloud2Frame(addr, n, *LAYOUTS[layout], 1 if is_dense else 0)


def msg(payload, n, layout, is_dense=False):
    return PointCloud2Message(payload, n, *LAYOUTS[layout], is_dense)


def frames_of(res):
    return [Frame.from_c(r) for r in res]


def assert_same_frames(got, want, what):
    assert len(got) == len(want), what
    for f in range(len(want)):
        assert_same_frame(got[f], want[f], 0, f"{what} frame {f}")


def sensor_messages(p, world, layouts, seed):
    """the world frames as sensor-frame payloads, one seeded pose each: (payloads, sensor_to_world, world_to_sensor)"""
    sw, ws = sensor_poses(p, len(world), seed)
    return [pack(to_sensor(world[f], ws[f]), layouts[f], seed + f) for f in range(len(world))], sw, ws


@pytest.mark.gpu
def test_config2_messages_over_waves_and_lanes(two_lanes):
    """64 distinct HDL-64 frames as 32-byte XYZIR messages, each with its own pose, over waves of 8 frames on two lanes;
    payloads in pageable host, pinned host and device memory; then one batch that mixes every layout and host with
    device payloads"""
    torch = pytest.importorskip("torch")
    p = synth.params(2)
    n = synth.points_per_frame(2)
    B = 64
    world = synth.frames(2, 4000, B)
    payloads, sw, _ = sensor_messages(p, world, ["xyzir32"] * B, 100)
    clouds = decode_batch(payloads, [n] * B, ["xyzir32"] * B, sw)
    names = list(LAYOUTS)
    mixed_layouts = [names[f % len(names)] for f in range(B)]
    mixed_payloads, mixed_sw, _ = sensor_messages(p, world, mixed_layouts, 300)
    mixed_clouds = decode_batch(mixed_payloads, [n] * B, mixed_layouts, mixed_sw)
    with ObstacleProcessor(p, n, max_batch=16) as op:
        plain = op.process_batch(clouds)
        plain_bytes = op.last_algorithmic_bytes
        mixed_plain = op.process_batch(mixed_clouds)
        pageable = op.process_batch_pointcloud2([msg(b, n, "xyzir32") for b in payloads], sw)
        alg_bytes = op.last_algorithmic_bytes
        pinned = [torch.from_numpy(b).pin_memory() for b in payloads]
        pinned_frames = frames_of(op.process_batch_pointcloud2_raw([desc(t.data_ptr(), n, "xyzir32") for t in pinned], sw))
        dev = [torch.from_numpy(b).cuda() for b in payloads]
        dev_frames = frames_of(op.process_batch_pointcloud2_raw([desc(t.data_ptr(), n, "xyzir32") for t in dev], sw))
        keep = [torch.from_numpy(b).cuda() if f % 2 else torch.from_numpy(b).pin_memory() for f, b in enumerate(mixed_payloads)]
        mixed = frames_of(op.process_batch_pointcloud2_raw([desc(t.data_ptr(), n, mixed_layouts[f]) for f, t in enumerate(keep)],
                                                           mixed_sw))
        chain = {}
        for f in (0, 37):  # the single-frame chain the call replaces
            op.accumulate_reset()
            op.accumulate_pointcloud2(payloads[f], n, *LAYOUTS["xyzir32"], transform=sw[f], is_dense=False)
            chain[f] = op.process_accumulated()
    assert alg_bytes - plain_bytes == B * n * (32 + 16)  # the decode reads point_step and writes 16 bytes per record
    assert_same_frames(pageable, plain, "pageable")
    assert_same_frames(pinned_frames, plain, "pinned")
    assert_same_frames(dev_frames, plain, "device")
    assert_same_frames(mixed, mixed_plain, "mixed layouts and memory")
    for f in (0, 37):
        assert_same_frame(chain[f], plain[f], 0, f"accumulate chain frame {f}")
        compare_frames(pageable[f], O.process(p, clouds[f]), p, f"frame {f} vs oracle: ")
    compare_frames(mixed[9], O.process(p, mixed_clouds[9]), p, "mixed frame 9 vs oracle: ")
    assert sum(fr.n_clusters for fr in pageable) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["xyz16", "xyzir32", "xyz22", "zxy26"])
def test_each_layout_without_transform_and_with_non_finite_records(layout):
    """transform16 = NULL (world-frame payloads), and posed messages with NaN / Inf records under both is_dense rules;
    a handle with every stage off returns the decoded clouds themselves"""
    p = synth.params(1)
    p.outputs = abi.OUT_ALL
    n = synth.points_per_frame(1)
    B = 6
    world = synth.frames(1, 600, B)
    sw, ws = sensor_poses(p, B, 21)
    sensor = [to_sensor(world[f], ws[f]) for f in range(B)]
    rng = np.random.default_rng(5)
    for f in range(1, B, 2):  # holes of a depth camera
        idx = rng.choice(n, 60, replace=False)
        sensor[f][idx[:20], 0] = np.nan
        sensor[f][idx[20:40], 1] = np.inf
        sensor[f][idx[40:], 2] = -np.inf
    payloads = [pack(s, layout, f) for f, s in enumerate(sensor)]
    dense = [False, False, False, True, False, True]
    msgs = [msg(payloads[f], n, layout, dense[f]) for f in range(B)]
    counts = [n] * B
    as_world = decode_batch(payloads, counts, [layout] * B)
    posed = decode_batch(payloads, counts, [layout] * B, sw, dense)
    raw = p.copy()
    raw.enable_crop = raw.enable_voxel = raw.enable_sor = raw.enable_plane = raw.enable_cluster = 0
    raw.outputs = abi.OUT_REMAINING
    with ObstacleProcessor(p, n, max_batch=4) as op:
        got_none = op.process_batch_pointcloud2(msgs, None)
        got_posed = op.process_batch_pointcloud2(msgs, sw)
        want_none = op.process_batch(as_world)
        want_posed = op.process_batch(posed)
    with ObstacleProcessor(raw, n, max_batch=4) as op:
        dec_none = op.process_batch_pointcloud2(msgs, None)
        dec_posed = op.process_batch_pointcloud2(msgs, sw)
    assert_same_frames(got_none, want_none, f"{layout}, no transform")
    assert_same_frames(got_posed, want_posed, f"{layout}, posed")
    for f in range(B):
        assert_bits_equal(dec_none[f].remaining_cloud, as_world[f], f"{layout} frame {f}: decoded cloud")
        assert_bits_equal(dec_posed[f].remaining_cloud, posed[f], f"{layout} frame {f}: decoded + transformed cloud")
    assert np.isnan(posed[1]).any() and np.isinf(posed[1]).any()
    compare_frames(got_posed[2], O.process(p, posed[2]), p, f"{layout} frame 2 vs oracle: ")


@pytest.mark.gpu
def test_grids_into_numpy_pinned_and_device_memory():
    """grids != NULL: frames and grids equal pcop_process_batch_occupancy on the decoded clouds and the oracle chain;
    outputs | OUT_DEVICE results download to the same arrays"""
    torch = pytest.importorskip("torch")
    p = synth.params(1)
    p.outputs = abi.OUT_ALL
    p.grid_opacity = 40
    pd = p.copy()
    pd.outputs = abi.OUT_ALL | abi.OUT_DEVICE
    n = synth.points_per_frame(1)
    B = 12
    world = synth.frames(1, 800, B)
    layouts = ["xyzrgb32", "xyz22", "zxy26", "xyz16"] * 3
    payloads, sw, ws = sensor_messages(p, world, layouts, 40)
    counts = np.full(B, n, np.int32)
    clouds = decode_batch(payloads, counts, layouts, sw)
    msgs = [msg(payloads[f], n, layouts[f]) for f in range(B)]
    with ObstacleProcessor(p, n, max_batch=4) as op:
        W, H = op.occupancy_dims()
        want, want_grids = op.process_batch_occupancy(clouds, ws, sw)
        got, grids = op.process_batch_pointcloud2(msgs, sw, ws, sw, grids=True)
        pinned = torch.full((B, H, W), 3, dtype=torch.int8).pin_memory()
        descs = [desc(b.ctypes.data, n, layouts[f])
                 for f, b in enumerate(payloads)]
        pinned_frames = frames_of(op.process_batch_pointcloud2_raw(descs, sw, ws, sw, pinned.data_ptr()))
        dev = torch.full((B, H, W), 7, dtype=torch.int8, device="cuda")
        op.process_batch_pointcloud2_raw(descs, sw, ws, sw, dev.data_ptr())
        g_dev = dev.cpu().numpy()
    with ObstacleProcessor(pd, n, max_batch=4) as op:
        dgrids = np.zeros((B, H, W), np.int8)
        dev_res = [_download_frame(op, r) for r in op.process_batch_pointcloud2_raw(descs, sw, ws, sw, dgrids.ctypes.data)]
    assert_same_frames(got, want, "grids: frames")
    assert_same_frames(pinned_frames, want, "pinned grids: frames")
    assert_same_frames(dev_res, want, "OUT_DEVICE: frames")
    oracle = oracle_grids(p, clouds, counts, ws, sw)
    for f in range(B):
        assert_bits_equal(grids[f], want_grids[f], f"frame {f}: grid vs pcop_process_batch_occupancy")
        assert_bits_equal(grids[f], oracle[f][0], f"frame {f}: grid vs oracle")
        assert_bits_equal(pinned.numpy()[f], oracle[f][0], f"frame {f}: pinned grid")
        assert_bits_equal(g_dev[f], oracle[f][0], f"frame {f}: device grid")
        assert_bits_equal(dgrids[f], oracle[f][0], f"frame {f}: OUT_DEVICE grid")
        assert (got[f].warnings & abi.WARN_SHADOW_DEGENERATE) == oracle[f][1]
    assert sum(int((g == 40).sum()) for g, _ in oracle) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["cluster", "voxel", "plane"])
def test_speculation_repeats(kind, monkeypatch):
    """the wave engine repeats a wave when a frame outgrew the path it guessed; the voxel decline repeats the whole
    wave, so the messages are decoded again (more k_pc2_ingest launches than waves), and the results still match"""
    p, clouds, counts, max_batch = _frames_needing_repeats(kind, monkeypatch)
    B = len(counts)
    layout = "xyz22" if kind == "voxel" else "xyzir32"
    payloads = [pack(clouds[f, :counts[f]], layout, 70 + f) for f in range(B)]
    msgs = [msg(payloads[f], int(counts[f]), layout) for f in range(B)]
    with ObstacleProcessor(p, clouds.shape[1], max_batch=max_batch) as op:
        op.enable_kernel_timing(True)  # (launch counts per kernel; timing runs every wave on one lane)
        got = op.process_batch_pointcloud2(msgs, None)  # (fresh handle: the first call speculates)
        launches = {k: v for k, (_, v) in op.kernel_times().items()}
    waves = -(-B // max_batch)
    if kind == "voxel":
        assert launches["k_pc2_ingest"] > waves, launches
    else:
        assert launches["k_pc2_ingest"] == waves, launches
        assert ("k_ece_route" if kind == "cluster" else "k_plane_loop_large") in launches, launches
    decoded = decode_batch(payloads, counts, [layout] * B, cap=clouds.shape[1])
    with ObstacleProcessor(p, clouds.shape[1], max_batch=max_batch) as op:
        want = op.process_batch(decoded, counts)
    assert_same_frames(got, want, kind)
    for f in range(B):
        compare_frames(got[f], O.process(p, decoded[f, :counts[f]]), p, f"{kind} frame {f}: ")


@pytest.mark.gpu
def test_ragged_batch_and_position_independence(monkeypatch):
    """an empty message with NULL data, a 3-point one and one at max_points among full ones; then 40 messages drawn
    from 6 sources in a pseudo-random order over three lanes with uneven waves: each equals its source's result"""
    monkeypatch.setenv("PCOP_LANES", "3")
    monkeypatch.setenv("PCOP_WAVE_FRAMES", "6")
    p = synth.params(1)
    p.outputs = abi.OUT_ALL
    n = synth.points_per_frame(1)
    counts = [n - 1777, 0, 3, n, 12345, n]
    B = len(counts)
    world = synth.frames(1, 900, B)
    layouts = ["xyz16", "xyz22", "zxy26", "xyzir32", "xyzrgb32", "xyz22"]
    sw, ws = sensor_poses(p, B, 50)
    payloads = [pack(to_sensor(world[f, :counts[f]], ws[f]), layouts[f], f) for f in range(B)]
    msgs = [PointCloud2Message(None, 0, *LAYOUTS["xyz22"]) if counts[f] == 0 else msg(payloads[f], counts[f], layouts[f])
            for f in range(B)]
    clouds = decode_batch(payloads, counts, layouts, sw, cap=n)
    order = np.random.default_rng(78).integers(0, B, 40)
    with ObstacleProcessor(p, n, max_batch=40) as op:
        want = op.process_batch(clouds, np.array(counts, np.int32))
        got = op.process_batch_pointcloud2(msgs, sw)
        for rep in range(2):  # the second call reuses every lane's buffers
            shuffled = op.process_batch_pointcloud2([msgs[k] for k in order], sw[order])
            bad = [f for f in range(len(order)) if shuffled[f].n_clusters != want[order[f]].n_clusters]
            assert not bad, f"call {rep}: {len(bad)} frames differ from their source, first {bad[:5]}"
            for f in range(len(order)):
                assert_same_frame(shuffled[f], want[order[f]], 0, f"call {rep} position {f} (source {order[f]})")
    assert_same_frames(got, want, "ragged")
    assert [fr.n_input for fr in got] == counts
    compare_frames(got[3], O.process(p, clouds[3]), p, "max_points frame vs oracle: ")


@pytest.mark.gpu
def test_no_allocation_after_the_first_call_and_the_accumulator_is_untouched():
    torch = pytest.importorskip("torch")
    p = synth.params(1)
    p.grid_opacity = 30
    n = synth.points_per_frame(1)
    B = 24
    world = synth.frames(1, 1000, B)
    layouts = ["xyzir32", "xyz22"] * (B // 2)
    payloads, sw, ws = sensor_messages(p, world, layouts, 60)
    pinned = [torch.from_numpy(b).pin_memory() for b in payloads]
    dev = [torch.from_numpy(b).cuda() for b in payloads]
    descs = [desc((dev[f] if f % 3 == 0 else pinned[f]).data_ptr(), n, layouts[f]) for f in range(B)]
    acc = synth.frame(1, 7)
    with ObstacleProcessor(p, n, max_batch=B) as op:
        W, H = op.occupancy_dims()
        grids = torch.empty((B, H, W), dtype=torch.int8, device="cuda")
        op.accumulate(acc[:n // 2])
        op.process_batch_pointcloud2_raw(descs, sw)
        op.process_batch_pointcloud2_raw(descs, sw, ws, sw, grids.data_ptr())
        torch.cuda.synchronize()
        free0, _ = torch.cuda.mem_get_info()
        for _ in range(3):
            op.process_batch_pointcloud2_raw(descs, sw)
            op.process_batch_pointcloud2_raw(descs, sw, ws, sw, grids.data_ptr())
            op.process_batch_pointcloud2_raw(descs[:1], sw[:1])
        torch.cuda.synchronize()
        free1, _ = torch.cuda.mem_get_info()
        assert op.accumulated_count == n // 2
        fr = op.process_accumulated()
        want = op.process(acc[:n // 2])
    assert free1 == free0, (free0, free1)
    assert_same_frame(fr, want, 0, "accumulated cloud after the batched calls")


@pytest.mark.gpu
def test_bad_arguments_leave_the_handle_usable():
    p = synth.params(1)
    n = synth.points_per_frame(1)
    world = synth.frames(1, 40, 2)
    payloads, sw, ws = sensor_messages(p, world, ["xyz16", "xyz22"], 80)
    good = [msg(payloads[0], n, "xyz16"), msg(payloads[1], n, "xyz22")]
    clouds = decode_batch(payloads, [n, n], ["xyz16", "xyz22"], sw)
    big = np.zeros((n + 1) * 16, np.uint8)
    res = (abi.FrameResult * 2)()
    with ObstacleProcessor(p, n, max_batch=2) as op:
        want = op.process_batch(clouds)
        W, H = op.occupancy_dims()
        grids = np.zeros((2, H, W), np.int8)
        cases = [
            ("n_points > max_points", [msg(big, n + 1, "xyz16"), good[1]], {}, abi.ERR_CAPACITY),
            ("offset beyond point_step", [good[0], PointCloud2Message(payloads[1], n, 22, 0, 4, 19)], {}, abi.ERR_BAD_PARAM),
            ("point_step < 4", [PointCloud2Message(payloads[0], n, 3, 0, 0, 0), good[1]], {}, abi.ERR_BAD_PARAM),
            ("negative offset", [PointCloud2Message(payloads[0], n, 16, -4, 4, 8), good[1]], {}, abi.ERR_BAD_PARAM),
            ("negative count", [PointCloud2Message(payloads[0], -1, 16, 0, 4, 8), good[1]], {}, abi.ERR_BAD_PARAM),
            ("grids without matrices", good, dict(grids=True), abi.ERR_BAD_PARAM),
        ]
        for what, msgs, kw, status in cases:
            with pytest.raises(PcopError) as e:
                op.process_batch_pointcloud2(msgs, sw, **kw)
            assert e.value.status == status, what
            assert_same_frames(op.process_batch_pointcloud2(good, sw), want, f"after {what}")
        L, h = op._lib, op._h
        st = L.pcop_process_batch_pointcloud2(h, None, 2, None, None, None, None, res)
        assert st == abi.ERR_BAD_PARAM
        st = L.pcop_process_batch_pointcloud2(h, None, 0, None, None, None, None, res)
        assert st == abi.OK
        assert op.process_batch_pointcloud2([], sw[:0]) == []
        frames, g = op.process_batch_pointcloud2(good, sw, ws, sw, grids=True)
        assert_same_frames(frames, want, "after the error paths")
        _, want_grids = op.process_batch_occupancy(clouds, ws, sw)
        assert_bits_equal(g, want_grids, "grids after the error paths")


def test_pointcloud2_frame_layout_matches_header(tmp_path):
    """CPU: the ctypes mirror of pcop_pointcloud2_frame has the header's size and offsets"""
    src = tmp_path / "sz.c"
    fields = ("data", "n_points", "point_step", "off_x", "off_y", "off_z", "is_dense")
    src.write_text('#include "pcop.h"\n#include <stdio.h>\n#include <stddef.h>\nint main(void){printf("%zu'
                   + " %zu" * len(fields) + '\\n",sizeof(pcop_pointcloud2_frame)'
                   + "".join(f",offsetof(pcop_pointcloud2_frame,{k})" for k in fields) + ");return 0;}\n")
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(abi.PointCloud2Frame)] + [getattr(abi.PointCloud2Frame, k).offset for k in fields]
