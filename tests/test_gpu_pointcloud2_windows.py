"""pcop_process_batch_pointcloud2_windows: frames built from several posed sensor-frame messages each (the node's
accumulate_count windows, or a multi-sensor rig), through the batched pipeline and the grid product.

Every frame is compared byte for byte against pcop_process_batch (or pcop_process_batch_occupancy) on the concatenations
the reference chain decodes (oracle fromPCLPointCloud2 -> transformPointCloud, message after message), and against the
single-frame chain pcop_accumulate_reset + pcop_accumulate_pointcloud2 per message + pcop_process_accumulated."""

import numpy as np
import pytest

import oracle_lib as O
from parity_util import assert_bits_equal, compare_frames
from pc2_util import LAYOUTS, decode, pack, sensor_poses, to_sensor
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, PcopError, PointCloud2Message, node_windows, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi
from pointcloud_obstacle_processing_b200.result import Frame
from test_gpu_occupancy_batch import assert_same_frame


@pytest.fixture
def two_lanes(monkeypatch):
    """waves of about 8 frames dealt to two lanes (read when the handle is created)"""
    monkeypatch.setenv("PCOP_LANES", "2")
    monkeypatch.setenv("PCOP_WAVE_FRAMES", "8")


def desc(addr, n, layout, is_dense=False):
    return abi.PointCloud2Frame(addr, n, *LAYOUTS[layout], 1 if is_dense else 0)


def frames_of(res):
    return [Frame.from_c(r) for r in res]


def assert_same_frames(got, want, what):
    assert len(got) == len(want), what
    for f in range(len(want)):
        assert_same_frame(got[f], want[f], 0, f"{what} frame {f}")


class Stream:
    """a message stream: payloads (numpy uint8), counts, layouts, is_dense flags, one pose per message, and windows"""

    def __init__(self, payloads, counts, layouts, dense, transforms, window_first):
        self.payloads, self.counts, self.layouts, self.dense = payloads, list(counts), list(layouts), list(dense)
        self.transforms = transforms
        self.first = np.asarray(window_first, np.int32)

    @property
    def B(self):
        return len(self.first) - 1

    def window(self, f):
        return range(self.first[f], self.first[f + 1])

    def messages(self):
        return [PointCloud2Message(self.payloads[m] if self.counts[m] else None, self.counts[m], *LAYOUTS[self.layouts[m]],
                                   self.dense[m]) for m in range(len(self.counts))]

    def descs(self, bufs):
        """descriptors of the same messages whose payloads sit in bufs (torch tensors, one per message)"""
        return [desc(bufs[m].data_ptr() if self.counts[m] else None, self.counts[m], self.layouts[m], self.dense[m])
                for m in range(len(self.counts))]

    def concat(self, f):
        """the world-frame concatenation of window f, the reference way"""
        parts = [decode(self.payloads[m], self.counts[m], self.layouts[m],
                        None if self.transforms is None else self.transforms[m], self.dense[m]) for m in self.window(f)]
        return np.concatenate(parts) if parts else np.zeros((0, 4), np.float32)

    def concats(self, cap):
        """[B, cap, 4] concatenations and their counts, for pcop_process_batch"""
        out = np.zeros((self.B, cap, 4), np.float32)
        counts = np.zeros(self.B, np.int32)
        for f in range(self.B):
            c = self.concat(f)
            out[f, :len(c)] = c
            counts[f] = len(c)
        return out, counts

    def chain(self, op, f):
        """the single-frame chain of window f: reset, one accumulate_pointcloud2 per message, then the pipeline"""
        op.accumulate_reset()
        for m in self.window(f):
            if self.counts[m]:
                op.accumulate_pointcloud2(self.payloads[m], self.counts[m], *LAYOUTS[self.layouts[m]],
                                          transform=None if self.transforms is None else self.transforms[m],
                                          is_dense=self.dense[m])
        return op.process_accumulated()


def config1_stream(p, B, seed, max_msgs=5):
    """B windows of 0..max_msgs messages cut from config-1 world frames, each message in its own sensor pose and a
    layout of LAYOUTS; some empty messages, NaN / Inf records in some messages under both is_dense rules"""
    n = synth.points_per_frame(1)
    world = synth.frames(1, seed, B)
    rng = np.random.default_rng(seed)
    names = list(LAYOUTS)
    payloads, counts, layouts, dense, first = [], [], [], [], [0]
    for f in range(B):
        k = 0 if f % 7 == 3 else (2 if f % 7 == 5 else int(rng.integers(1, max_msgs + 1)))
        cuts = np.sort(rng.integers(0, n + 1, max(k - 1, 0)))
        end = n - int(rng.integers(0, 2000)) if f % 2 else n
        cuts = np.minimum(cuts, end)
        bounds = np.concatenate([[0], cuts, [end if k else 0]]).astype(int)
        if f % 7 == 5:
            bounds[:] = 0  # a window of empty messages only
        for j in range(k):
            counts.append(int(bounds[j + 1] - bounds[j]))
            layouts.append(names[len(layouts) % len(names)])
            dense.append(bool(rng.random() < 0.3))
            payloads.append(world[f, bounds[j]:bounds[j + 1]])
        first.append(len(counts))
    sw, ws = sensor_poses(p, len(counts), seed + 1)
    for m in range(len(counts)):
        s = to_sensor(payloads[m], ws[m])
        if counts[m] > 100 and m % 3 == 1:  # holes of a depth camera
            idx = rng.choice(counts[m], 30, replace=False)
            s[idx[:10], 0] = np.nan
            s[idx[10:20], 1] = np.inf
            s[idx[20:], 2] = -np.inf
        payloads[m] = pack(s, layouts[m], seed + m)
    return Stream(payloads, counts, layouts, dense, sw, first)


@pytest.mark.gpu
def test_config1_windows_over_waves_and_lanes(two_lanes):
    """params.yaml (SOR on): windows of 0-5 messages with mixed layouts, one pose per message, NaN / Inf records, over
    three waves on two lanes; payloads in pageable host, pinned host and device memory, and all three in one call"""
    torch = pytest.importorskip("torch")
    p = synth.params(1)
    p.outputs = abi.OUT_ALL
    n = synth.points_per_frame(1)
    s = config1_stream(p, 24, 500)
    assert any(s.first[f] == s.first[f + 1] for f in range(s.B))  # an empty window
    assert any(s.first[f] < s.first[f + 1] and all(s.counts[m] == 0 for m in s.window(f)) for f in range(s.B))
    clouds, counts = s.concats(n)
    pinned = [torch.from_numpy(b).pin_memory() for b in s.payloads]
    dev = [torch.from_numpy(b).cuda() for b in s.payloads]
    mixed = [(dev, pinned)[m % 3 - 1][m] if m % 3 else s.payloads[m] for m in range(len(s.counts))]
    mixed_descs = [desc(b.data_ptr() if hasattr(b, "data_ptr") else b.ctypes.data, s.counts[m], s.layouts[m], s.dense[m])
                   for m, b in enumerate(mixed)]
    with ObstacleProcessor(p, n, max_batch=16) as op:
        want = op.process_batch(clouds, counts)
        pageable = op.process_batch_pointcloud2_windows(s.messages(), s.first, s.transforms)
        got_pinned = frames_of(op.process_batch_pointcloud2_windows_raw(s.descs(pinned), s.first, s.transforms))
        got_dev = frames_of(op.process_batch_pointcloud2_windows_raw(s.descs(dev), s.first, s.transforms))
        got_mixed = frames_of(op.process_batch_pointcloud2_windows_raw(mixed_descs, s.first, s.transforms))
        chain = [s.chain(op, f) for f in range(s.B)]
    assert [fr.n_input for fr in pageable] == list(counts)
    for what, got in (("pageable", pageable), ("pinned", got_pinned), ("device", got_dev), ("mixed", got_mixed),
                      ("accumulate chain", chain)):
        assert_same_frames(got, want, what)
    full = [f for f in range(s.B) if counts[f] == n]  # (config-1 frames carry depth holes: NaN records)
    assert len(full) >= 2
    for f in full[:2]:
        compare_frames(pageable[f], O.process(p, clouds[f, :counts[f]]), p, f"frame {f} vs oracle: ")
    assert sum(fr.n_clusters for fr in pageable) > 0


@pytest.mark.gpu
def test_grids_into_host_and_device_memory_and_the_node_chain(two_lanes):
    """grids != NULL: frames and grids equal pcop_process_batch_occupancy on the concatenations with the same pose
    pairs, in host and device memory; one frame also equals the chain that ends in pcop_process_batch_occupancy(NULL)"""
    torch = pytest.importorskip("torch")
    p = synth.params(1)
    p.outputs = abi.OUT_ALL
    p.grid_opacity = 40
    n = synth.points_per_frame(1)
    s = config1_stream(p, 12, 700, max_msgs=4)
    clouds, counts = s.concats(n)
    sw, ws = sensor_poses(p, s.B, 701)
    with ObstacleProcessor(p, n, max_batch=16) as op:
        W, H = op.occupancy_dims()
        want, want_grids = op.process_batch_occupancy(clouds, ws, sw, counts)
        got, grids = op.process_batch_pointcloud2_windows(s.messages(), s.first, s.transforms, ws, sw, grids=True)
        dev = torch.full((s.B, H, W), 7, dtype=torch.int8, device="cuda")
        got_dev = frames_of(op.process_batch_pointcloud2_windows_raw(s.descs([torch.from_numpy(b).cuda() for b in s.payloads]),
                                                                     s.first, s.transforms, ws, sw, dev.data_ptr()))
        g_dev = dev.cpu().numpy()
        f = int(np.argmax(counts))
        op.accumulate_reset()
        for m in s.window(f):
            if s.counts[m]:
                op.accumulate_pointcloud2(s.payloads[m], s.counts[m], *LAYOUTS[s.layouts[m]], transform=s.transforms[m],
                                          is_dense=s.dense[m])
        node, node_grid = op.process_batch_occupancy(None, ws[f:f + 1], sw[f:f + 1])
    assert_same_frames(got, want, "grids: frames")
    assert_same_frames(got_dev, want, "device grids: frames")
    for k in range(s.B):
        assert_bits_equal(grids[k], want_grids[k], f"frame {k}: grid")
        assert_bits_equal(g_dev[k], want_grids[k], f"frame {k}: device grid")
    assert_same_frame(node[0], got[f], 0, f"frame {f} vs the accumulate chain with grids")
    assert_bits_equal(node_grid[0], grids[f], f"frame {f}: grid vs the accumulate chain")
    assert int((grids == 40).sum()) > 0


@pytest.mark.gpu
def test_large_windows_take_the_repeat_paths():
    """config-2 HDL-64 messages, 2-5 per window (240 000 - 600 000 points), one pose each: max_points above the partition voxel path's
    limit (LSD path), plane-stage inputs above 8 slices of the large tier (windowed plane kernel), and a crop survivor
    with a NaN y in one message (the fused voxel path declines its frame: the wave is decoded again from the staging)"""
    p = synth.params(2)
    p.downsample_size = 0.04
    p.outputs = abi.OUT_ALL
    n1 = synth.points_per_frame(2)
    sizes = [2, 5, 3, 4, 2, 3]
    M = sum(sizes)
    world = synth.frames(2, 40, M)
    sw, ws = sensor_poses(p, M, 41)
    sensor = [to_sensor(world[m], ws[m]) for m in range(M)]
    # message 3 (window 1): a record with a NaN y is copied untransformed (is_dense = 0), so its sensor-frame record
    # holds the world coordinates of a crop survivor
    k = O.crop(p, world[3])[1][100]
    sensor[3][k] = world[3][k]
    sensor[3][k, 1] = np.nan
    layouts = ["xyzir32" if m % 2 else "xyz22" for m in range(M)]
    payloads = [pack(sensor[m], layouts[m], m) for m in range(M)]
    s = Stream(payloads, [n1] * M, layouts, [False] * M, sw, np.concatenate([[0], np.cumsum(sizes)]))
    cap = 5 * n1
    clouds, counts = s.concats(cap)
    with ObstacleProcessor(p, cap, max_batch=3) as op:
        op.enable_kernel_timing(True)  # (launch counts per kernel; timing runs every wave on one lane)
        got = op.process_batch_pointcloud2_windows(s.messages(), s.first, s.transforms)
        launches = {k: v for k, (_, v) in op.kernel_times().items()}
    with ObstacleProcessor(p, cap, max_batch=3) as op:
        want = op.process_batch(clouds, counts)
    assert np.isnan(clouds[1, n1 + k, 1]) and clouds[1, n1 + k, 0] == world[3, k, 0]
    assert [fr.n_input for fr in got] == [k * n1 for k in sizes]
    assert max(fr.n_sor for fr in got) > 131072, [fr.n_sor for fr in got]  # (8 slices of the large plane tier)
    assert "k_plane_loop_windows" in launches, launches
    assert any(k.startswith("k_vf_") for k in launches) and not any(k.startswith("k_vp_") for k in launches), launches
    assert "k_voxel_keys" in launches, launches                 # the repeat of the declined wave: generic kernels
    assert launches["k_pc2_ingest"] > 2, launches               # ... decoded again from the staging
    assert_same_frames(got, want, "large windows")


@pytest.mark.gpu
def test_one_wave_of_more_than_65535_messages():
    """tiny 1-3-record messages, more than 65 535 of them in one wave (the decode grid is 1-D over record tiles), in
    one device allocation; sampled frames equal the chain, every frame equals pcop_process_batch"""
    torch = pytest.importorskip("torch")
    p = synth.params(1)
    p.outputs = abi.OUT_ALL
    B, per = 4, 17000
    rng = np.random.default_rng(9)
    counts = rng.integers(1, 4, B * per)
    layouts = [("xyz16", "xyz22", "xyzir32")[m % 3] for m in range(B * per)]
    world = synth.frames(1, 900, 2 * B).reshape(B, -1, 4)  # (two config-1 frames per window)
    payloads, off = [], np.zeros(B, int)
    for m in range(B * per):
        f = m // per
        payloads.append(pack(world[f, off[f]:off[f] + counts[m]], layouts[m], 0))
        off[f] += counts[m]
    sizes = [len(b) for b in payloads]
    starts = np.concatenate([[0], np.cumsum([(k + 15) // 16 * 16 for k in sizes])])
    flat = np.zeros(starts[-1], np.uint8)
    for m, b in enumerate(payloads):
        flat[starts[m]:starts[m] + sizes[m]] = b
    dev = torch.from_numpy(flat).cuda()
    descs = [desc(dev.data_ptr() + int(starts[m]), int(counts[m]), layouts[m]) for m in range(B * per)]
    s = Stream(payloads, counts, layouts, [False] * (B * per), None, np.arange(B + 1) * per)
    cap = int(off.max())
    clouds, n = s.concats(cap)
    with ObstacleProcessor(p, cap, max_batch=B) as op:
        got = frames_of(op.process_batch_pointcloud2_windows_raw(descs, s.first))
        want = op.process_batch(clouds, n)
        chain = s.chain(op, 2)
    assert_same_frames(got, want, "tiny messages")
    assert_same_frame(chain, got[2], 0, "tiny messages: chain frame 2")


@pytest.mark.gpu
def test_edges_and_errors_leave_the_handle_usable():
    """a window that fills max_points and one a record over it; malformed window_first; the accumulator is untouched;
    a second call of the same shape allocates nothing"""
    torch = pytest.importorskip("torch")
    p = synth.params(1)
    p.outputs = abi.OUT_ALL
    n = synth.points_per_frame(1)
    world = synth.frames(1, 60, 2)
    sw, ws = sensor_poses(p, 4, 61)
    cuts = [0, 7000, 19000, n]
    payloads = [pack(to_sensor(world[0, cuts[j]:cuts[j + 1]], ws[j]), "xyz22", j) for j in range(3)]
    payloads.append(pack(to_sensor(world[1, :1], ws[3]), "xyz16", 3))
    counts = [cuts[1], cuts[2] - cuts[1], n - cuts[2], 1]
    full = Stream(payloads[:3], counts[:3], ["xyz22"] * 3, [False] * 3, sw[:3], [0, 0, 3, 3])  # empty, full, empty
    over = Stream(payloads, counts, ["xyz22"] * 3 + ["xyz16"], [False] * 4, sw, [0, 4])
    acc = synth.frame(1, 7)[:5000]
    with ObstacleProcessor(p, n, max_batch=4) as op:
        op.accumulate(acc)
        got = op.process_batch_pointcloud2_windows(full.messages(), full.first, full.transforms)
        assert op.accumulated_count == 5000
        with pytest.raises(PcopError) as e:
            op.process_batch_pointcloud2_windows(over.messages(), over.first, over.transforms)
        assert e.value.status == abi.ERR_CAPACITY and "window 0" in str(e.value)
        msgs = full.messages()
        for bad in ([1, 2, 3], [0, 2, 1, 3], [0, 5, 3], [0, 1, 2], [0, 3, 4]):
            with pytest.raises(PcopError) as e:
                op.process_batch_pointcloud2_windows(msgs, bad, full.transforms)
            assert e.value.status == abi.ERR_BAD_PARAM, bad
        arr = (abi.PointCloud2Frame * 3)(*full.descs([torch.from_numpy(b) for b in full.payloads]))
        res = (abi.FrameResult * 3)()
        assert op._lib.pcop_process_batch_pointcloud2_windows(op._h, arr, 3, None, 1, None, None, None, None, res) == abi.ERR_BAD_PARAM
        assert op._lib.pcop_process_batch_pointcloud2_windows(op._h, arr, 0, None, 0, None, None, None, None, res) == abi.OK
        assert op.process_batch_pointcloud2_windows([], [0]) == []
        again = op.process_batch_pointcloud2_windows(msgs, full.first, full.transforms)
        torch.cuda.synchronize()
        free0, _ = torch.cuda.mem_get_info()
        for _ in range(3):
            op.process_batch_pointcloud2_windows(msgs, full.first, full.transforms)
        torch.cuda.synchronize()
        free1, _ = torch.cuda.mem_get_info()
        assert op.accumulated_count == 5000
        from_acc = op.process_accumulated()
        want_acc = op.process(acc)
        empty = op.process_accumulated()
        chain = full.chain(op, 1)
        want = op.process_batch(full.concats(n)[0], full.concats(n)[1])
    assert free1 == free0, (free0, free1)
    assert [fr.n_input for fr in got] == [0, n, 0]
    assert_same_frames(got, want, "full window")
    assert_same_frames(again, want, "after the error paths")
    assert_same_frame(chain, got[1], 0, "full window vs chain")
    for f in (0, 2):
        assert_same_frame(got[f], empty, 0, f"empty window {f} vs an empty accumulator")
    assert_same_frame(from_acc, want_acc, 0, "accumulated cloud after the windows calls")


@pytest.mark.gpu
def test_algorithmic_bytes_count_every_message_of_a_mixed_window():
    p = synth.params(1)
    n = synth.points_per_frame(1)
    world = synth.frame(1, 80)
    sw, ws = sensor_poses(p, 3, 81)
    cuts, layouts = [0, 9000, 21000, n], ["xyz16", "xyz22", "xyzir32"]
    payloads = [pack(to_sensor(world[cuts[j]:cuts[j + 1]], ws[j]), layouts[j], j) for j in range(3)]
    s = Stream(payloads, np.diff(cuts), layouts, [False] * 3, sw, [0, 3])
    with ObstacleProcessor(p, n, max_batch=1) as op:
        op.process_batch(*s.concats(n))
        plain = op.last_algorithmic_bytes
        op.process_batch_pointcloud2_windows(s.messages(), s.first, s.transforms)
        got = op.last_algorithmic_bytes
    assert got - plain == sum((LAYOUTS[layouts[j]][0] + 16) * (cuts[j + 1] - cuts[j]) for j in range(3))


def test_node_windows():
    """CPU: od.cpp:690-701 -- K messages accumulated, the next one triggers the run and is not added"""
    first, kept, trig = node_windows(11, 2)
    assert first.tolist() == [0, 2, 4, 6] and kept.tolist() == [0, 1, 3, 4, 6, 7] and trig.tolist() == [2, 5, 8]
    first, kept, trig = node_windows(5, 0)
    assert first.tolist() == [0] * 6 and kept.tolist() == [] and trig.tolist() == [0, 1, 2, 3, 4]
    first, kept, trig = node_windows(7, 1)
    assert first.tolist() == [0, 1, 2, 3] and kept.tolist() == [0, 2, 4] and trig.tolist() == [1, 3, 5]
    first, kept, trig = node_windows(450, 200)
    assert first.tolist() == [0, 200, 400] and trig.tolist() == [200, 401]
    assert kept.tolist() == list(range(200)) + list(range(201, 401))
    assert [len(a) for a in node_windows(0, 200)] == [1, 0, 0]
    assert [len(a) for a in node_windows(200, 200)] == [1, 0, 0]  # (no trigger yet: nothing is processed)
    with pytest.raises(ValueError):
        node_windows(3, -1)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [0, 2, 3])
def test_node_replay_equals_the_windows_call(K):
    """a literal replay of od.cpp:690-701 on the single-frame chain (grids with the TFs looked up while the trigger
    message is handled) equals one windows call built with node_windows; the stream ends in a partial window"""
    p = synth.params(1)
    p.grid_opacity = 20
    n = synth.points_per_frame(1)
    N = 4 * (K + 1) + max(K - 1, 0)
    world = synth.frames(1, 120, N)
    rng = np.random.default_rng(K)
    counts = rng.integers(1000, n // max(K, 1) + 1, N)
    sw, ws = sensor_poses(p, N, 121)
    layouts = [("xyzrgb32", "xyz16", "zxy26")[m % 3] for m in range(N)]
    payloads = [pack(to_sensor(world[m, :counts[m]], ws[m]), layouts[m], m) for m in range(N)]
    with ObstacleProcessor(p, n, max_batch=8) as op:
        replay, replay_grids = [], []
        current_frame_count = 0
        for m in range(N):  # cloud_cb
            if current_frame_count < K:
                op.accumulate_pointcloud2(payloads[m], int(counts[m]), *LAYOUTS[layouts[m]], transform=sw[m])
                current_frame_count += 1
            else:
                fr, g = op.process_batch_occupancy(None, ws[m:m + 1], sw[m:m + 1])
                replay.append(fr[0])
                replay_grids.append(g[0])
                current_frame_count = 0
        op.accumulate_reset()
        first, kept, trig = node_windows(N, K)
        msgs = [PointCloud2Message(payloads[m], int(counts[m]), *LAYOUTS[layouts[m]]) for m in kept]
        got, grids = op.process_batch_pointcloud2_windows(msgs, first, sw[kept].reshape(-1, 4, 4), ws[trig], sw[trig],
                                                          grids=True)
    assert len(got) == len(replay) == 4
    assert_same_frames(got, replay, f"K = {K}")
    for f in range(len(got)):
        assert_bits_equal(grids[f], replay_grids[f], f"K = {K} frame {f}: grid")
