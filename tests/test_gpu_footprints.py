"""GPU: obstacle footprints (PCOP_OUT_FOOTPRINTS).

The stage-isolated pcop_cluster_footprints equals both restatements of footprint_util on every CPU case, on a
multi-piece blob and on a cluster whose extreme members exceed one shared-memory tile.  Every pcop_process* entry point
with the bit returns, beside byte-identical results, the footprints both restatements compute from its remaining cloud
and clusters.  Also: non-finite singletons, result lifetime, launch counts, buffers given back, and every error."""
import ctypes as C

import numpy as np
import pytest

import depth_util as D
import footprint_util as F
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, PcopError, PointCloud2Message, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi

pytestmark = pytest.mark.gpu

ARRAYS = ["crop_kept_idx", "voxel_keys", "voxel_centroids", "sor_kept_idx", "plane_inlier_idx", "remaining_cloud",
          "remaining_src_idx", "cluster_offsets", "cluster_indices", "obstacles"]
COUNTS = ["status", "warnings", "n_input", "n_crop", "n_voxel", "n_sor", "n_remaining", "n_clusters",
          "n_cluster_points", "n_plane_passes", "n_plane_inliers"]
PY_MAX = 20000  # largest cluster the Python restatement checks (the C++ one checks every cluster)


@pytest.fixture
def two_lanes(monkeypatch):
    monkeypatch.setenv("PCOP_LANES", "2")
    monkeypatch.setenv("PCOP_WAVE_FRAMES", "8")


def assert_same(a, b, what):
    for k, (x, y) in enumerate(zip(a, b)):
        x, y = np.ascontiguousarray(x), np.ascontiguousarray(y)
        assert x.shape == y.shape, f"{what}: array {k} shape {x.shape} vs {y.shape}"
        assert x.tobytes() == y.tobytes(), f"{what}: array {k} differs"


def check_against_restatements(got, cloud, off, idx, what):
    assert_same(got, F.oracle_footprints(cloud, off, idx), what + " (C++)")
    if len(off) < 2 or np.diff(off).max() <= PY_MAX:
        assert_same(got, F.numpy_footprints(cloud, off, idx), what + " (Python)")


def check_frame(fr, what):
    assert fr.boxes is not None and fr.hull_offsets is not None and fr.hull_indices is not None, what
    check_against_restatements((fr.boxes, fr.hull_offsets, fr.hull_indices), fr.remaining_cloud, fr.cluster_offsets,
                               fr.cluster_indices, what)


def assert_same_frames(got, want, what):
    assert len(got) == len(want), what
    for f, (g, w) in enumerate(zip(got, want)):
        for k in COUNTS:
            assert getattr(g, k) == getattr(w, k), f"{what} frame {f}: {k}"
        for k in ARRAYS:
            a, b = getattr(g, k), getattr(w, k)
            assert (a is None) == (b is None), f"{what} frame {f}: {k}"
            if a is not None:
                assert a.tobytes() == b.tobytes(), f"{what} frame {f}: {k} differs"
        assert np.array_equal(g.plane_pass_coeff, w.plane_pass_coeff) and np.array_equal(g.plane_coeff, w.plane_coeff)


def with_outputs(p, outputs):
    q = p.copy()
    q.outputs = outputs
    return q


def test_cluster_footprints_equal_both_restatements():
    rng = np.random.default_rng(5)
    big = {
        "blob_200k": F.concat([F.blob(rng, 200000, 2.0)], rng),  # multi-piece, small union of piece hulls
        "polygon_100k": F.concat([F.convex_polygon(205, 0.5)], rng),  # every member extreme: beyond one tile
        "circle_120k": F.concat([F.circle(120000, 50.0, 0.5, 3.0, -2.0)], rng),
        "two_big": F.concat([F.circle(9000, 2.0), F.blob(rng, 30000, 1.0), F.circle(4097, 1.0, 0.0, 9.0, 9.0)], rng),
        # two consecutive multi-piece clusters, every member extreme, members in random order: the union of the piece
        # hulls is the whole cluster, beyond one tile, and the second point in (x, y) order is on the lower chain
        "two_all_extreme_multi_piece": F.concat([F.sheared_polygon(45), F.sheared_polygon(44, 1.0, 3.0e6),
                                                 F.blob(rng, 100, 1.0)], rng, mix=True),
    }
    with ObstacleProcessor(synth.params(1), 250000) as op:
        for name, (cloud, off, idx) in list(F.cases().items()) + list(big.items()):
            got = op.cluster_footprints(cloud, off, idx)
            check_against_restatements(got, cloud, off, idx, name)
        cloud, off, idx = big["polygon_100k"]
        boxes, hoff, hidx = op.cluster_footprints(cloud, off, idx)
        assert len(hidx) == len(cloud) > 100000  # the large-candidate path ran
        cloud, off, idx = big["two_all_extreme_multi_piece"]
        boxes, hoff, hidx = op.cluster_footprints(cloud, off, idx)
        sizes = np.diff(off)
        assert sizes[0] > 4096 and sizes[1] > 4096 and (np.diff(hoff)[:2] == sizes[:2]).all()
        cloud, off, idx = F.cases()["all_extreme_4096_second_on_lower_chain"]
        assert len(op.cluster_footprints(cloud, off, idx)[2]) == 4096  # one piece, filled, every member a vertex


@pytest.mark.parametrize("config,frames", [(1, 12), (2, 12), (3, 10), (4, 2)])
def test_batch_results_unchanged_and_footprints_exact(two_lanes, config, frames):
    p = with_outputs(synth.params(config), abi.OUT_ALL)
    clouds = synth.frames(config, 40, frames)
    with ObstacleProcessor(p, synth.points_per_frame(config), max_batch=16) as op:
        plain = op.process_batch(clouds)
        assert all(fr.boxes is None and fr.hulls is None for fr in plain)
        op.set_params(with_outputs(p, abi.OUT_ALL | abi.OUT_FOOTPRINTS))
        got = op.process_batch(clouds)
        again = op.process_batch(clouds)
    assert_same_frames(got, plain, f"config {config}")
    assert sum(fr.n_clusters for fr in got) > 0
    for f, fr in enumerate(got):
        check_frame(fr, f"config {config} frame {f}")
        assert_same((fr.boxes, fr.hull_offsets, fr.hull_indices),
                    (again[f].boxes, again[f].hull_offsets, again[f].hull_indices), "second call")


def test_every_entry_point(two_lanes):
    p = with_outputs(synth.params(1), abi.OUT_ALL)
    pf = with_outputs(p, abi.OUT_ALL | abi.OUT_FOOTPRINTS)
    n = synth.points_per_frame(1)
    B = 12
    clouds = synth.frames(1, 7, B)
    eye = np.tile(np.eye(4, dtype=np.float32), (B, 1, 1))
    msgs = [PointCloud2Message(np.ascontiguousarray(c).view(np.uint8), len(c), 16, 0, 4, 8, True) for c in clouds]
    first = np.arange(B + 1, dtype=np.int32)
    with ObstacleProcessor(p, n, max_batch=16) as op:
        def both(call):
            op.set_params(p)
            a = call()
            op.set_params(pf)
            b = call()
            return a, b

        a, b = both(lambda: [op.process(clouds[0])])
        assert_same_frames(b, a, "process")
        check_frame(b[0], "process")

        def acc():
            op.accumulate(clouds[1][: n // 2])
            op.accumulate(clouds[2][: n // 2])
            return [op.process_accumulated()]
        a, b = both(acc)
        assert_same_frames(b, a, "process_accumulated")
        check_frame(b[0], "process_accumulated")

        (fa, ga), (fb, gb) = both(lambda: op.process_batch_occupancy(clouds, eye, eye))
        assert_same_frames(fb, fa, "occupancy")
        assert ga.tobytes() == gb.tobytes()
        for f, fr in enumerate(fb):
            check_frame(fr, f"occupancy frame {f}")

        a, b = both(lambda: op.process_batch_pointcloud2_windows(msgs, first, eye))
        assert_same_frames(b, a, "pointcloud2 windows")
        for f, fr in enumerate(b):
            check_frame(fr, f"pointcloud2 windows frame {f}")

        # OUT_DEVICE: the footprint pointers are device pointers into the call's pack buffer
        op.set_params(with_outputs(p, abi.OUT_ALL | abi.OUT_FOOTPRINTS | abi.OUT_DEVICE))
        res = op.process_batch_raw(clouds.ctypes.data, n, np.full(B, n, np.int32))
        for f in range(B):
            r, fp = res[f], op.last_footprints(f)
            assert fp.n_clusters == r.n_clusters
            cloud = op.download(C.cast(r.remaining_cloud, C.c_void_p).value, r.n_remaining * 4, np.float32).reshape(-1, 4)
            off = op.download(C.cast(r.cluster_offsets, C.c_void_p).value, r.n_clusters + 1, np.int32)
            idx = op.download(C.cast(r.cluster_indices, C.c_void_p).value, r.n_cluster_points, np.int32)
            got = (op.download(C.cast(fp.boxes, C.c_void_p).value, fp.n_clusters * 8, np.float32).reshape(-1, 8),
                   op.download(C.cast(fp.hull_offsets, C.c_void_p).value, fp.n_clusters + 1, np.int32),
                   op.download(C.cast(fp.hull_indices, C.c_void_p).value, fp.n_hull_vertices, np.int32))
            check_against_restatements(got, cloud, off, idx, f"OUT_DEVICE frame {f}")

    p3 = with_outputs(synth.params(3), abi.OUT_ALL)
    images = [D.scene_image(k) for k in range(3)]
    with ObstacleProcessor(p3, 2 * images[0].width * images[0].height, max_batch=4) as op:
        wf = np.array([0, 1, 3], np.int32)
        op.set_params(p3)
        a = op.process_batch_depth_windows(images, wf)
        op.set_params(with_outputs(p3, abi.OUT_ALL | abi.OUT_FOOTPRINTS))
        b = op.process_batch_depth_windows(images, wf)
        assert_same_frames(b, a, "depth windows")
        for f, fr in enumerate(b):
            check_frame(fr, f"depth windows frame {f}")


def test_nonfinite_points_are_singletons():
    p = synth.params(1)
    p.enable_crop = p.enable_voxel = p.enable_sor = p.enable_plane = 0
    p.euc_min_cluster_size = 1
    p.outputs = abi.OUT_DEFAULT | abi.OUT_FOOTPRINTS
    rng = np.random.default_rng(9)
    cloud = F.blob(rng, 3000, 0.3)
    bad = rng.choice(3000, 40, replace=False)
    specials = np.array([np.nan, np.inf, -np.inf, 1.0], np.float32)
    for k, i in enumerate(bad):
        cloud[i, k % 3] = specials[k % 3]
        cloud[i, (k + 1) % 3] = specials[(k // 3) % 4]
    with ObstacleProcessor(p, len(cloud)) as op:
        fr = op.process(cloud)
    check_frame(fr, "non-finite")
    nonfinite = ~np.isfinite(fr.remaining_cloud[:, :3]).all(axis=1)
    assert nonfinite.sum() == 40
    sizes = np.diff(fr.cluster_offsets)
    for k, members in enumerate(fr.clusters):
        if nonfinite[members].any():
            assert sizes[k] == 1 and fr.hulls[k].tolist() == members.tolist()
            assert fr.boxes[k].view(np.uint32)[[0, 1, 2]].tolist() == fr.remaining_cloud[members[0], :3].view(np.uint32).tolist()


def test_results_of_a_call_outlive_the_next_call():
    p = with_outputs(synth.params(2), abi.OUT_DEFAULT | abi.OUT_FOOTPRINTS)
    B = 6
    clouds = synth.frames(2, 3, 2 * B)
    n = synth.points_per_frame(2)
    counts = np.full(B, n, np.int32)

    def read(op, f):
        fp = op.last_footprints(f)
        return fp, (np.ctypeslib.as_array(fp.boxes, (fp.n_clusters * 8,)).copy(),
                    np.ctypeslib.as_array(fp.hull_offsets, (fp.n_clusters + 1,)).copy(),
                    np.ctypeslib.as_array(fp.hull_indices, (max(fp.n_hull_vertices, 1),))[:fp.n_hull_vertices].copy())

    with ObstacleProcessor(p, n, max_batch=B) as op:
        op.process_batch_raw(clouds.ctypes.data, n, counts)
        first = [read(op, f) for f in range(B)]
        op.process_batch_raw(clouds[B:].ctypes.data, n, counts)
        for f, (fp, arrays) in enumerate(first):
            again = (np.ctypeslib.as_array(fp.boxes, (fp.n_clusters * 8,)),
                     np.ctypeslib.as_array(fp.hull_offsets, (fp.n_clusters + 1,)),
                     np.ctypeslib.as_array(fp.hull_indices, (max(fp.n_hull_vertices, 1),))[:fp.n_hull_vertices])
            assert_same(again, arrays, f"call k frame {f} after call k + 1")


def test_launch_counts():
    p = with_outputs(synth.params(2), abi.OUT_DEFAULT)
    clouds = synth.frames(2, 0, 8)
    n = synth.points_per_frame(2)
    with ObstacleProcessor(p, n, max_batch=8) as never:  # (second calls: the first one sets the route history)
        never.process_batch(clouds)
        never.process_batch(clouds)
        base = never.last_launch_count
    with ObstacleProcessor(p, n, max_batch=8) as op:
        op.set_params(with_outputs(p, abi.OUT_DEFAULT | abi.OUT_FOOTPRINTS))
        op.enable_kernel_timing(True)
        op.process_batch(clouds)
        on = op.last_launch_count
        kt = op.kernel_times()
        op.enable_kernel_timing(False)
        op.set_params(p)
        op.process_batch(clouds)
        off = op.last_launch_count
    assert off == base
    fp = {k: v[1] for k, v in kt.items() if k.startswith("k_fp_")}
    waves = kt["k_pack_scan"][1]
    assert fp["k_fp_piece"] == fp["k_fp_csr"] == fp["k_fp_combine"] == waves  # (frames above one tile: all three)
    assert on == off + sum(fp.values())


def toggle_cycle():
    p = with_outputs(synth.params(1), abi.OUT_DEFAULT)
    clouds = synth.frames(1, 0, 4)
    with ObstacleProcessor(p, synth.points_per_frame(1), max_batch=4) as op:
        for outputs in (abi.OUT_DEFAULT, abi.OUT_DEFAULT | abi.OUT_FOOTPRINTS, abi.OUT_DEFAULT,
                        abi.OUT_ALL | abi.OUT_FOOTPRINTS | abi.OUT_DEVICE):
            op.set_params(with_outputs(p, outputs))
            if outputs & abi.OUT_DEVICE:
                op.process_batch_raw(clouds.ctypes.data, clouds.shape[1], np.full(4, clouds.shape[1], np.int32))
            else:
                frames = op.process_batch(clouds)
                assert (frames[0].boxes is None) == (not outputs & abi.OUT_FOOTPRINTS)


def test_toggling_the_bit_gives_back_every_buffer():
    torch = pytest.importorskip("torch")
    toggle_cycle()
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    toggle_cycle()
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    assert free1 == free0, (free0, free1)


def test_errors_leave_the_handle_usable():
    p = with_outputs(synth.params(1), abi.OUT_DEFAULT | abi.OUT_FOOTPRINTS)
    cloud = synth.frame(1, 0)
    n = len(cloud)
    with ObstacleProcessor(p, n) as op:
        L, h = op._lib, op._h
        fr = op.process(cloud)
        off, idx = fr.cluster_offsets, fr.cluster_indices
        rem = np.ascontiguousarray(fr.remaining_cloud)
        want = (fr.boxes, fr.hull_offsets, fr.hull_indices)

        def valid(what):
            assert_same(op.cluster_footprints(rem, off, idx), want, f"after {what}")
            op.process(cloud)
            fp = abi.FrameFootprints()
            assert L.pcop_last_footprints(h, 0, C.byref(fp)) == abi.OK and fp.n_clusters == fr.n_clusters, what

        fp = abi.FrameFootprints()
        for what, frame, out in (("NULL out", 0, None), ("frame -1", -1, C.byref(fp)), ("frame 1", 1, C.byref(fp))):
            assert L.pcop_last_footprints(h, frame, out) == abi.ERR_BAD_PARAM, what
            valid(what)
        assert L.pcop_last_footprints(None, 0, C.byref(fp)) == abi.ERR_BAD_PARAM
        with pytest.raises(PcopError):  # a failed call: no footprints until the next call succeeds
            op.process(np.zeros((n + 1, 4), np.float32))
        assert L.pcop_last_footprints(h, 0, C.byref(fp)) == abi.ERR_BAD_PARAM
        valid("a failed call")
        op.set_params(with_outputs(p, abi.OUT_DEFAULT))  # without the bit: NULL pointers
        op.process(cloud)
        assert L.pcop_last_footprints(h, 0, C.byref(fp)) == abi.OK
        assert not fp.boxes and not fp.hull_offsets and not fp.hull_indices and fp.n_hull_vertices == 0
        op.set_params(p)

        P = len(rem)
        bad_off = [("offsets[0] != 0", off + 1, idx, P), ("decreasing offsets", off[::-1].copy(), idx, P),
                   ("offsets[c] > p", off, idx, int(off[-1]) - 1)]
        hi = idx.copy()
        hi[len(hi) // 2] = P
        lo = idx.copy()
        lo[0] = -1
        bad_off += [("index >= p", off, hi, P), ("index < 0", off, lo, P)]
        vp = C.c_void_p
        out_b, out_o, out_i, nh = np.zeros((len(off), 8), np.float32), np.zeros(len(off) + 1, np.int32), \
            np.zeros(len(idx) + 1, np.int32), C.c_int32()
        ptr = lambda a: a.ctypes.data_as(vp)  # noqa: E731
        for what, o, i, pp in bad_off:
            if what == "offsets[c] > p":
                r = rem[:pp]
            else:
                r = rem
            st = L.pcop_cluster_footprints(h, ptr(r), pp, ptr(np.ascontiguousarray(o, np.int32)),
                                           ptr(np.ascontiguousarray(i, np.int32)), len(o) - 1, ptr(out_b), ptr(out_o),
                                           ptr(out_i), C.byref(nh))
            assert st == abi.ERR_BAD_PARAM, what
            valid(what)
        c = len(off) - 1
        args = [ptr(rem), P, ptr(off), ptr(idx), c, ptr(out_b), ptr(out_o), ptr(out_i), C.byref(nh)]
        for k, what in ((0, "NULL cloud"), (2, "NULL offsets"), (3, "NULL indices"), (5, "NULL boxes"),
                        (6, "NULL hull_offsets"), (7, "NULL hull_indices"), (8, "NULL n_hull")):
            a = list(args)
            a[k] = None
            assert L.pcop_cluster_footprints(h, *a) == abi.ERR_BAD_PARAM, what
            valid(what)
        a = list(args)
        a[4] = -1
        assert L.pcop_cluster_footprints(h, *a) == abi.ERR_BAD_PARAM
        valid("c < 0")
        a = list(args)
        a[1] = n + 1
        assert L.pcop_cluster_footprints(h, *a) == abi.ERR_CAPACITY
        valid("p > max_points")
        big_off = np.zeros(n + 2, np.int32)
        a = list(args)
        a[2], a[4] = ptr(big_off), n + 1
        assert L.pcop_cluster_footprints(h, *a) == abi.ERR_CAPACITY
        valid("c > max_points")
