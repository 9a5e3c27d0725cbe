"""pcop_process_batch_depth_windows, pcop_accumulate_depth_image and pcop_depth_image_to_xyz: the cloud of a depth
camera built on the GPU from its 16UC1 / 32FC1 images.

The decode equals the depth_image_proc restatement (depth_util.oracle_to_xyz) bit for bit.  Every frame of the
windows call equals, byte for byte, pcop_process_batch_pointcloud2_windows on the point_step-32 XYZRGB messages
depth_image_proc publishes for the same images (depth_util.to_pointcloud2), with the same poses and is_dense = 0, and
the single-frame chain pcop_accumulate_reset + pcop_accumulate_depth_image per image + pcop_process_accumulated."""
import ctypes as C

import numpy as np
import pytest

import depth_util as D
import oracle_lib as O
from parity_util import assert_bits_equal, compare_frames
from pc2_util import LAYOUTS
from shadow_util import rigid
from pointcloud_obstacle_processing_b200 import DepthImage, ObstacleProcessor, PcopError, PointCloud2Message, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi
from pointcloud_obstacle_processing_b200.result import Frame
from test_gpu_occupancy_batch import assert_same_frame

S = 640 * 480  # pixels of a config-3 image


@pytest.fixture
def two_lanes(monkeypatch):
    """waves of about 8 frames dealt to two lanes (read when the handle is created)"""
    monkeypatch.setenv("PCOP_LANES", "2")
    monkeypatch.setenv("PCOP_WAVE_FRAMES", "8")


def frames_of(res):
    return [Frame.from_c(r) for r in res]


def assert_same_frames(got, want, what):
    assert len(got) == len(want), what
    for f in range(len(want)):
        assert_same_frame(got[f], want[f], 0, f"{what} frame {f}")


def camera_poses(M, seed):
    """world <- camera poses close to the camera frame (config 3's crop box keeps most of the scene)"""
    rng = np.random.default_rng(seed)
    return np.stack([rigid(rng.uniform(-0.3, 0.3), rng.uniform(-0.1, 0.1), rng.uniform(-0.1, 0.1),
                           rng.uniform(-0.4, 0.4, 3))[0] for _ in range(M)]).astype(np.float32)


def raw(im):
    """the image's payload bytes (uint8, step * height), or None for an image of 0 pixels"""
    return np.ascontiguousarray(D.raw_bytes(im)) if im.width * im.height else None


def cdesc(im, addr):
    return abi.DepthImageC(addr, im.width, im.height, im.step, D.encoding(im), im.fx, im.fy, im.cx, im.cy)


def download_frame(op, r):
    """a Frame of an OUT_DEVICE result: counts and plane record from r, the arrays of the enabled stages downloaded"""
    c = abi.FrameResult()
    C.memmove(C.byref(c), C.byref(r), C.sizeof(abi.FrameResult))
    arrays = dict(crop_kept_idx=(r.n_crop, np.int32, None), voxel_keys=(r.n_voxel, np.uint32, None),
                  voxel_centroids=(r.n_voxel, np.float32, 4), sor_kept_idx=(r.n_sor, np.int32, None),
                  plane_inlier_idx=(r.n_plane_inliers, np.int32, None), remaining_cloud=(r.n_remaining, np.float32, 4),
                  remaining_src_idx=(r.n_remaining, np.int32, None), cluster_offsets=(r.n_clusters + 1, np.int32, None),
                  cluster_indices=(r.n_cluster_points, np.int32, None), obstacles=(r.n_clusters, np.float32, 4))
    present = [name for name in arrays if getattr(r, name)]  # (a disabled stage returns no array)
    for name in present:
        setattr(c, name, None)
    fr = Frame.from_c(c)
    for name in present:
        count, dtype, cols = arrays[name]
        a = op.download(getattr(r, name), count * (cols or 1), dtype)
        setattr(fr, name, a.reshape(count, cols) if cols else a)
    return fr


class Images:
    """a depth-image stream: images, one pose each, windows, and the equivalent XYZRGB PointCloud2 messages"""

    def __init__(self, images, transforms, window_first):
        self.images = [DepthImage(*im) for im in images]
        self.transforms = transforms
        self.first = np.asarray(window_first, np.int32)
        self.n = [im.width * im.height for im in self.images]

    @property
    def B(self):
        return len(self.first) - 1

    def window(self, f):
        return range(self.first[f], self.first[f + 1])

    def messages(self):
        return [PointCloud2Message(D.to_pointcloud2(im, m) if self.n[m] else None, self.n[m], *LAYOUTS["xyzrgb32"])
                for m, im in enumerate(self.images)]

    def descs(self, bufs):
        """descriptors of the same images whose payloads sit in bufs (torch uint8 tensors or None, one per image)"""
        return [cdesc(im, bufs[m].data_ptr() if self.n[m] else None) for m, im in enumerate(self.images)]

    def tensors(self, torch, device):
        out = []
        for im in self.images:
            r = raw(im)
            t = None if r is None else torch.from_numpy(r)
            out.append(None if t is None else (t.cuda() if device else t.pin_memory()))
        return out

    def concat(self, f):
        """the world-frame concatenation of window f, decoded by the oracle and transformed the reference way"""
        parts = [O.transform(D.oracle_to_xyz(self.images[m]), self.transforms[m], is_dense=False)
                 for m in self.window(f) if self.n[m]]
        return np.concatenate(parts) if parts else np.zeros((0, 4), np.float32)

    def chain(self, op, f):
        op.accumulate_reset()
        for m in self.window(f):
            op.accumulate_depth_image(self.images[m], transform=self.transforms[m])
        return op.process_accumulated()


def mixed_stream(B, seed, max_imgs=4):
    """B windows of 0..max_imgs images: config-3 scenes as 16UC1 and 32FC1 (window 0: one 16UC1 scene, window 2: one
    32FC1 scene), random images of odd width, padded rows and an unaligned base, empty images, a window of empty
    images only"""
    rng = np.random.default_rng(seed)
    empty = [DepthImage(None, 0, 7, 0, abi.DEPTH_16UC1, 500.0, 500.0, 1.0, 1.0),
             DepthImage(None, 5, 0, 20, "32FC1", 500.0, 510.0, 2.5, 0.5)]
    images, first, scene = [], [0], 0

    def pick():
        nonlocal scene
        k = int(rng.integers(0, 6))
        if k <= 1:
            scene += 1
            return D.scene_image(seed + scene, float32=k == 1)
        if k == 2:
            return empty[int(rng.integers(0, 2))]
        W, H = int(rng.integers(1, 200)), int(rng.integers(1, 120))
        return D.random_image(rng, W, H, u16=bool(rng.integers(0, 2)), pad=int(rng.integers(0, 4)),
                              offset=int(rng.integers(0, 3)) * 2)

    for f in range(B):
        if f == 0:
            win = [D.scene_image(seed)]
        elif f == 2:
            win = [D.scene_image(seed + 100, float32=True)]
        elif f % 6 == 1:
            win = []
        elif f % 6 == 3:
            win = list(empty)
        else:
            win = [pick() for _ in range(int(rng.integers(1, max_imgs + 1)))]
        images += win
        first.append(len(images))
    return Images(images, camera_poses(len(images), seed + 1), first)


@pytest.mark.gpu
@pytest.mark.parametrize("camera,float32", [(D.CONFIG3, False), (D.CONFIG3, True), (D.QHD, False)])
def test_depth_image_to_xyz_equals_the_oracle(camera, float32):
    """scene images (aligned path) and random images with an odd width, padded rows or a base 2 bytes off (scalar
    path), from pageable, pinned and device memory"""
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(5)
    u16 = not float32
    images = [D.scene_image(3, camera, float32=float32),
              D.random_image(rng, 64, 48, u16=u16),
              D.random_image(rng, 37, 11, u16=u16),
              D.random_image(rng, 64, 9, u16=u16, pad=3),
              D.random_image(rng, 64, 9, u16=u16, offset=2),
              D.random_image(rng, 33, 7, u16=u16, pad=5, offset=2)]
    with ObstacleProcessor(synth.params(3), camera[0] * camera[1]) as op:
        for k, im in enumerate(images):
            want = D.oracle_to_xyz(im)
            assert_bits_equal(op.depth_image_to_xyz(im), want, f"image {k}: pageable")
            r = raw(im)
            for kind, t in (("pinned", torch.from_numpy(r).pin_memory()), ("device", torch.from_numpy(r).cuda())):
                for shift in (0, 2):  # (a copy whose first pixel is 2 bytes into the buffer)
                    if shift:
                        t2 = torch.zeros(r.size + 2, dtype=torch.uint8, device=t.device)
                        t2[2:] = t
                        if kind == "pinned":
                            t2 = t2.pin_memory()
                        addr = t2.data_ptr() + 2
                    else:
                        addr = t.data_ptr()
                    out = np.empty((im.width * im.height, 4), np.float32)
                    op._check(op._lib.pcop_depth_image_to_xyz(op._h, C.byref(cdesc(im, addr)),
                                                              out.ctypes.data_as(C.c_void_p)))
                    assert_bits_equal(out, want, f"image {k}: {kind} + {shift}")


@pytest.mark.gpu
def test_windows_equal_the_pointcloud2_call_over_waves_and_lanes(two_lanes):
    """windows of 0-4 images, 16UC1 and 32FC1 mixed, empty images and windows, over three waves on two lanes; images
    in pageable host, pinned host and device memory and mixed; the single-frame chain; two frames against the oracle
    pipeline on the oracle-decoded concatenation"""
    torch = pytest.importorskip("torch")
    p = synth.params(3)
    p.outputs = abi.OUT_ALL
    s = mixed_stream(18, 300)
    cap = max(4 * S, max(sum(s.n[m] for m in s.window(f)) for f in range(s.B)))
    pinned, dev = s.tensors(torch, False), s.tensors(torch, True)
    keep = [raw(im) for im in s.images]  # (the pageable payloads of `mixed` must outlive the call)
    dd, dp = s.descs(dev), s.descs(pinned)
    mixed = [(dd, dp)[m % 3 - 1][m] if m % 3 else cdesc(s.images[m], None if keep[m] is None else keep[m].ctypes.data)
             for m in range(len(s.images))]
    with ObstacleProcessor(p, cap, max_batch=16) as op:
        want = op.process_batch_pointcloud2_windows(s.messages(), s.first, s.transforms)
        got = op.process_batch_depth_windows(s.images, s.first, s.transforms)
        got_pinned = frames_of(op.process_batch_depth_windows_raw(s.descs(pinned), s.first, s.transforms))
        got_dev = frames_of(op.process_batch_depth_windows_raw(s.descs(dev), s.first, s.transforms))
        got_mixed = frames_of(op.process_batch_depth_windows_raw(mixed, s.first, s.transforms))
        chain = {f: s.chain(op, f) for f in (0, 1, 2, 3, 4, 5)}
    assert [fr.n_input for fr in got] == [sum(s.n[m] for m in s.window(f)) for f in range(s.B)]
    assert {D.encoding(im) for im in s.images if im.width * im.height} == {abi.DEPTH_16UC1, abi.DEPTH_32FC1}
    assert max(s.first[f + 1] - s.first[f] for f in range(s.B)) >= 3
    for what, g in (("pageable", got), ("pinned", got_pinned), ("device", got_dev), ("mixed", got_mixed)):
        assert_same_frames(g, want, what)
    for f, fr in chain.items():
        assert_same_frame(fr, got[f], 0, f"frame {f} vs the accumulate chain")
    for f in (0, 2):
        compare_frames(got[f], O.process(p, s.concat(f)), p, f"frame {f} vs oracle: ")
    assert sum(fr.n_clusters for fr in got) > 0


@pytest.mark.gpu
def test_grids_and_device_results(two_lanes):
    """grids in host and device memory equal the PointCloud2 call's; the node chain that ends in
    pcop_process_batch_occupancy(NULL); outputs | OUT_DEVICE results equal the PointCloud2 call's"""
    torch = pytest.importorskip("torch")
    p = synth.params(3)
    p.outputs = abi.OUT_ALL
    p.grid_opacity = 40
    s = mixed_stream(10, 800, max_imgs=3)
    cap = max(3 * S, max(sum(s.n[m] for m in s.window(f)) for f in range(s.B)))
    sw = camera_poses(s.B, 801)
    ws = np.stack([np.linalg.inv(m.astype(np.float64)).astype(np.float32) for m in sw])
    msgs = s.messages()
    with ObstacleProcessor(p, cap, max_batch=16) as op:
        W, H = op.occupancy_dims()
        want, want_grids = op.process_batch_pointcloud2_windows(msgs, s.first, s.transforms, ws, sw, grids=True)
        got, grids = op.process_batch_depth_windows(s.images, s.first, s.transforms, ws, sw, grids=True)
        g_dev = torch.full((s.B, H, W), 7, dtype=torch.int8, device="cuda")
        got_dev = frames_of(op.process_batch_depth_windows_raw(s.descs(s.tensors(torch, True)), s.first, s.transforms,
                                                               ws, sw, g_dev.data_ptr()))
        g_dev = g_dev.cpu().numpy()
        f = 0
        op.accumulate_reset()
        for m in s.window(f):
            op.accumulate_depth_image(s.images[m], s.transforms[m])
        node, node_grid = op.process_batch_occupancy(None, ws[f:f + 1], sw[f:f + 1])
    pd = p.copy()
    pd.outputs = abi.OUT_ALL | abi.OUT_DEVICE
    with ObstacleProcessor(pd, cap, max_batch=16) as op:
        dev_res = [download_frame(op, r) for r in op.process_batch_depth_windows_raw(
            s.descs(s.tensors(torch, False)), s.first, s.transforms)]
    with ObstacleProcessor(p, cap, max_batch=16) as op:
        plain = op.process_batch_pointcloud2_windows(msgs, s.first, s.transforms)
    assert_same_frames(got, want, "grids: frames")
    assert_same_frames(got_dev, want, "device grids: frames")
    for k in range(s.B):
        assert_bits_equal(grids[k], want_grids[k], f"frame {k}: grid")
        assert_bits_equal(g_dev[k], want_grids[k], f"frame {k}: device grid")
    assert_same_frame(node[0], got[f], 0, "frame 0 vs the accumulate chain with grids")
    assert_bits_equal(node_grid[0], grids[f], "frame 0: grid vs the accumulate chain")
    assert int((grids == 40).sum()) > 0
    assert_same_frames(dev_res, plain, "OUT_DEVICE")


@pytest.mark.gpu
def test_qhd_windows_of_two_and_a_voxel_decline_repeat():
    """960 x 540 images two per window (the decode of the qhd camera); then a wave whose fused voxel path declines a
    frame, decoded again from the staging"""
    p = synth.params(3)
    p.outputs = abi.OUT_ALL
    qhd = [D.scene_image(20 + k, D.QHD) for k in range(6)]
    s = Images(qhd, camera_poses(6, 21), [0, 2, 4, 6])
    with ObstacleProcessor(p, 2 * 960 * 540, max_batch=4) as op:
        want = op.process_batch_pointcloud2_windows(s.messages(), s.first, s.transforms)
        got = op.process_batch_depth_windows(s.images, s.first, s.transforms)
        chain = s.chain(op, 1)
    assert [fr.n_input for fr in got] == [2 * 960 * 540] * 3
    assert_same_frames(got, want, "qhd windows of 2")
    assert_same_frame(chain, got[1], 0, "qhd: chain frame 1")

    # config 1 (params.yaml): the fused voxel path starts on the partition kernels.  An image of one depth through a
    # lens of fx = 10^7 puts every pixel into one voxel (a bucket above the partition path's limit), so the wave
    # repeats on the LSD path and decodes its images again from the staging.
    p1 = synth.params(1)
    p1.outputs = abi.OUT_ALL
    spot = DepthImage.from_array(np.full((480, 640), 1000, np.uint16), 1.0e7, 1.0e7, 319.5, 239.5)
    z_up = np.array([[0, 0, 1, 0], [-1, 0, 0, 1.0], [0, -1, 0, 0.1], [0, 0, 0, 1]], np.float32)  # world <- camera
    s = Images([D.scene_image(30), spot], np.stack([z_up, z_up]), [0, 1, 2])
    with ObstacleProcessor(p1, S, max_batch=4) as op:
        want = op.process_batch_pointcloud2_windows(s.messages(), s.first, s.transforms)
    with ObstacleProcessor(p1, S, max_batch=4) as op:
        op.enable_kernel_timing(True)
        got = op.process_batch_depth_windows(s.images, s.first, s.transforms)
        launches = {k: v for k, (_, v) in op.kernel_times().items()}
    assert got[1].n_crop == S and got[1].n_voxel == 1, (got[1].n_crop, got[1].n_voxel)
    assert any(k.startswith("k_vp_") for k in launches) and any(k.startswith("k_vf_") for k in launches), launches
    assert launches["k_depth_ingest"] == 2, launches  # (one wave, decoded twice)
    assert_same_frames(got, want, "declined wave")


@pytest.mark.gpu
def test_algorithmic_bytes_and_launches():
    p = synth.params(3)
    ims = [D.scene_image(40), D.scene_image(41, float32=True), D.random_image(np.random.default_rng(2), 33, 7, pad=1)]
    s = Images(ims, camera_poses(3, 42), [0, 3])
    cap = sum(s.n)
    with ObstacleProcessor(p, cap, max_batch=1) as op:  # (fresh handles: both calls take the same route)
        op.process_batch(s.concat(0)[None], np.array([cap], np.int32))
        plain_bytes, plain_launches = op.last_algorithmic_bytes, op.last_launch_count
    with ObstacleProcessor(p, cap, max_batch=1) as op:
        op.process_batch_depth_windows(s.images, s.first, s.transforms)
        got_bytes, got_launches = op.last_algorithmic_bytes, op.last_launch_count
        assert op.stage_times_us()["h2d"] > 0
    assert got_bytes - plain_bytes == 18 * S + 20 * S + 18 * 33 * 7
    assert got_launches == plain_launches + 1


@pytest.mark.gpu
def test_errors_leave_the_handle_usable():
    """every BAD_PARAM and CAPACITY condition of the three calls, each followed by a valid call on the same handle"""
    p = synth.params(3)
    p.outputs = abi.OUT_ALL
    good = D.scene_image(50)
    s = Images([good, D.random_image(np.random.default_rng(3), 21, 5, u16=False, pad=1)], camera_poses(2, 51),
               [0, 2])
    px = np.zeros((4, 6), np.uint16)
    bad = [good._replace(width=-1), good._replace(height=-2), good._replace(data=None), good._replace(encoding=3),
           good._replace(step=1279), good._replace(step=1281), good._replace(encoding=abi.DEPTH_32FC1),
           good._replace(fx=0.0), good._replace(fy=float("nan")), good._replace(fx=float("inf")),
           good._replace(cx=float("inf")), good._replace(cy=float("nan")),
           DepthImage.from_array(px.astype(np.float32), 1, 1, 1, 1)._replace(step=26)]
    with ObstacleProcessor(p, S + 200, max_batch=4) as op:
        want = op.process_batch_depth_windows(s.images, s.first, s.transforms)
        xyz = op.depth_image_to_xyz(good)

        def valid(what):
            assert_same_frames(op.process_batch_depth_windows(s.images, s.first, s.transforms), want, what)
            assert_bits_equal(op.depth_image_to_xyz(good), xyz, what)

        for k, b in enumerate(bad):
            for call in (lambda: op.process_batch_depth_windows([s.images[1], b], [0, 2], s.transforms),
                         lambda: op.accumulate_depth_image(b),
                         lambda: op.depth_image_to_xyz(b)):
                with pytest.raises(PcopError) as e:
                    call()
                assert e.value.status == abi.ERR_BAD_PARAM, (k, b[1:])
            assert op.accumulated_count == 0
            valid(f"after bad image {k}")
        for first in ([1, 2], [0, 2, 1], [0, 3], [0, 1]):  # window_first checks
            with pytest.raises(PcopError) as e:
                op.process_batch_depth_windows(s.images, first, s.transforms)
            assert e.value.status == abi.ERR_BAD_PARAM, first
            valid(f"after window_first {first}")
        with pytest.raises(PcopError) as e:  # a grid without its matrices
            op.process_batch_depth_windows_raw([], [0], None, None, None, 1)
        assert e.value.status == abi.ERR_BAD_PARAM
        with pytest.raises(ValueError):
            op.process_batch_depth_windows(s.images, s.first, s.transforms[:1])
        valid("after the matrix checks")
        # the check order: window_first, then each window's images, then its capacity
        with pytest.raises(PcopError) as e:
            op.process_batch_depth_windows([good, bad[3]], [0, 3], None)
        assert e.value.status == abi.ERR_BAD_PARAM and "window_first" in str(e.value)
        with pytest.raises(PcopError) as e:
            op.process_batch_depth_windows([good, bad[3]], [0, 2], None)
        assert e.value.status == abi.ERR_BAD_PARAM and "image 1" in str(e.value)
        with pytest.raises(PcopError) as e:
            op.process_batch_depth_windows([good, good], [0, 2], None)
        assert e.value.status == abi.ERR_CAPACITY and "window 0" in str(e.value)
        valid("after a window over max_points")
        big = DepthImage.from_array(np.ones((481, 641), np.uint16), 500, 500, 320, 240)
        for call in (lambda: op.accumulate_depth_image(big), lambda: op.depth_image_to_xyz(big)):
            with pytest.raises(PcopError) as e:
                call()
            assert e.value.status == abi.ERR_CAPACITY
        op.accumulate_depth_image(good)
        with pytest.raises(PcopError) as e:
            op.accumulate_depth_image(good)
        assert e.value.status == abi.ERR_CAPACITY and op.accumulated_count == S
        assert op.accumulate_depth_image(s.images[1], s.transforms[1]) == S + 21 * 5
        op.accumulate_reset()
        valid("after the capacity errors")
        q = p.copy()
        q.block_size = 0.01  # (a 2000 x 2000 grid: above PCOP_OCC_BATCH_MAX_CELLS)
        op.set_params(q)
        eye = np.eye(4, dtype=np.float32)[None]
        with pytest.raises(PcopError) as e:
            op.process_batch_depth_windows([good], [0, 1], None, eye, eye, grids=True)
        assert e.value.status == abi.ERR_CAPACITY
        op.set_params(p)
        valid("after the grid capacity error")
        assert op.process_batch_depth_windows([], [0]) == []
        assert op.depth_image_to_xyz(DepthImage(None, 0, 3, 0, "16UC1", 1, 1, 0, 0)).shape == (0, 4)
        assert op.accumulate_depth_image(DepthImage(None, 4, 0, 8, "mono16", 1, 1, 0, 0)) == 0
        chain = s.chain(op, 0)
    assert_same_frame(chain, want[0], 0, "chain after the errors")
