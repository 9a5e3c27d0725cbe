"""Host-side mirror of the reference's five stage wrappers + frame driver, over the C ABI (include/pcop.h).

Method names follow the reference's free functions (minibot_cr18/src/obstacle_detection.cpp):
  crop                         <- build_initial_occupancy_grid_dataset crop loop   (od.cpp:195-215)
  downsample_cloud             <- downsample_cloud                                 (od.cpp:271-296)
  remove_statistical_outliers  <- remove_statistical_outliers                      (od.cpp:316-340)
  segment_plane_and_extract_indices <- same name                                   (od.cpp:342-428)
  extract_euclidian_clusters   <- same name (sic)                                  (od.cpp:430-455)
  centroid_radius              <- PointWithRad/PointIndicesArray output            (msg/*.msg, od.cpp:806-814)
  process / process_batch      <- cloud_cb's process branch                        (od.cpp:699-927)
  process_batch_occupancy      <- the same + the occupancy grid it publishes        (od.cpp:699-852)

There is no CPU fallback: constructing an ObstacleProcessor without a usable B200-class device raises.
"""
import collections
import ctypes as C
import os

import numpy as np

from . import _ctypes_abi as abi
from ._ctypes_abi import DepthImageC, FrameFootprints, FrameResult, Params, PointCloud2Frame
from .result import Frame


class PointCloud2Message(collections.namedtuple("PointCloud2Message",
                                                "data n_points point_step off_x off_y off_z is_dense",
                                                defaults=(False,))):
    """The fields of a sensor_msgs/PointCloud2 message that the decode reads: data (bytes or uint8 array, host),
    n_points = width * height, point_step and the byte offsets of the FLOAT32 fields x, y, z."""


# sensor_msgs/Image encodings of a depth image -> PCOP_DEPTH_*
DEPTH_ENCODINGS = {"16UC1": abi.DEPTH_16UC1, "mono16": abi.DEPTH_16UC1, "32FC1": abi.DEPTH_32FC1}


class DepthImage(collections.namedtuple("DepthImage", "data width height step encoding fx fy cx cy")):
    """A depth image (sensor_msgs/Image) and the pinhole model of its CameraInfo: data (bytes or numpy array, host),
    width, height, step (bytes per row), encoding (PCOP_DEPTH_* or a key of DEPTH_ENCODINGS), and
    image_geometry::PinholeCameraModel's fx, fy, cx, cy."""

    @classmethod
    def from_array(cls, depth, fx, fy, cx, cy):
        """a [H, W] uint16 (16UC1 millimetres) or float32 (32FC1 metres) array, rows possibly padded (step = the
        array's row stride); its pixels must be contiguous along a row"""
        depth = np.asarray(depth)
        enc = {np.dtype(np.uint16): abi.DEPTH_16UC1, np.dtype(np.float32): abi.DEPTH_32FC1}.get(depth.dtype)
        if enc is None or depth.ndim != 2:
            raise ValueError("depth image must be a [H, W] uint16 or float32 array")
        if depth.shape[1] > 1 and depth.strides[1] != depth.itemsize:
            raise ValueError("the pixels of a row must be contiguous")
        H, W = depth.shape
        step = depth.strides[0] if H > 1 else W * depth.itemsize
        return cls(depth, W, H, int(step), enc, float(fx), float(fy), float(cx), float(cy))


def _depth_descriptors(images):
    """DepthImage sequence -> (host buffers to keep alive, DepthImageC list)"""
    keep, descs = [], []
    for im in images:
        im = DepthImage(*im)
        enc = DEPTH_ENCODINGS[im.encoding] if isinstance(im.encoding, str) else int(im.encoding)
        if im.data is None:
            ptr, buf = None, None
        elif isinstance(im.data, np.ndarray):
            buf = im.data
            if not (buf.flags.c_contiguous or (buf.ndim == 2 and buf.strides[1] == buf.itemsize and buf.strides[0] > 0)):
                buf = np.ascontiguousarray(buf)
            ptr = buf.ctypes.data if buf.size else None
        else:
            buf = np.frombuffer(im.data, np.uint8)
            ptr = buf.ctypes.data if buf.size else None
        keep.append(buf)
        descs.append(DepthImageC(ptr, im.width, im.height, im.step, enc, im.fx, im.fy, im.cx, im.cy))
    return keep, descs


_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpcop.so")
_lib = None

EXPORTS = [
    "pcop_abi_version", "pcop_global_error", "pcop_last_error", "pcop_params_init_code_defaults",
    "pcop_params_init_params_yaml", "pcop_create", "pcop_destroy", "pcop_set_params", "pcop_process",
    "pcop_process_batch", "pcop_last_elapsed_us", "pcop_stage_times_us", "pcop_last_launch_count",
    "pcop_last_algorithmic_bytes", "pcop_crop", "pcop_voxel", "pcop_sor", "pcop_plane", "pcop_cluster",
    "pcop_centroid_radius", "pcop_enable_kernel_timing", "pcop_kernel_timing_count", "pcop_kernel_timing_get",
    "pcop_last_sort_pass_keys",
    "pcop_last_d2h_bytes",
    "pcop_accumulate",
    "pcop_accumulated_count",
    "pcop_process_accumulated",
    "pcop_accumulate_reset",
    "pcop_transform",
    "pcop_accumulate_pointcloud2",
    "pcop_pointcloud2_to_xyz",
    "pcop_cloud_to_pointcloud2",
    "pcop_occupancy_dims",
    "pcop_occupancy_grid",
    "pcop_occupancy_shadows",
    "pcop_download",
    "pcop_process_batch_occupancy",
    "pcop_process_batch_pointcloud2",
    "pcop_process_batch_pointcloud2_windows",
    "pcop_process_batch_depth_windows",
    "pcop_accumulate_depth_image",
    "pcop_depth_image_to_xyz",
    "pcop_last_footprints",
    "pcop_cluster_footprints",
]


class PcopError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"pcop status {status}: {message}")
        self.status = status


def load_library():
    """Load libpcop.so (building it in-tree if missing).  Raises if the CUDA library cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from ._build import build_cuda
        build_cuda()
    L = C.CDLL(LIB_PATH)
    vp, i32, u32 = C.c_void_p, C.c_int32, C.c_uint32
    pi32, pu32 = C.POINTER(C.c_int32), C.POINTER(C.c_uint32)
    L.pcop_abi_version.restype = C.c_int
    L.pcop_global_error.restype = C.c_char_p
    L.pcop_last_error.restype = C.c_char_p
    L.pcop_last_error.argtypes = [vp]
    L.pcop_params_init_code_defaults.argtypes = [C.POINTER(Params)]
    L.pcop_params_init_params_yaml.argtypes = [C.POINTER(Params)]
    L.pcop_create.argtypes = [C.POINTER(Params), C.c_int, C.c_size_t, C.c_int, C.POINTER(vp)]
    L.pcop_destroy.argtypes = [vp]
    L.pcop_set_params.argtypes = [vp, C.POINTER(Params)]
    L.pcop_process.argtypes = [vp, vp, i32, C.POINTER(FrameResult)]
    L.pcop_process_batch.argtypes = [vp, vp, C.c_size_t, vp, i32, C.POINTER(FrameResult)]
    L.pcop_last_elapsed_us.restype = C.c_float
    L.pcop_last_elapsed_us.argtypes = [vp]
    L.pcop_stage_times_us.argtypes = [vp, C.POINTER(C.c_float)]
    L.pcop_last_launch_count.restype = C.c_int64
    L.pcop_last_launch_count.argtypes = [vp]
    L.pcop_last_algorithmic_bytes.restype = C.c_double
    L.pcop_last_algorithmic_bytes.argtypes = [vp]
    L.pcop_last_sort_pass_keys.restype = C.c_int64
    L.pcop_last_sort_pass_keys.argtypes = [vp]
    L.pcop_last_d2h_bytes.restype = C.c_double
    L.pcop_last_d2h_bytes.argtypes = [vp]
    L.pcop_accumulate.argtypes = [vp, vp, C.c_int32, vp, C.c_int32, vp]
    L.pcop_accumulated_count.argtypes = [vp]
    L.pcop_accumulated_count.restype = C.c_int32
    L.pcop_process_accumulated.argtypes = [vp, vp]
    L.pcop_accumulate_reset.argtypes = [vp]
    L.pcop_transform.argtypes = [vp, vp, C.c_int32, vp, C.c_int32, vp]
    L.pcop_accumulate_pointcloud2.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, C.c_int32, vp]
    L.pcop_pointcloud2_to_xyz.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp]
    L.pcop_cloud_to_pointcloud2.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp]
    L.pcop_download.argtypes = [vp, vp, vp, C.c_size_t]
    L.pcop_occupancy_dims.argtypes = [vp, vp, vp]
    L.pcop_occupancy_grid.argtypes = [vp, vp, C.c_int32, vp, vp, vp]
    L.pcop_occupancy_shadows.argtypes = [vp, vp, C.c_int32, vp, vp, C.c_int32, vp, vp, vp, vp, vp]
    L.pcop_process_batch_occupancy.argtypes = [vp, vp, C.c_size_t, vp, i32, vp, vp, vp, C.POINTER(FrameResult)]
    L.pcop_process_batch_pointcloud2.argtypes = [vp, C.POINTER(PointCloud2Frame), i32, vp, vp, vp, vp,
                                                 C.POINTER(FrameResult)]
    L.pcop_process_batch_pointcloud2_windows.argtypes = [vp, C.POINTER(PointCloud2Frame), i32, vp, i32, vp, vp, vp, vp,
                                                         C.POINTER(FrameResult)]
    L.pcop_process_batch_depth_windows.argtypes = [vp, C.POINTER(DepthImageC), i32, vp, i32, vp, vp, vp, vp,
                                                   C.POINTER(FrameResult)]
    L.pcop_accumulate_depth_image.argtypes = [vp, C.POINTER(DepthImageC), vp, vp]
    L.pcop_depth_image_to_xyz.argtypes = [vp, C.POINTER(DepthImageC), vp]
    L.pcop_enable_kernel_timing.argtypes = [vp, C.c_int]
    L.pcop_kernel_timing_count.argtypes = [vp]
    L.pcop_kernel_timing_get.argtypes = [vp, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_double),
                                         C.POINTER(C.c_int64)]
    L.pcop_crop.argtypes = [vp, vp, i32, vp, vp, pi32]
    L.pcop_voxel.argtypes = [vp, vp, i32, vp, vp, pi32, pu32]
    L.pcop_sor.argtypes = [vp, vp, i32, vp, vp, pi32, pu32]
    L.pcop_plane.argtypes = [vp, vp, i32, vp, vp, pi32, pi32, vp, vp, vp, vp, vp, pi32, pu32]
    L.pcop_cluster.argtypes = [vp, vp, i32, vp, vp, pi32, pi32]
    L.pcop_centroid_radius.argtypes = [vp, vp, i32, vp, vp, i32, vp]
    L.pcop_last_footprints.argtypes = [vp, i32, C.POINTER(FrameFootprints)]
    L.pcop_cluster_footprints.argtypes = [vp, vp, i32, vp, vp, i32, vp, vp, vp, pi32]
    _lib = L
    return L


def params_yaml() -> Params:
    """Parameter values of the reference's minibot_cr18/params.yaml."""
    p = Params()
    load_library().pcop_params_init_params_yaml(C.byref(p))
    return p


def params_code_defaults() -> Params:
    """Defaults of the nh.param(...) calls at od.cpp:940-975."""
    p = Params()
    load_library().pcop_params_init_code_defaults(C.byref(p))
    return p


def node_windows(n_messages: int, accumulate_count: int):
    """The processing callbacks of the reference node over a stream of n_messages messages (od.cpp:690-701): with
    K = accumulate_count, messages j(K+1) .. j(K+1)+K-1 are converted, transformed and appended, and message j(K+1)+K
    runs the pipeline on them without being added itself.  A trailing window that never sees its trigger message is not
    processed; K = 0 gives one empty frame per message.
    Returns (window_first int32 [J + 1] over the kept messages, kept int64 [J K]: the stream index of every kept
    message, triggers int64 [J]: the stream index of each window's trigger message, during which the node looks up the
    grid TFs, od.cpp:592, 570, 634) -- window_first and the kept messages are what process_batch_pointcloud2_windows
    takes."""
    n, k = int(n_messages), int(accumulate_count)
    if n < 0 or k < 0:
        raise ValueError("n_messages and accumulate_count must be >= 0")
    J = n // (k + 1)
    starts = np.arange(J, dtype=np.int64) * (k + 1)
    kept = (starts[:, None] + np.arange(k, dtype=np.int64)[None, :]).reshape(-1)
    return np.arange(J + 1, dtype=np.int32) * k, kept, starts + k


def _pc2_descriptors(messages):
    """PointCloud2Message sequence -> (host buffers to keep alive, PointCloud2Frame list)"""
    keep, frames = [], []
    for m in messages:
        m = PointCloud2Message(*m)
        if m.data is None:
            buf = np.zeros(0, np.uint8)
        elif isinstance(m.data, np.ndarray):
            buf = np.ascontiguousarray(m.data.reshape(-1)).view(np.uint8)
        else:
            buf = np.frombuffer(m.data, np.uint8)
        keep.append(buf)
        frames.append(PointCloud2Frame(buf.ctypes.data if buf.size else None, m.n_points, m.point_step, m.off_x,
                                       m.off_y, m.off_z, 1 if m.is_dense else 0))
    return keep, frames


def _mats(m, count, what):
    """[count, 4, 4] float32 matrices (or None) -> (array kept alive, pointer)"""
    if m is None:
        return None, None
    m = np.ascontiguousarray(m, np.float32).reshape(-1, 16)
    if m.shape[0] != count:
        raise ValueError(f"one {what} matrix per {'message' if what == 'transform' else 'frame'} ({count})")
    return m, m.ctypes.data_as(C.c_void_p)


def _f32(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] != 4:
        raise ValueError("cloud must be [n, 4] float32 (pcl::PointXYZ layout)")
    return a


class ObstacleProcessor:
    """One handle = one device = one caller at a time (the reference node is single-threaded, od.cpp:1014)."""

    def __init__(self, params: Params, max_points: int, max_batch: int = 1, device: int = 0):
        self._lib = load_library()
        self._h = C.c_void_p()
        self.params = params.copy()
        self.max_points, self.max_batch, self.device = int(max_points), int(max_batch), int(device)
        st = self._lib.pcop_create(C.byref(self.params), device, max_points, max_batch, C.byref(self._h))
        if st != abi.OK:
            raise PcopError(st, (self._lib.pcop_global_error() or b"").decode())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.pcop_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, st):
        if st != abi.OK:
            raise PcopError(st, (self._lib.pcop_last_error(self._h) or b"").decode())

    def set_params(self, params: Params):
        self._check(self._lib.pcop_set_params(self._h, C.byref(params)))
        self.params = params.copy()

    # ---- whole pipeline ------------------------------------------------------------
    def _host_results_only(self):
        """Frame.from_c copies out of HOST result pointers; with outputs | OUT_DEVICE they are device addresses."""
        if self.params.outputs & abi.OUT_DEVICE:
            raise ValueError("outputs | OUT_DEVICE leaves the result arrays on the GPU: call process_batch_raw() and "
                             "read them with download() / copy_device()")

    def last_footprints(self, frame: int) -> FrameFootprints:
        """pcop_last_footprints: frame `frame` of the last pcop_process* call (device pointers with OUT_DEVICE)"""
        fp = FrameFootprints()
        self._check(self._lib.pcop_last_footprints(self._h, frame, C.byref(fp)))
        return fp

    def _frames(self, res):
        """Frames of the last call's host results, with their footprints"""
        return [Frame.from_c(r).set_footprints(self.last_footprints(f)) for f, r in enumerate(res)]

    def process(self, cloud) -> Frame:
        self._host_results_only()
        cloud = _f32(cloud)
        r = FrameResult()
        self._check(self._lib.pcop_process(self._h, cloud.ctypes.data_as(C.c_void_p), cloud.shape[0], C.byref(r)))
        return self._frames([r])[0]

    def process_batch_raw(self, ptr: int, frame_stride_points: int, counts: np.ndarray):
        """Frames at a raw host or device address; returns the ctypes result array (valid until the next call)."""
        counts = np.ascontiguousarray(counts, dtype=np.int32)
        res = (FrameResult * len(counts))()
        self._check(self._lib.pcop_process_batch(self._h, C.c_void_p(ptr), frame_stride_points,
                                                 counts.ctypes.data_as(C.c_void_p), len(counts), res))
        return res

    def process_batch(self, clouds, counts=None):
        """clouds: float32 [B, n, 4] (host).  Returns a list of Frame."""
        self._host_results_only()
        clouds = np.ascontiguousarray(clouds, dtype=np.float32)
        assert clouds.ndim == 3 and clouds.shape[2] == 4
        if counts is None:
            counts = np.full(clouds.shape[0], clouds.shape[1], np.int32)
        res = self.process_batch_raw(clouds.ctypes.data, clouds.shape[1], counts)
        return self._frames(res)

    # ---- pipeline + occupancy grid (the node's published product) --------------------------
    def occupancy_dims(self):
        """(width, height) of the occupancy grid (od.cpp:958-959)"""
        w, h = C.c_int32(), C.c_int32()
        self._check(self._lib.pcop_occupancy_dims(self._h, C.byref(w), C.byref(h)))
        return w.value, h.value

    def process_batch_occupancy_raw(self, ptr, frame_stride_points: int, counts, world_to_sensor, sensor_to_world,
                                    grids_ptr: int):
        """pcop_process_batch_occupancy on frames at a raw host or device address (ptr = None: the accumulated cloud,
        batch 1), grids written to a raw host or device address ([B, H, W] int8).  world_to_sensor / sensor_to_world:
        [B, 4, 4] float32 (one pose per frame).  Returns the ctypes result array (valid until the next call)."""
        counts = np.ascontiguousarray(np.zeros(1, np.int32) if counts is None else counts, dtype=np.int32)
        B = len(counts)
        ws = np.ascontiguousarray(world_to_sensor, np.float32).reshape(-1, 16)
        sw = np.ascontiguousarray(sensor_to_world, np.float32).reshape(-1, 16)
        if ws.shape[0] != B or sw.shape[0] != B:
            raise ValueError(f"one world_to_sensor and one sensor_to_world matrix per frame ({B})")
        res = (FrameResult * B)()
        self._check(self._lib.pcop_process_batch_occupancy(
            self._h, None if ptr is None else C.c_void_p(ptr), frame_stride_points, counts.ctypes.data_as(C.c_void_p), B,
            ws.ctypes.data_as(C.c_void_p), sw.ctypes.data_as(C.c_void_p), C.c_void_p(grids_ptr), res))
        return res

    def process_batch_occupancy(self, clouds, world_to_sensor, sensor_to_world, counts=None):
        """clouds: float32 [B, n, 4] (host), or None for the accumulated cloud (B = 1; the accumulator is emptied).
        world_to_sensor / sensor_to_world: [B, 4, 4] float32, frame f's TF lookups (od.cpp:592 / 570, 634).
        Returns (list of Frame, grids int8 [B, H, W]): every frame through the pipeline and the occupancy grid the node
        publishes for it (initial data set, shadows, obstacle marks).  The grids land in a pageable numpy array, whose
        copies hold the host once per wave; for throughput pass pinned or device memory to
        process_batch_occupancy_raw."""
        self._host_results_only()
        w, h = self.occupancy_dims()
        if clouds is None:
            ptr, stride, counts = None, 1, np.zeros(1, np.int32)
        else:
            clouds = np.ascontiguousarray(clouds, dtype=np.float32)
            assert clouds.ndim == 3 and clouds.shape[2] == 4
            if counts is None:
                counts = np.full(clouds.shape[0], clouds.shape[1], np.int32)
            ptr, stride = clouds.ctypes.data, clouds.shape[1]
        grids = np.empty((len(counts), h, w), np.int8)
        res = self.process_batch_occupancy_raw(ptr, stride, counts, world_to_sensor, sensor_to_world, grids.ctypes.data)
        return self._frames(res), grids

    # ---- raw PointCloud2 messages, one pose each (od.cpp:688-696 + 699-852 per message) ------------------
    def process_batch_pointcloud2_raw(self, frames, transforms=None, world_to_sensor=None, sensor_to_world=None,
                                      grids_ptr=None):
        """pcop_process_batch_pointcloud2.  frames: a sequence of PointCloud2Frame (data = host or device address).
        transforms / world_to_sensor / sensor_to_world: [B, 4, 4] float32 or None; grids_ptr: raw host or device
        address of [B, H, W] int8, or None (pipeline only).  Returns the ctypes result array (valid until the next
        call)."""
        B = len(frames)
        arr = (PointCloud2Frame * max(B, 1))(*frames)
        (t, tp), (ws, wsp), (sw, swp) = _mats(transforms, B, "transform"), _mats(world_to_sensor, B, "world_to_sensor"), \
            _mats(sensor_to_world, B, "sensor_to_world")
        res = (FrameResult * max(B, 1))()
        self._check(self._lib.pcop_process_batch_pointcloud2(
            self._h, arr, B, tp, wsp, swp, None if grids_ptr is None else C.c_void_p(grids_ptr), res))
        return res[:B] if B else []

    def process_batch_pointcloud2(self, messages, transforms=None, world_to_sensor=None, sensor_to_world=None,
                                  grids=False):
        """messages: a sequence of PointCloud2Message (host payloads).  transforms: [B, 4, 4] float32, message f's
        world <- sensor pose, or None when the payloads are already in the world frame.  Returns the list of Frame, or
        (frames, grids int8 [B, H, W]) with grids=True (then world_to_sensor / sensor_to_world are required, as in
        process_batch_occupancy; a replay of single messages passes its poses as transforms and sensor_to_world).
        Pageable payloads and grids hold the host per copy; for throughput pass pinned or device memory to
        process_batch_pointcloud2_raw."""
        self._host_results_only()
        keep, frames = _pc2_descriptors(messages)
        g = None
        if grids:
            w, h = self.occupancy_dims()
            g = np.empty((len(frames), h, w), np.int8)
        res = self.process_batch_pointcloud2_raw(frames, transforms, world_to_sensor, sensor_to_world,
                                                 None if g is None else g.ctypes.data)
        out = self._frames(res)
        return (out, g) if grids else out

    # ---- accumulation windows: several posed messages per frame (od.cpp:688-701 per processing callback) ----------
    def process_batch_pointcloud2_windows_raw(self, messages, window_first, transforms=None, world_to_sensor=None,
                                              sensor_to_world=None, grids_ptr=None):
        """pcop_process_batch_pointcloud2_windows.  messages: a sequence of PointCloud2Frame (data = host or device
        address); window_first: int [B + 1], frame f = messages window_first[f] .. window_first[f + 1] - 1 concatenated.
        transforms: [n_messages, 4, 4] float32 or None; world_to_sensor / sensor_to_world: [B, 4, 4] float32 or None;
        grids_ptr: raw host or device address of [B, H, W] int8, or None.  Returns the ctypes result array (valid until
        the next call)."""
        M = len(messages)
        first = np.ascontiguousarray(window_first, np.int32).reshape(-1)
        if first.size < 1:
            raise ValueError("window_first needs batch + 1 entries")
        B = first.size - 1
        arr = (PointCloud2Frame * max(M, 1))(*messages)
        (t, tp), (ws, wsp), (sw, swp) = _mats(transforms, M, "transform"), _mats(world_to_sensor, B, "world_to_sensor"), \
            _mats(sensor_to_world, B, "sensor_to_world")
        res = (FrameResult * max(B, 1))()
        self._check(self._lib.pcop_process_batch_pointcloud2_windows(
            self._h, arr, M, first.ctypes.data_as(C.c_void_p), B, tp, wsp, swp,
            None if grids_ptr is None else C.c_void_p(grids_ptr), res))
        return res[:B] if B else []

    def process_batch_pointcloud2_windows(self, messages, window_first, transforms=None, world_to_sensor=None,
                                          sensor_to_world=None, grids=False):
        """messages: a sequence of PointCloud2Message (host payloads), one pose each in transforms ([n_messages, 4, 4]
        float32 world <- sensor, or None).  Frame f is the world-frame concatenation of messages window_first[f] ..
        window_first[f + 1] - 1 -- what the node accumulates before a processing callback (node_windows() builds
        window_first for an accumulate_count), or the messages of several sensors at one time step.  Returns the list
        of Frame, or (frames, grids int8 [B, H, W]) with grids=True (world_to_sensor / sensor_to_world: [B, 4, 4], one
        pair per frame)."""
        self._host_results_only()
        keep, frames = _pc2_descriptors(messages)
        g = None
        if grids:
            w, h = self.occupancy_dims()
            g = np.empty((len(window_first) - 1, h, w), np.int8)
        res = self.process_batch_pointcloud2_windows_raw(frames, window_first, transforms, world_to_sensor,
                                                         sensor_to_world, None if g is None else g.ctypes.data)
        out = self._frames(res)
        return (out, g) if grids else out

    # ---- depth images: the depth camera's cloud built on the device (depth_image_proc + od.cpp:688-701) ----------
    def process_batch_depth_windows_raw(self, images, window_first, transforms=None, world_to_sensor=None,
                                        sensor_to_world=None, grids_ptr=None):
        """pcop_process_batch_depth_windows.  images: a sequence of DepthImageC (data = host or device address); the
        other arguments and the result as process_batch_pointcloud2_windows_raw."""
        M = len(images)
        first = np.ascontiguousarray(window_first, np.int32).reshape(-1)
        if first.size < 1:
            raise ValueError("window_first needs batch + 1 entries")
        B = first.size - 1
        arr = (DepthImageC * max(M, 1))(*images)
        (t, tp), (ws, wsp), (sw, swp) = _mats(transforms, M, "transform"), _mats(world_to_sensor, B, "world_to_sensor"), \
            _mats(sensor_to_world, B, "sensor_to_world")
        res = (FrameResult * max(B, 1))()
        self._check(self._lib.pcop_process_batch_depth_windows(
            self._h, arr, M, first.ctypes.data_as(C.c_void_p), B, tp, wsp, swp,
            None if grids_ptr is None else C.c_void_p(grids_ptr), res))
        return res[:B] if B else []

    def process_batch_depth_windows(self, images, window_first, transforms=None, world_to_sensor=None,
                                    sensor_to_world=None, grids=False):
        """images: a sequence of DepthImage (host payloads), one pose each in transforms ([n_images, 4, 4] float32
        world <- camera, or None).  Frame f is the world-frame concatenation of the clouds of images window_first[f] ..
        window_first[f + 1] - 1, each the cloud depth_image_proc builds from the image.  Returns the list of Frame, or
        (frames, grids int8 [B, H, W]) with grids=True, as process_batch_pointcloud2_windows."""
        self._host_results_only()
        keep, descs = _depth_descriptors(images)
        g = None
        if grids:
            w, h = self.occupancy_dims()
            g = np.empty((len(window_first) - 1, h, w), np.int8)
        res = self.process_batch_depth_windows_raw(descs, window_first, transforms, world_to_sensor, sensor_to_world,
                                                   None if g is None else g.ctypes.data)
        out = self._frames(res)
        return (out, g) if grids else out

    def accumulate_depth_image(self, image, transform=None) -> int:
        """the cloud of one DepthImage (depth_image_proc), world transform (is_dense = false) and append, on the
        device; returns the accumulated point count"""
        keep, (d,) = _depth_descriptors([image])
        t = None if transform is None else np.ascontiguousarray(transform, dtype=np.float32).reshape(16)
        total = C.c_int32()
        self._check(self._lib.pcop_accumulate_depth_image(self._h, C.byref(d),
                                                          None if t is None else t.ctypes.data_as(C.c_void_p),
                                                          C.byref(total)))
        return total.value

    def depth_image_to_xyz(self, image):
        """the stage-isolated decode of one DepthImage (no transform): float32 [width * height, 4]"""
        keep, (d,) = _depth_descriptors([image])
        n = d.width * d.height
        out = np.empty((max(n, 1), 4), np.float32)
        self._check(self._lib.pcop_depth_image_to_xyz(self._h, C.byref(d), out.ctypes.data_as(C.c_void_p)))
        return out[:n].copy()

    # ---- accumulator ingest (od.cpp:691-698) ------------------------------------------
    def accumulate(self, cloud, transform=None, is_dense=False) -> int:
        """pcl_ros::transformPointCloud(cloud, world_T_sensor) + `passthrough_input_cloud +=` (od.cpp:696-697), on
        the device.  transform: 4x4 float (row-major) or None for identity.  Returns the accumulated point count."""
        cloud = _f32(cloud)
        t = None if transform is None else np.ascontiguousarray(transform, dtype=np.float32).reshape(16)
        total = C.c_int32()
        self._check(self._lib.pcop_accumulate(self._h, cloud.ctypes.data_as(C.c_void_p), cloud.shape[0],
                                              None if t is None else t.ctypes.data_as(C.c_void_p),
                                              1 if is_dense else 0, C.byref(total)))
        return total.value

    def accumulate_pointcloud2(self, data, n_points, point_step, off_x, off_y, off_z, transform=None, is_dense=False) -> int:
        """sensor_msgs/PointCloud2 payload (bytes / uint8 array) -> PointXYZ + world transform + append, one kernel
        (od.cpp:688-689 + 696-697)"""
        buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, np.uint8)
        t = None if transform is None else np.ascontiguousarray(transform, dtype=np.float32).reshape(16)
        total = C.c_int32()
        self._check(self._lib.pcop_accumulate_pointcloud2(self._h, buf.ctypes.data_as(C.c_void_p), n_points, point_step,
                                                          off_x, off_y, off_z,
                                                          None if t is None else t.ctypes.data_as(C.c_void_p),
                                                          1 if is_dense else 0, C.byref(total)))
        return total.value

    def pointcloud2_to_xyz(self, data, n_points, point_step, off_x, off_y, off_z):
        buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, np.uint8)
        out = np.empty((max(n_points, 1), 4), np.float32)
        self._check(self._lib.pcop_pointcloud2_to_xyz(self._h, buf.ctypes.data_as(C.c_void_p), n_points, point_step, off_x,
                                                      off_y, off_z, out.ctypes.data_as(C.c_void_p)))
        return out[:n_points].copy()

    def cloud_to_pointcloud2(self, cloud, point_step=16, off_x=0, off_y=4, off_z=8, device_ptr=None, n=None):
        """pcl::toROSMsg of a PointXYZ cloud (od.cpp:290-294): the sensor_msgs/PointCloud2 payload as a uint8 array
        [n * point_step].  `cloud` is a host array [n, 4], or pass device_ptr + n for a device-resident result array."""
        if device_ptr is None:
            cloud = _f32(cloud)
            n = cloud.shape[0]
            src = cloud.ctypes.data_as(C.c_void_p)
        else:
            src = C.c_void_p(int(device_ptr))
        out = np.empty(max(n * point_step, 1), np.uint8)
        self._check(self._lib.pcop_cloud_to_pointcloud2(self._h, src, n, point_step, off_x, off_y, off_z,
                                                        out.ctypes.data_as(C.c_void_p)))
        return out[:n * point_step]

    def occupancy_grid(self, cloud=None):
        """build_initial_occupancy_grid_dataset (od.cpp:175-269) without the crop output: returns (grid int8 [H, W],
        counts int64 [H, W], row_avg int64 [H]).  cloud=None: the accumulated cloud."""
        w, h = C.c_int32(), C.c_int32()
        self._check(self._lib.pcop_occupancy_dims(self._h, C.byref(w), C.byref(h)))
        grid = np.empty((h.value, w.value), np.int8)
        counts = np.empty((h.value, w.value), np.int64)
        avg = np.empty(h.value, np.int64)
        if cloud is None:
            ptr, n = None, 0
        else:
            cloud = _f32(cloud)
            ptr, n = cloud.ctypes.data_as(C.c_void_p), cloud.shape[0]
        self._check(self._lib.pcop_occupancy_grid(self._h, ptr, n, grid.ctypes.data_as(C.c_void_p),
                                                  counts.ctypes.data_as(C.c_void_p), avg.ctypes.data_as(C.c_void_p)))
        return grid, counts, avg

    def handle_shadow_casting(self, grid, remaining_cloud, cluster_offsets, cluster_indices, world_to_sensor,
                              sensor_to_world):
        """handle_shadow_casting for every cluster + the obstacle marks (od.cpp:584-672, 817-833) on `grid`
        (int8 [H, W], e.g. from occupancy_grid()).  The two 4x4 matrices stand for the TF lookups
        "kinect2_link" <- "world" (od.cpp:592) and "world" <- "kinect2_link" (od.cpp:570, 634).
        Returns (grid int8 [H, W], shadow_records int32 [C, 6], warnings)."""
        w, h = C.c_int32(), C.c_int32()
        self._check(self._lib.pcop_occupancy_dims(self._h, C.byref(w), C.byref(h)))
        grid = np.array(grid, dtype=np.int8, order="C", copy=True)
        if grid.shape != (h.value, w.value):
            raise ValueError(f"grid must be [{h.value}, {w.value}]")
        cloud = _f32(remaining_cloud) if len(remaining_cloud) else np.zeros((0, 4), np.float32)
        off = np.ascontiguousarray(cluster_offsets, np.int32)
        idx = np.ascontiguousarray(cluster_indices, np.int32)
        n_clusters = max(len(off) - 1, 0)
        ws = np.ascontiguousarray(world_to_sensor, np.float32).reshape(16)
        sw = np.ascontiguousarray(sensor_to_world, np.float32).reshape(16)
        rec = np.zeros((max(n_clusters, 1), 6), np.int32)
        warn = C.c_uint32(0)
        self._check(self._lib.pcop_occupancy_shadows(
            self._h, cloud.ctypes.data_as(C.c_void_p) if cloud.shape[0] else None, cloud.shape[0],
            off.ctypes.data_as(C.c_void_p) if n_clusters else None, idx.ctypes.data_as(C.c_void_p) if n_clusters else None,
            n_clusters, ws.ctypes.data_as(C.c_void_p), sw.ctypes.data_as(C.c_void_p), grid.ctypes.data_as(C.c_void_p),
            rec.ctypes.data_as(C.c_void_p), C.byref(warn)))
        return grid, rec[:n_clusters].copy(), warn.value

    @property
    def accumulated_count(self) -> int:
        return int(self._lib.pcop_accumulated_count(self._h))

    def accumulate_reset(self):
        self._check(self._lib.pcop_accumulate_reset(self._h))

    def process_accumulated(self) -> Frame:
        """the pipeline on the accumulated cloud (od.cpp:699 ff); the accumulator is emptied (od.cpp:701)"""
        self._host_results_only()
        r = FrameResult()
        self._check(self._lib.pcop_process_accumulated(self._h, C.byref(r)))
        return self._frames([r])[0]

    def transform(self, cloud, transform, is_dense=False):
        cloud = _f32(cloud)
        t = np.ascontiguousarray(transform, dtype=np.float32).reshape(16)
        out = np.empty((max(cloud.shape[0], 1), 4), np.float32)
        self._check(self._lib.pcop_transform(self._h, cloud.ctypes.data_as(C.c_void_p), cloud.shape[0],
                                             t.ctypes.data_as(C.c_void_p), 1 if is_dense else 0,
                                             out.ctypes.data_as(C.c_void_p)))
        return out[:cloud.shape[0]].copy()

    def download(self, device_ptr, count, dtype):
        """copy `count` elements of a device result array (outputs | OUT_DEVICE) to a numpy array"""
        out = np.empty(count, dtype=dtype)
        addr = C.cast(device_ptr, C.c_void_p).value if not isinstance(device_ptr, int) else device_ptr
        if count:
            self._check(self._lib.pcop_download(self._h, out.ctypes.data_as(C.c_void_p), C.c_void_p(addr), out.nbytes))
        return out

    def copy_device(self, dst_device_addr: int, src_device_ptr, nbytes: int):
        """device -> device copy of a result array (e.g. into a torch tensor that NCCL sends on)"""
        addr = C.cast(src_device_ptr, C.c_void_p).value if not isinstance(src_device_ptr, int) else src_device_ptr
        if nbytes:
            self._check(self._lib.pcop_download(self._h, C.c_void_p(dst_device_addr), C.c_void_p(addr), nbytes))

    # ---- timing / accounting of the last call ----------------------------------------
    @property
    def last_elapsed_us(self) -> float:
        return float(self._lib.pcop_last_elapsed_us(self._h))

    @property
    def last_launch_count(self) -> int:
        return int(self._lib.pcop_last_launch_count(self._h))

    @property
    def last_algorithmic_bytes(self) -> float:
        return float(self._lib.pcop_last_algorithmic_bytes(self._h))

    @property
    def last_sort_pass_keys(self) -> int:
        return int(self._lib.pcop_last_sort_pass_keys(self._h))

    @property
    def last_d2h_bytes(self) -> float:
        return float(self._lib.pcop_last_d2h_bytes(self._h))

    def enable_kernel_timing(self, enable=True):
        """CUDA-event pairs around every kernel launch; totals accumulate until enabled again."""
        self._check(self._lib.pcop_enable_kernel_timing(self._h, 1 if enable else 0))

    def kernel_times(self):
        """{kernel name: (total device us, launches)} since timing was enabled."""
        out = {}
        for i in range(self._lib.pcop_kernel_timing_count(self._h)):
            name, us, n = C.c_char_p(), C.c_double(), C.c_int64()
            self._check(self._lib.pcop_kernel_timing_get(self._h, i, C.byref(name), C.byref(us), C.byref(n)))
            out[name.value.decode()] = (us.value, n.value)
        return out

    def stage_times_us(self):
        us = (C.c_float * len(abi.STAGE_NAMES))()
        self._check(self._lib.pcop_stage_times_us(self._h, us))
        return dict(zip(abi.STAGE_NAMES, [float(x) for x in us]))

    # ---- the five wrappers, stage-isolated -------------------------------------------
    def crop(self, cloud):
        cloud = _f32(cloud)
        n = cloud.shape[0]
        out = np.empty((max(n, 1), 4), np.float32)
        kept = np.empty(max(n, 1), np.int32)
        m = C.c_int32()
        self._check(self._lib.pcop_crop(self._h, cloud.ctypes.data_as(C.c_void_p), n, out.ctypes.data_as(C.c_void_p),
                                        kept.ctypes.data_as(C.c_void_p), C.byref(m)))
        return out[:m.value].copy(), kept[:m.value].copy()

    def downsample_cloud(self, cloud):
        cloud = _f32(cloud)
        n = cloud.shape[0]
        out = np.empty((max(n, 1), 4), np.float32)
        keys = np.empty(max(n, 1), np.uint32)
        v, w = C.c_int32(), C.c_uint32()
        self._check(self._lib.pcop_voxel(self._h, cloud.ctypes.data_as(C.c_void_p), n, out.ctypes.data_as(C.c_void_p),
                                         keys.ctypes.data_as(C.c_void_p), C.byref(v), C.byref(w)))
        return out[:v.value].copy(), keys[:v.value].copy(), w.value

    def remove_statistical_outliers(self, cloud):
        cloud = _f32(cloud)
        n = cloud.shape[0]
        out = np.empty((max(n, 1), 4), np.float32)
        kept = np.empty(max(n, 1), np.int32)
        s, w = C.c_int32(), C.c_uint32()
        self._check(self._lib.pcop_sor(self._h, cloud.ctypes.data_as(C.c_void_p), n, out.ctypes.data_as(C.c_void_p),
                                       kept.ctypes.data_as(C.c_void_p), C.byref(s), C.byref(w)))
        return out[:s.value].copy(), kept[:s.value].copy(), w.value

    def segment_plane_and_extract_indices(self, cloud):
        cloud = _f32(cloud)
        n = cloud.shape[0]
        vp = C.c_void_p
        rem = np.empty((max(n, 1), 4), np.float32)
        src = np.empty(max(n, 1), np.int32)
        inl = np.empty(max(n, 1), np.int32)
        pp = np.zeros(abi.MAX_PASSES, np.int32)
        pi = np.zeros(abi.MAX_PASSES, np.int32)
        pc = np.zeros((abi.MAX_PASSES, 4), np.float32)
        lc = np.zeros(4, np.float32)
        p, npass, ninl, w = C.c_int32(), C.c_int32(), C.c_int32(), C.c_uint32()
        self._check(self._lib.pcop_plane(self._h, cloud.ctypes.data_as(vp), n, rem.ctypes.data_as(vp),
                                         src.ctypes.data_as(vp), C.byref(p), C.byref(npass), pp.ctypes.data_as(vp),
                                         pi.ctypes.data_as(vp), pc.ctypes.data_as(vp), lc.ctypes.data_as(vp),
                                         inl.ctypes.data_as(vp), C.byref(ninl), C.byref(w)))
        return dict(remaining=rem[:p.value].copy(), src=src[:p.value].copy(), n_passes=npass.value, pass_points=pp,
                    pass_inliers=pi, pass_coeff=pc, last_coeff=lc, inliers=inl[:ninl.value].copy(), warnings=w.value)

    def extract_euclidian_clusters(self, cloud):
        cloud = _f32(cloud)
        n = cloud.shape[0]
        offs = np.zeros(n + 2, np.int32)
        idx = np.zeros(n + 1, np.int32)
        c, l = C.c_int32(), C.c_int32()
        self._check(self._lib.pcop_cluster(self._h, cloud.ctypes.data_as(C.c_void_p), n,
                                           offs.ctypes.data_as(C.c_void_p), idx.ctypes.data_as(C.c_void_p),
                                           C.byref(c), C.byref(l)))
        return offs[:c.value + 1].copy(), idx[:l.value].copy()

    def centroid_radius(self, cloud, offsets, indices):
        cloud = _f32(cloud)
        offsets = np.ascontiguousarray(offsets, np.int32)
        indices = np.ascontiguousarray(indices, np.int32)
        c = len(offsets) - 1
        out = np.zeros((max(c, 1), 4), np.float32)
        self._check(self._lib.pcop_centroid_radius(self._h, cloud.ctypes.data_as(C.c_void_p), cloud.shape[0],
                                                   offsets.ctypes.data_as(C.c_void_p),
                                                   indices.ctypes.data_as(C.c_void_p), c,
                                                   out.ctypes.data_as(C.c_void_p)))
        return out[:c].copy()

    def cluster_footprints(self, cloud, offsets, indices):
        """pcop_cluster_footprints: every cluster's box and ground-plane convex hull, stage-isolated.  Returns (boxes
        float32 [C, 8], hull_offsets int32 [C + 1], hull_indices int32 [H])."""
        cloud = _f32(cloud) if len(cloud) else np.zeros((0, 4), np.float32)
        offsets = np.ascontiguousarray(offsets, np.int32)
        indices = np.ascontiguousarray(indices, np.int32)
        c = len(offsets) - 1
        boxes = np.zeros((max(c, 1), 8), np.float32)
        hoff = np.zeros(c + 1, np.int32)
        hidx = np.zeros(max(len(indices), 1), np.int32)
        n = C.c_int32()
        self._check(self._lib.pcop_cluster_footprints(
            self._h, cloud.ctypes.data_as(C.c_void_p), cloud.shape[0], offsets.ctypes.data_as(C.c_void_p),
            (indices if len(indices) else hidx).ctypes.data_as(C.c_void_p), c, boxes.ctypes.data_as(C.c_void_p),
            hoff.ctypes.data_as(C.c_void_p), hidx.ctypes.data_as(C.c_void_p), C.byref(n)))
        return boxes[:c].copy(), hoff, hidx[:n.value].copy()
