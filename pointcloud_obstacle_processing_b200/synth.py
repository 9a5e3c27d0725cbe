"""Synthetic frames + parameter sets of the five BASELINE.json configs (ctypes over synth/synth.cpp)."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from ._ctypes_abi import Params

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "synth", "libpcop_synth.so")
_lib = None


def _load():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            from ._build import build_synth
            build_synth()
        lib = C.CDLL(_LIB_PATH)
        lib.pcop_synth_points.restype = C.c_int32
        lib.pcop_synth_points.argtypes = [C.c_int]
        lib.pcop_synth_frame.restype = C.c_int32
        lib.pcop_synth_frame.argtypes = [C.c_int, C.c_int, C.c_void_p]
        lib.pcop_synth_params.restype = C.c_int
        lib.pcop_synth_params.argtypes = [C.c_int, C.POINTER(Params)]
        lib.pcop_synth_depth_camera.restype = None
        lib.pcop_synth_depth_camera.argtypes = [C.c_int, C.c_int, C.c_int] + [C.c_double] * 4 + [C.c_void_p]
        _lib = lib
    return _lib


def points_per_frame(config: int) -> int:
    return int(_load().pcop_synth_points(config))


def params(config: int) -> Params:
    p = Params()
    if _load().pcop_synth_params(config, C.byref(p)) != 0:
        raise ValueError(f"unknown config {config}")
    return p


def frame(config: int, index: int = 0, out: np.ndarray = None) -> np.ndarray:
    """One frame as float32 [n, 4] (pcl::PointXYZ layout)."""
    n = points_per_frame(config)
    if n <= 0:
        raise ValueError(f"unknown config {config}")
    if out is None:
        out = np.empty((n, 4), dtype=np.float32)
    assert out.dtype == np.float32 and out.flags.c_contiguous and out.size == n * 4
    _load().pcop_synth_frame(config, index, out.ctypes.data_as(C.c_void_p))
    return out


def frames(config: int, first: int, count: int, out: np.ndarray = None, threads: int = None) -> np.ndarray:
    """`count` frames [count, n, 4]; generated on a thread pool (the generator releases the GIL)."""
    n = points_per_frame(config)
    if out is None:
        out = np.empty((count, n, 4), dtype=np.float32)
    threads = threads or min(32, os.cpu_count() or 1)
    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(lambda k: frame(config, first + k, out[k]), range(count)))
    return out


def depth_camera_frame(index: int, width: int, height: int, fx: float, fy: float, cx: float, cy: float) -> np.ndarray:
    """Config 3's scene of frame `index` seen by another pinhole camera: float32 [height * width, 4] in the camera
    frame, point v * width + u = pixel (u, v), NaN where the camera has no return.  The 640 x 480 camera at fx = fy =
    525, cx = 319.5, cy = 239.5 gives frame(3, index)."""
    out = np.empty((width * height, 4), dtype=np.float32)
    _load().pcop_synth_depth_camera(index, width, height, fx, fy, cx, cy, out.ctypes.data_as(C.c_void_p))
    return out
