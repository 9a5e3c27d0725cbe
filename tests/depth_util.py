"""Depth images for the depth-ingest tests and benchmark: TEST INFRASTRUCTURE.

Two restatements of depth_image_proc's depth image -> PointXYZ conversion: the C++ oracle (depth_oracle.cpp, built
with the pipeline oracle's flags into a temporary directory) and an independent numpy one (float32 arrays, one
rounded op at a time).  Also the XYZRGB PointCloud2 message depth_image_proc publishes for an image, and depth images
rendered from the synthetic config-3 scene."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from pc2_util import pack
from pointcloud_obstacle_processing_b200 import DEPTH_ENCODINGS, DepthImage, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SRC = os.path.join(_ROOT, "tests", "depth_oracle.cpp")
_lib = None

QNAN = np.array(0x7FC00000, np.uint32).view(np.float32)  # std::numeric_limits<float>::quiet_NaN()
CONFIG3 = (640, 480, 525.0, 525.0, 319.5, 239.5)               # width, height, fx, fy, cx, cy
QHD = (960, 540, 540.686, 540.686, 479.75, 269.75)             # kinect2_bridge qhd: half the hd calibration


def oracle():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="pcop_depth_oracle_"), "libdepth_oracle.so")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-std=c++17", "-Wall",
                               "-Wextra", "-shared", "-I", os.path.join(_ROOT, "include"), "-o", out, _SRC])
        _lib = C.CDLL(out)
        _lib.pcop_oracle_depth_image_to_xyz.argtypes = [C.POINTER(abi.DepthImageC), C.c_void_p]
    return _lib


def encoding(image):
    e = image.encoding
    return DEPTH_ENCODINGS[e] if isinstance(e, str) else int(e)


def raw_bytes(image):
    """the image's payload as uint8 (a view of the caller's buffer)"""
    d = image.data
    if isinstance(d, np.ndarray):
        if d.flags.c_contiguous:
            return d.reshape(-1).view(np.uint8)
        # a padded view of a larger array (DepthImage.from_array): step * height bytes from its first pixel
        return np.ctypeslib.as_array((C.c_ubyte * (image.step * image.height)).from_address(d.ctypes.data))
    return np.frombuffer(d, np.uint8)


def oracle_to_xyz(image):
    """pcop_oracle_depth_image_to_xyz: float32 [width * height, 4]"""
    image = DepthImage(*image)
    raw = np.ascontiguousarray(raw_bytes(image)) if image.width * image.height else np.zeros(1, np.uint8)
    d = abi.DepthImageC(raw.ctypes.data, image.width, image.height, image.step, encoding(image), image.fx, image.fy,
                        image.cx, image.cy)
    out = np.empty((max(image.width * image.height, 1), 4), np.float32)
    assert oracle().pcop_oracle_depth_image_to_xyz(C.byref(d), out.ctypes.data_as(C.c_void_p)) == 0
    return out[:image.width * image.height].copy()


def numpy_to_xyz(image):
    """the same conversion in numpy, written from the semantics rather than from the oracle"""
    image = DepthImage(*image)
    W, H, step = image.width, image.height, image.step
    u16 = encoding(image) == abi.DEPTH_16UC1
    dt = np.dtype("<u2") if u16 else np.dtype("<f4")
    raw = np.ascontiguousarray(raw_bytes(image))
    depth = np.empty((H, W), dt)
    for v in range(H):
        depth[v] = raw[v * step:v * step + W * dt.itemsize].view(dt)
    d = depth.astype(np.float32)  # (uint16 -> float32 is exact)
    valid = depth != 0 if u16 else np.isfinite(d)
    unit = np.float64(np.float32(0.001)) if u16 else np.float64(1.0)
    kx, ky = np.float32(unit / np.float64(image.fx)), np.float32(unit / np.float64(image.fy))
    cx, cy = np.float32(image.cx), np.float32(image.cy)
    u = np.arange(W, dtype=np.float32)[None, :]
    v = np.arange(H, dtype=np.float32)[:, None]
    with np.errstate(all="ignore"):
        x = ((u - cx) * d) * kx
        y = ((v - cy) * d) * ky
        z = d * np.float32(0.001) if u16 else d
    out = np.empty((H, W, 4), np.float32)
    out[..., 0] = np.where(valid, x, QNAN)
    out[..., 1] = np.where(valid, y, QNAN)
    out[..., 2] = np.where(valid, z, QNAN)
    out[..., 3] = np.float32(1.0)
    return out.reshape(-1, 4)


def to_pointcloud2(image, seed=0):
    """the payload of the point_step-32 XYZRGB PointCloud2 depth_image_proc publishes for the image (rgb filler)"""
    return pack(numpy_to_xyz(image), "xyzrgb32", seed)


def depth16(cloud, width, height):
    """a camera-frame organised cloud -> 16UC1 millimetres [height, width] (0 where the cloud has no point)"""
    z = cloud[:, 2].astype(np.float64).reshape(height, width)
    return np.where(np.isfinite(z), np.rint(z * 1000.0), 0).astype(np.uint16)


def depth32(cloud, width, height):
    """the same as 32FC1 metres (NaN where the cloud has no point)"""
    return np.ascontiguousarray(cloud[:, 2].reshape(height, width), np.float32)


def scene_image(index, camera=CONFIG3, float32=False):
    """config 3's scene of frame `index` as a 16UC1 (or 32FC1) DepthImage of `camera` (CONFIG3: the config-3 frame
    quantised to millimetres; QHD: 960 x 540 at kinect2 qhd intrinsics)"""
    W, H, fx, fy, cx, cy = camera
    cloud = synth.frame(3, index) if camera == CONFIG3 else synth.depth_camera_frame(index, W, H, fx, fy, cx, cy)
    img = depth32(cloud, W, H) if float32 else depth16(cloud, W, H)
    return DepthImage.from_array(img, fx, fy, cx, cy)


def random_image(rng, width, height, u16=True, pad=0, offset=0):
    """an image of random depths with the edge values of its encoding, rows padded by `pad` pixels, its data starting
    `offset` bytes into a buffer (a uint8 view); returns the DepthImage"""
    dt = np.uint16 if u16 else np.float32
    step = (width + pad) * np.dtype(dt).itemsize
    if u16:
        px = rng.integers(0, 65536, (height, width + pad)).astype(np.uint16)
        px[rng.random((height, width + pad)) < 0.1] = 0
        edge = np.array([0, 1, 65535, 2, 500, 4500], np.uint16)
    else:
        px = rng.uniform(-2.0, 8.0, (height, width + pad)).astype(np.float32)
        px[rng.random((height, width + pad)) < 0.05] = np.nan
        edge = np.array([0.0, -0.0, np.nan, np.inf, -np.inf, -1.5, 3.0e38, -3.0e38, 1.0e-40, 65535.0], np.float32)
    flat = px.reshape(-1)
    k = min(len(edge), flat.size)
    flat[:k] = edge[:k]
    buf = np.zeros(offset + px.nbytes + 16, np.uint8)
    buf[offset:offset + px.nbytes] = px.view(np.uint8).reshape(-1)
    fx, fy = rng.uniform(300.0, 900.0, 2)
    cx, cy = rng.uniform(0.0, max(width, 1)), rng.uniform(0.0, max(height, 1))
    return DepthImage(buf[offset:offset + step * height], width, height, step,
                      abi.DEPTH_16UC1 if u16 else abi.DEPTH_32FC1, float(fx), float(fy), float(cx), float(cy))
