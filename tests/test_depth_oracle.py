"""CPU: the two restatements of depth_image_proc's depth image -> PointXYZ conversion agree bit for bit, the
pcop_depth_image layout matches the header, and the Python depth-image helpers."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import depth_util as D
from pointcloud_obstacle_processing_b200 import DEPTH_ENCODINGS, DepthImage
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def assert_bits(a, b, what):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    assert a.shape == b.shape, what
    bad = np.flatnonzero(a.view(np.uint32) != b.view(np.uint32))
    assert bad.size == 0, f"{what}: {bad.size} words differ, first at {bad[:4]}: {a.reshape(-1)[bad[:4]]} vs {b.reshape(-1)[bad[:4]]}"


@pytest.mark.parametrize("u16", [True, False])
@pytest.mark.parametrize("shape", [(64, 48, 0, 0), (37, 11, 0, 0), (40, 9, 3, 0), (33, 7, 5, 2), (1, 1, 0, 0),
                                   (8, 1, 0, 4), (1, 9, 1, 1)])
def test_oracle_and_numpy_agree(u16, shape):
    """random depths with 0, 1, 65535 / NaN, +-Inf, -0.0, negative, huge and subnormal values; odd widths, padded
    steps, data at odd offsets, arbitrary cx / cy and fx != fy"""
    W, H, pad, off = shape
    rng = np.random.default_rng(W * 1000 + H * 10 + pad + (0 if u16 else 7))
    for _ in range(3):
        im = D.random_image(rng, W, H, u16=u16, pad=pad, offset=off)
        assert im.fx != im.fy
        a, b = D.oracle_to_xyz(im), D.numpy_to_xyz(im)
        assert a.shape == (W * H, 4)
        assert_bits(a, b, f"{shape} u16={u16}")


def test_special_values_follow_the_semantics():
    W, H = 6, 2
    px = np.array([[0, 1, 65535, 1000, 2, 3], [7, 0, 0, 9, 1, 65534]], np.uint16)
    im = DepthImage.from_array(px, 500.0, 400.0, 2.25, 0.75)
    got = D.oracle_to_xyz(im).reshape(H, W, 4)
    assert np.all(got[..., 3] == 1.0)
    assert got[0, 0, :3].view(np.uint32).tolist() == [0x7FC00000] * 3
    assert got[0, 2, 2] == np.float32(65535) * np.float32(0.001)
    kx = np.float32(np.float64(np.float32(0.001)) / 500.0)
    assert got[0, 3, 0] == (np.float32(3) - np.float32(2.25)) * np.float32(1000) * kx
    f = np.array([[0.0, -0.0, np.nan, np.inf, -np.inf, 2.5]], np.float32)
    got = D.oracle_to_xyz(DepthImage.from_array(f, 500.0, 400.0, 2.25, 0.75))
    assert got[0, 2] == 0.0 and got[1, 2] == 0.0 and np.signbit(got[1, 2])
    assert np.all(np.isnan(got[2:5, :3])) and got[5, 2] == np.float32(2.5)


def test_scene_images():
    im = D.scene_image(0)
    assert (im.width, im.height, im.step, im.encoding) == (640, 480, 1280, abi.DEPTH_16UC1)
    holes = float(np.mean(im.data == 0))
    assert 0.08 < holes < 0.3, holes
    xyz = D.numpy_to_xyz(im)
    z = xyz[:, 2][np.isfinite(xyz[:, 2])]
    assert 0.5 <= z.min() and z.max() <= 4.5
    q = D.scene_image(0, D.QHD)
    assert (q.width, q.height, q.step) == (960, 540, 1920)
    assert_bits(D.oracle_to_xyz(q), D.numpy_to_xyz(q), "qhd scene")
    f = D.scene_image(1, float32=True)
    assert f.encoding == abi.DEPTH_32FC1 and f.step == 2560
    assert_bits(D.oracle_to_xyz(f), D.numpy_to_xyz(f), "32FC1 scene")


def test_to_pointcloud2_carries_the_points():
    from pc2_util import LAYOUTS
    import oracle_lib as O
    im = D.random_image(np.random.default_rng(3), 13, 5, u16=False, pad=2)
    msg = D.to_pointcloud2(im, 4)
    assert msg.size == 13 * 5 * 32
    assert_bits(O.pointcloud2_to_xyz(msg, 65, *LAYOUTS["xyzrgb32"]), D.oracle_to_xyz(im), "decoded XYZRGB message")


def test_from_array_and_encodings():
    assert DEPTH_ENCODINGS == {"16UC1": abi.DEPTH_16UC1, "mono16": abi.DEPTH_16UC1, "32FC1": abi.DEPTH_32FC1}
    big = np.arange(7 * 12, dtype=np.uint16).reshape(7, 12)
    im = DepthImage.from_array(big[:, :9], 1.0, 2.0, 3.0, 4.0)
    assert (im.width, im.height, im.step, im.encoding) == (9, 7, 24, abi.DEPTH_16UC1)
    assert_bits(D.numpy_to_xyz(im), D.numpy_to_xyz(DepthImage.from_array(np.ascontiguousarray(big[:, :9]), 1, 2, 3, 4)),
                "padded view")
    with pytest.raises(ValueError):
        DepthImage.from_array(np.zeros((2, 2), np.int32), 1, 1, 1, 1)
    with pytest.raises(ValueError):
        DepthImage.from_array(np.zeros((2, 4), np.uint16)[:, ::2], 1, 1, 1, 1)


def test_depth_image_layout_matches_header(tmp_path):
    src = tmp_path / "sz.c"
    fields = ["data", "width", "height", "step", "encoding", "fx", "fy", "cx", "cy"]
    src.write_text('#include "pcop.h"\n#include <stdio.h>\n#include <stddef.h>\nint main(void){printf("%zu'
                   + " %zu" * len(fields) + '\\n",sizeof(pcop_depth_image)'
                   + "".join(f",offsetof(pcop_depth_image,{f})" for f in fields)
                   + ');printf("%d %d\\n",PCOP_DEPTH_16UC1,PCOP_DEPTH_32FC1);return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(abi.DepthImageC)] + [getattr(abi.DepthImageC, f).offset for f in fields] + \
        [abi.DEPTH_16UC1, abi.DEPTH_32FC1]
