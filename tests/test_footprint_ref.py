"""CPU: the two restatements of the obstacle footprints (PCOP_OUT_FOOTPRINTS) agree bit for bit on known-answer and
random clusters, the exactness case defeats plain double arithmetic, and the pcop_frame_footprints layout matches the
header."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import footprint_util as F
from pointcloud_obstacle_processing_b200 import Frame
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = F.cases()


def assert_same(a, b, what):
    for k, (x, y) in enumerate(zip(a, b)):
        x, y = np.ascontiguousarray(x), np.ascontiguousarray(y)
        assert x.shape == y.shape, f"{what}: array {k} shape {x.shape} vs {y.shape}"
        assert x.tobytes() == y.tobytes(), f"{what}: array {k} differs"


@pytest.mark.parametrize("name", sorted(CASES))
def test_restatements_agree(name):
    cloud, off, idx = CASES[name]
    assert_same(F.oracle_footprints(cloud, off, idx), F.numpy_footprints(cloud, off, idx), name)


def hull_of(name, k=0):
    cloud, off, idx = CASES[name]
    boxes, hoff, hidx = F.oracle_footprints(cloud, off, idx)
    return cloud, boxes[k], hidx[hoff[k]:hoff[k + 1]]


def test_known_answers():
    cloud, box, h = hull_of("one_point")
    assert len(h) == 1 and box.tolist() == [1.5, -2.0, 0.0, 0.0, 1.5, -2.0, 0.0, 0.0]
    cloud, box, h = hull_of("two_points")
    assert cloud[h, :2].tolist() == [[-1.0, 0.5], [1.0, 2.0]]
    cloud, box, h = hull_of("all_identical")
    assert h.tolist() == [0] and box[2] == 0.0 and box[6] == 6.0
    cloud, box, h = hull_of("collinear")
    assert cloud[h, :2].tolist() == [[-1.0, 0.5], [2.5, 2.25]] and h.tolist() == [1, 3]
    cloud, box, h = hull_of("stacked_in_z")  # the corners, each as its smallest index
    assert cloud[h, :2].tolist() == [[0, 0], [1, 0], [1, 1], [0, 1]]
    _, off, idx = CASES["stacked_in_z"]
    for v in h:
        same = [int(i) for i in idx if cloud[i, 0] == cloud[v, 0] and cloud[i, 1] == cloud[v, 1]]
        assert v == min(same) and len(same) == 6
    cloud, box, h = hull_of("signed_zeros")  # +-0 are one point; the box orders -0 below +0
    assert h.tolist() == [0, 2, 1] and np.signbit(box[0]) and np.signbit(box[1]) and not np.signbit(box[5])
    cloud, box, h = hull_of("square_boundary")  # points on the edges are not vertices
    assert len(h) == 4
    cloud, box, h = hull_of("convex_position_64")
    assert len(h) == 64
    cloud, box, h = hull_of("convex_position_exact_1024")
    assert len(h) == len(cloud) == 1024
    for k, name in enumerate(("nan", "inf")):
        cloud, box, h = hull_of("nonfinite_singletons", k)
        assert len(h) == 1 and box.view(np.uint32)[[0, 1, 2, 4, 5, 6]].tolist() == \
            cloud[h[0], [0, 1, 2, 0, 1, 2]].view(np.uint32).tolist()
    boxes, hoff, hidx = F.oracle_footprints(*CASES["empty_clusters"])
    assert hoff.tolist() == [0, 0, 3, 3] and not boxes[0].any() and not boxes[2].any()


def test_exactness_case_defeats_plain_double():
    a, b, c = F.EXACT_A, F.EXACT_B, F.EXACT_C
    # as the monotone chain evaluates it (A < C < B in x) and with the pivot C
    for p, q, r in ((a, c, b), (a, b, c)):
        exact = F.orient_exact_sign(p, q, r)
        assert exact != 0 and F.orient_plain_double_sign(p, q, r) == -exact
        assert np.sign(F.oracle().pcop_oracle_orient2d(*p, *q, *r)) == exact
    # C lies right of A -> B: the hull is the triangle A, B, C counter-clockwise
    cloud, box, h = hull_of("exactness")
    assert h.tolist() == [0, 2, 1]


def test_all_extreme_sets_put_the_second_point_on_the_lower_chain():
    """the sets that would overflow a monotone chain's stack by one entry: every point extreme, the second point in
    (x, y) order a lower-chain vertex (the hull starts at the first point and walks the lower chain first)"""
    cloud, off, idx = CASES["all_extreme_4096_second_on_lower_chain"]
    boxes, hoff, hidx = F.oracle_footprints(cloud, off, idx)
    assert len(hidx) == len(cloud) == 4096
    order = np.lexsort((cloud[:, 1], cloud[:, 0]))
    assert hidx[0] == order[0] and hidx[1] == order[1]
    p = F.sheared_polygon(45)
    o = np.lexsort((p[:, 1], p[:, 0]))
    b, hoff, hidx = F.oracle_footprints(p, [0, len(p)], np.arange(len(p)))
    assert len(hidx) == len(p) > 4096 and hidx[1] == o[1]


def test_convex_position_keeps_every_extreme_point():
    cloud, off, idx = CASES["convex_position_1000"]
    boxes, hoff, hidx = F.numpy_footprints(cloud, off, idx)
    assert 990 <= len(hidx) <= 1000  # (float rounding may pull a few points just inside)


def test_frame_hulls_and_layout(tmp_path):
    fr = Frame(n_clusters=2)
    assert fr.hulls is None and fr.boxes is None
    fr.hull_offsets, fr.hull_indices = np.array([0, 3, 4], np.int32), np.array([5, 1, 2, 7], np.int32)
    assert [h.tolist() for h in fr.hulls] == [[5, 1, 2], [7]]
    src = tmp_path / "sz.c"
    fields = ["n_clusters", "n_hull_vertices", "boxes", "hull_offsets", "hull_indices"]
    src.write_text('#include "pcop.h"\n#include <stdio.h>\n#include <stddef.h>\nint main(void){printf("%zu'
                   + " %zu" * len(fields) + '\\n",sizeof(pcop_frame_footprints)'
                   + "".join(f",offsetof(pcop_frame_footprints,{f})" for f in fields)
                   + ');printf("%d %d %zu %zu\\n",PCOP_OUT_FOOTPRINTS,PCOP_OUT_ALL & PCOP_OUT_FOOTPRINTS,'
                   'sizeof(pcop_frame_result),sizeof(pcop_params));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(abi.FrameFootprints)] + [getattr(abi.FrameFootprints, f).offset for f in fields] + \
        [abi.OUT_FOOTPRINTS, 0, C.sizeof(abi.FrameResult), C.sizeof(abi.Params)]
