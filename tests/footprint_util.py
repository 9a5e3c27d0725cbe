"""Obstacle footprints (PCOP_OUT_FOOTPRINTS) for the footprint tests and benchmark: TEST INFRASTRUCTURE.

Two restatements of the box and convex hull of include/pcop.h: the C++ oracle (footprint_oracle.cpp: Shewchuk's
filtered orient2d and Andrew's monotone chain, built with the pipeline oracle's flags into a temporary directory) and
an independent Python one here (every coordinate of a cluster scaled by one power of two to an exact integer,
quickhull on integer cross products, a numpy totalOrder box).  Also the clusters the tests feed both with."""
import ctypes as C
import math
import os
import subprocess
import tempfile
from fractions import Fraction

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SRC = os.path.join(_ROOT, "tests", "footprint_oracle.cpp")
_lib = None


def oracle():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="pcop_footprint_oracle_"), "libfootprint_oracle.so")
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-std=c++17", "-Wall",
                               "-Wextra", "-shared", "-o", out, _SRC])
        _lib = C.CDLL(out)
        _lib.pcop_oracle_orient2d.restype = C.c_double
        _lib.pcop_oracle_orient2d.argtypes = [C.c_float] * 6
        _lib.pcop_oracle_cluster_footprints.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                                        C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def oracle_footprints(cloud, offsets, indices):
    """(boxes float32 [C, 8], hull_offsets int32 [C + 1], hull_indices int32 [H]) from the C++ restatement"""
    cloud = np.ascontiguousarray(cloud, np.float32).reshape(-1, 4)
    offsets = np.ascontiguousarray(offsets, np.int32)
    indices = np.ascontiguousarray(indices, np.int32)
    c = len(offsets) - 1
    boxes = np.zeros((max(c, 1), 8), np.float32)
    hoff = np.zeros(c + 1, np.int32)
    hidx = np.zeros(max(len(indices), 1), np.int32)
    n = C.c_int32()
    oracle().pcop_oracle_cluster_footprints(_ptr(cloud), len(cloud), _ptr(offsets), _ptr(indices if len(indices) else hidx),
                                            c, _ptr(boxes), _ptr(hoff), _ptr(hidx), C.byref(n))
    return boxes[:c].copy(), hoff, hidx[:n.value].copy()


# ---- the independent restatement -------------------------------------------------------------------------------
def _order_keys(v):
    """IEEE totalOrder of float32 as uint32"""
    u = np.ascontiguousarray(v, np.float32).view(np.uint32)
    return np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint32)


def _from_keys(k):
    k = np.asarray(k, np.uint32)
    return np.where(k & np.uint32(0x80000000), k & np.uint32(0x7FFFFFFF), ~k).astype(np.uint32).view(np.float32)


def box(pts):
    """float32 [8] of the members pts [n, 4] (n >= 1)"""
    if len(pts) == 1:
        return np.array([pts[0, 0], pts[0, 1], pts[0, 2], 0, pts[0, 0], pts[0, 1], pts[0, 2], 0], np.float32)
    k = _order_keys(pts[:, :3])
    out = np.zeros(8, np.float32)
    out[0:3] = _from_keys(k.min(axis=0))
    out[4:7] = _from_keys(k.max(axis=0))
    return out


def _scaled(xy):
    """exact integers of the float32 coordinates xy [n, 2] (all finite), scaled by one common power of two"""
    m, e = np.frexp(xy.astype(np.float64))  # xy = m * 2^e, |m| in [0.5, 1): 24-bit integer mantissa at 2^(e - 24)
    mant = np.ldexp(m, 24).astype(np.int64)
    e = e.astype(np.int64) - 24
    nz = mant != 0
    e0 = int(e[nz].min()) if nz.any() else 0
    shift = np.where(nz, e - e0, 0)
    return [(int(a) << int(s), int(b) << int(t)) for a, b, s, t in zip(mant[:, 0], mant[:, 1], shift[:, 0], shift[:, 1])]


def _cross(o, a, b):
    return (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0])


def hull(pts, idx):
    """remaining-cloud indices of the hull vertices of the members pts [n, 4] with indices idx, counter-clockwise from
    the lexicographically smallest (x, y)"""
    if len(pts) == 1:
        return [int(idx[0])]
    first = {}  # distinct (x, y) -> smallest index; +0 and -0 are one value
    for q, i in zip(_scaled(pts[:, :2]), idx):
        if q not in first or i < first[q]:
            first[q] = int(i)
    P = list(first)
    if len(P) == 1:
        return [first[P[0]]]
    a, b = min(P), max(P)
    out = [a]

    def side(p, q, S):  # the points of S strictly right of p -> q (outside a counter-clockwise hull)
        return [s for s in S if _cross(p, q, s) < 0]

    # quickhull, iteratively: the vertices strictly between p and q, in order, from the points right of p -> q
    def chain(p, q, S):
        res, stack = [], [(p, q, S, False)]
        while stack:
            p, q, S, emit = stack.pop()
            if emit:
                res.append(p)
                continue
            if not S:
                continue
            d = (q[0] - p[0], q[1] - p[1])
            # the farthest point; among equally far ones the one furthest along p -> q (an end of that edge)
            far = max(S, key=lambda s: (-_cross(p, q, s), d[0] * s[0] + d[1] * s[1]))
            stack.append((far, q, side(far, q, S), False))
            stack.append((far, None, None, True))
            stack.append((p, far, side(p, far, S), False))
        return res

    out += chain(a, b, side(a, b, P))
    out.append(b)
    out += chain(b, a, side(b, a, P))
    return [first[q] for q in out]


def numpy_footprints(cloud, offsets, indices):
    """(boxes, hull_offsets, hull_indices) from the Python restatement"""
    cloud = np.asarray(cloud, np.float32).reshape(-1, 4)
    c = len(offsets) - 1
    boxes = np.zeros((c, 8), np.float32)
    hoff, hidx = [0], []
    for k in range(c):
        idx = np.asarray(indices[offsets[k]:offsets[k + 1]], np.int64)
        if len(idx):
            pts = cloud[idx]
            boxes[k] = box(pts)
            hidx += hull(pts, idx)
        hoff.append(len(hidx))
    return boxes, np.array(hoff, np.int32), np.array(hidx, np.int32)


# ---- predicates for the exactness case -----------------------------------------------------------------------------
def orient_exact_sign(a, b, c):
    f = [Fraction(float(v)) for v in (*a, *b, *c)]
    d = (f[0] - f[4]) * (f[3] - f[5]) - (f[1] - f[5]) * (f[2] - f[4])
    return (d > 0) - (d < 0)


def orient_plain_double_sign(a, b, c):
    """the determinant of orient2d's first stage, in plain double arithmetic (float inputs widened)"""
    ax, ay, bx, by, cx, cy = (float(np.float32(v)) for v in (*a, *b, *c))
    d = (ax - cx) * (by - cy) - (ay - cy) * (bx - cx)
    return (d > 0) - (d < 0)


# ---- clusters ------------------------------------------------------------------------------------------------------
def circle(n, r=1.0, z=0.0, cx=0.0, cy=0.0):
    """n points on a circle: with n large most are extreme (float rounding leaves a few just inside)"""
    t = np.arange(n) * (2 * math.pi / n)
    p = np.zeros((n, 4), np.float32)
    p[:, 0] = cx + r * np.cos(t)
    p[:, 1] = cy + r * np.sin(t)
    p[:, 2] = z
    p[:, 3] = 1.0
    return p


def blob(rng, n, scale=1.0):
    p = np.zeros((n, 4), np.float32)
    p[:, :3] = rng.normal(size=(n, 3)) * scale
    p[:, 3] = 1.0
    return p


def concat(clusters, rng=None, mix=False):
    """one cloud from a list of member arrays: (cloud, offsets, indices); members shuffled over the cloud when rng, and
    with mix the member order inside every cluster as well (its pieces are then no contiguous runs of the input)"""
    cloud = np.concatenate(clusters) if clusters else np.zeros((0, 4), np.float32)
    sizes = [len(c) for c in clusters]
    perm = rng.permutation(len(cloud)) if rng is not None else np.arange(len(cloud))
    inv = np.empty_like(perm)
    inv[perm] = np.arange(len(cloud))
    out = cloud[perm]  # out[j] = cloud[perm[j]], so cloud point i sits at inv[i]
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    inv = inv.astype(np.int32)
    if mix:
        for k in range(len(sizes)):
            inv[offsets[k]:offsets[k + 1]] = rng.permutation(inv[offsets[k]:offsets[k + 1]])
    return np.ascontiguousarray(out), offsets, inv


# a near-collinear triple across many binades: orient2d(A, C, B) and orient2d(A, B, C) (the pivot last) have the
# wrong sign in plain double arithmetic -- A - B and A - C round -- while the exact sign puts C right of A -> B
EXACT_A = (float.fromhex("0x1.69f74p-51"), float.fromhex("0x1.28f03ap-50"))
EXACT_B = (6.0, 10.0)
EXACT_C = (3.0, 5.0)


def _pts(xy, z=None):
    xy = np.asarray(xy, np.float32).reshape(-1, 2)
    p = np.zeros((len(xy), 4), np.float32)
    p[:, :2] = xy
    p[:, 2] = 0.0 if z is None else z
    p[:, 3] = 1.0
    return p


def cases():
    """{name: (cloud, offsets, indices)}: the known-answer and random clusters both restatements must agree on"""
    rng = np.random.default_rng(2024)
    out = {}
    out["one_point"] = concat([_pts([[1.5, -2.0]])])
    out["two_points"] = concat([_pts([[1.0, 2.0], [-1.0, 0.5]])])
    out["all_identical"] = concat([_pts([[0.25, 0.5]] * 7, z=np.arange(7, dtype=np.float32))])
    out["collinear"] = concat([_pts([[k * 0.5, k * 0.25 + 1.0] for k in (3, -2, 0, 5, 1, 5, -2)])])
    # duplicates stacked in z: a square with a column of points at every corner and inside, members shuffled
    sq = [[x, y] for x in (0.0, 1.0) for y in (0.0, 1.0)] + [[0.5, 0.5]]
    out["stacked_in_z"] = concat([_pts(sq * 6, z=np.repeat(np.arange(6, dtype=np.float32), 5))], rng)
    out["signed_zeros"] = concat([_pts([[0.0, 0.0], [-0.0, 1.0], [1.0, -0.0], [-0.0, -0.0], [0.0, 1.0], [1.0, 0.0],
                                        [-0.0, 0.5]])])
    out["convex_position_64"] = concat([circle(64, 2.0, 0.3, 1.0, -1.0)], rng)
    out["convex_position_1000"] = concat([circle(1000, 5.0)], rng)
    sqb = [[x, y] for x in range(11) for y in range(11) if x in (0, 10) or y in (0, 10)]
    out["convex_position_exact_1024"] = concat([convex_polygon(20, 1.0)], rng)
    out["all_extreme_4096_second_on_lower_chain"] = concat([all_extreme_second_on_lower(4096, rng)], rng, mix=True)
    out["square_boundary"] = concat([_pts(np.array(sqb, np.float32) * 0.1)], rng)
    nf = _pts([[np.nan, 1.0]])
    out["nonfinite_singletons"] = concat([nf, _pts([[np.inf, -np.inf]]), _pts([[1.0, 2.0]]),
                                          _pts([[-np.inf, 0.0]], z=np.float32(np.nan))])
    out["exactness"] = concat([_pts([EXACT_A, EXACT_C, EXACT_B])])
    out["exactness_in_a_cluster"] = concat([_pts([EXACT_A, EXACT_C, EXACT_B, [3.0, 4.0], [1.0, 3.0]] +
                                                 [[float(np.float32(EXACT_C[0] * k / 7)), float(np.float32(EXACT_C[1] * k / 7))]
                                                  for k in range(1, 14)])], rng)
    # random: blobs of many sizes, lattice points (duplicates and collinear runs), clusters of mixed scale
    cl = [blob(rng, n, s) for n, s in ((3, 1.0), (17, 0.1), (150, 2.0), (1000, 1.0), (4096, 0.5), (5000, 3.0))]
    cl.append(_pts(rng.integers(-4, 5, size=(400, 2)).astype(np.float32) * 0.25, z=rng.normal(size=400)))
    cl.append(_pts(rng.normal(size=(300, 2)).astype(np.float32) * np.float32(2.0 ** -20) + np.float32(1000.0)))
    out["random_clusters"] = concat(cl, rng)
    out["random_20k"] = concat([blob(rng, 20000, 1.0), circle(20000, 3.0, 0.0, 10.0, 10.0)], rng)
    out["empty_clusters"] = (_pts([[1, 1], [2, 2], [3, 1]]), np.array([0, 0, 3, 3], np.int32), np.array([2, 0, 1], np.int32))
    return out


def convex_polygon(m, z=0.0):
    """every vertex extreme: the polygon whose edges are all primitive integer vectors of max-norm <= m, in angle
    order (about 2.43 m^2 vertices; integer coordinates below m^3, exact in float32 for m <= 250)"""
    a, b = np.meshgrid(np.arange(-m, m + 1), np.arange(-m, m + 1))
    a, b = a.ravel(), b.ravel()
    keep = (np.gcd(a, b) == 1)
    a, b = a[keep], b[keep]
    order = np.argsort(np.arctan2(b, a), kind="stable")
    xy = np.cumsum(np.stack([a[order], b[order]], 1), axis=0)
    p = np.zeros((len(xy), 4), np.float32)
    p[:, :2] = xy - xy.min(axis=0)
    p[:, 2] = z
    p[:, 3] = 1.0
    return p


def sheared_polygon(m, z=0.0, dx=0.0):
    """convex_polygon(m) under x' = 97 x + y, y' = -y (still exact in float32 for m <= 45): every vertex is extreme, and
    the second point in (x, y) order is a vertex of the lower chain -- the order in which a monotone chain's stack
    peaks at one more entry than there are points, unless the upper pass leaves the lower chain out"""
    p = convex_polygon(m, z)
    x, y = p[:, 0].astype(np.float64), p[:, 1].astype(np.float64)
    p[:, 0] = 97.0 * x + y + dx
    p[:, 1] = -y
    return p


def all_extreme_second_on_lower(n, rng, m=45):
    """n vertices of sheared_polygon(m), among them its first two and its last in (x, y) order (so the second point
    stays on the lower chain)"""
    p = sheared_polygon(m)
    order = np.lexsort((p[:, 1], p[:, 0]))
    keep = np.concatenate([order[:2], order[-1:], rng.choice(order[2:-1], n - 3, replace=False)])
    return p[np.sort(keep)]
