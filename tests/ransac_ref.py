"""Literal numpy restatement of the RANSAC plane loop (segment_plane_and_extract_indices, od.cpp:364-399):
pcl::SACSegmentation<SACMODEL_PERPENDICULAR_PLANE, SAC_RANSAC>::segment re-seeded per pass, then ExtractIndices.
Written from PCL's ransac.hpp / sac_model_plane.hpp / sac_model_perpendicular_plane.hpp, independently of the oracle
(no oracle import), so that the parameters the defaults never reach are pinned by two restatements.

What it restates exactly: the mt19937 stream, drawIndexSample on a persistent shuffled_indices array, isSampleGood's
ratio test with up to 1000 draws, computeModelCoefficients in float32 in the same operation order, the perpendicular
angle test in float64 (cosine domain), the float32 distance predicate, the adaptive-k rule with its clamps, the
max_iterations and max_skip limits, the od.cpp:379 loop rule, the break on no inliers and the order-preserving
extraction.  optimizeModelCoefficients (optimize_coefficients = 1) is not restated: with it the result stops at the
RANSAC model and inlier set, and the refined model is checked by invariants.
"""
import math

import numpy as np

MAX_PASSES = 16  # PCOP_MAX_PLANE_PASSES_RECORDED
WARN_PLANE_BREAK = 4
DBL_EPS = 2.220446049250313e-16
HALF_PI = 1.57079632679489661923
F32 = np.float32


class Rng:
    """boost::mt19937(seed) + uniform_int<>(0, INT_MAX): rnd = raw >> 1 (bucket size 2, never rejects).  numpy's
    legacy RandomState seeded with an integer is init_genrand(seed), the same raw stream."""

    def __init__(self, seed):
        self._rs = np.random.RandomState(seed & 0xFFFFFFFF)
        self._buf = np.zeros(0, np.uint32)
        self._pos = 0
        self.used = 0

    def rnd(self):
        if self._pos == len(self._buf):
            self._buf = self._rs.randint(0, 2 ** 32, size=4096, dtype=np.uint64).astype(np.uint32)
            self._pos = 0
        r = int(self._buf[self._pos]) >> 1
        self._pos += 1
        self.used += 1
        return r


def collinear(p0, p1, p2):
    """isSampleGood of SampleConsensusModelPlane: bad iff (p1 - p0) / (p2 - p0) has three equal components"""
    with np.errstate(all="ignore"):
        a = (p1 - p0) / (p2 - p0)
    return bool(a[0] == a[1]) and bool(a[2] == a[1])


def compute_model(p0, p1, p2):
    """computeModelCoefficients in float32: cross product, true division by the norm, d = -(n . p0)"""
    a = p1 - p0
    b = p2 - p0
    nx = a[1] * b[2] - a[2] * b[1]
    ny = a[2] * b[0] - a[0] * b[2]
    nz = a[0] * b[1] - a[1] * b[0]
    norm = np.sqrt((nx * nx + ny * ny) + nz * nz)
    nx, ny, nz = nx / norm, ny / norm, nz / norm
    d = -((nx * p0[0] + ny * p0[1]) + nz * p0[2])
    return np.array([nx, ny, nz, d], F32)


def model_valid(co, angle, axis):
    """SampleConsensusModelPerpendicularPlane::isModelValid: the angle between the normal and the axis, folded to
    [0, pi/2], must not exceed eps (an int handed to setEpsAngle as radians); eps <= 0 or >= pi/2 never rejects"""
    eps = float(angle)
    if not eps > 0.0 or eps >= HALF_PI:
        return True
    nx, ny, nz = float(co[0]), float(co[1]), float(co[2])
    ax, ay, az = (float(v) for v in np.asarray(axis, F32))
    dot = (nx * ax + ny * ay) + nz * az
    nn = math.sqrt((nx * nx + ny * ny) + nz * nz)
    na = math.sqrt((ax * ax + ay * ay) + az * az)
    return not (abs(dot) / (nn * na) < math.cos(eps))


def within(co, pts, thr):
    """the float32 predicate |((a x + b y) + (c z + d))| < thr, per point"""
    x, y, z = pts[:, 0], pts[:, 1], pts[:, 2]
    a, b, c, d = (F32(v) for v in co)
    with np.errstate(invalid="ignore", over="ignore"):
        return np.abs((a * x + b * y) + (c * z + d)) < F32(thr)


def segment_once(p, pts):
    """one SACSegmentation::segment call on pts ([n, >=3] float32).  Returns a dict: ok, sel (index of the selected
    hypothesis in draw order), iterations, rnd_used, coeff (the RANSAC model) and inliers (its selection)."""
    pts = np.ascontiguousarray(pts[:, :3], F32)
    n = len(pts)
    out = dict(ok=False, sel=-1, iterations=0, rnd_used=0, coeff=np.zeros(4, F32), inliers=np.zeros(0, np.int64))
    if n < 3:  # getSamples: fewer points than the sample size, empty selection
        return out
    thr = F32(p.plane_segment_dist_thres)
    angle, axis = p.plane_segment_angle, list(p.plane_axis)
    rng = Rng(p.ransac_seed)
    shuf = np.arange(n, dtype=np.int64)
    max_iter = int(p.plane_max_iterations)
    max_skip = 10 * max_iter
    # math.log here, det_log in the oracle and on the device: they can differ in the last bit, which changes the
    # result only if k lies within about 1e-15 of an integer
    log_probability = math.log(1.0 - float(p.plane_probability))
    one_over_indices = 1.0 / n
    iterations, skipped, best, k = 0, 0, -2147483647, 1.0
    best_co = None
    while iterations < k and skipped < max_skip:
        good = False
        for _ in range(1000):
            for i in range(3):
                j = i + rng.rnd() % (n - i)
                shuf[i], shuf[j] = shuf[j], shuf[i]
            s = pts[shuf[:3]]
            if not collinear(s[0], s[1], s[2]):
                good = True
                break
        if not good:
            break
        if collinear(s[0], s[1], s[2]):  # computeModelCoefficients repeats the test (cannot fail after a good sample)
            skipped += 1
            continue
        co = compute_model(s[0], s[1], s[2])
        cnt = int(within(co, pts, thr).sum()) if model_valid(co, angle, axis) else 0
        if cnt > best:
            best = cnt
            best_co = co
            out["sel"] = iterations
            w = best * one_over_indices
            p_no_outliers = 1.0 - (w * w) * w
            p_no_outliers = max(DBL_EPS, p_no_outliers)
            p_no_outliers = min(1.0 - DBL_EPS, p_no_outliers)
            k = log_probability / math.log(p_no_outliers)
        iterations += 1
        if iterations > max_iter:
            break
    out["iterations"] = iterations
    out["rnd_used"] = rng.used
    if best_co is None:
        out["sel"] = -1
        return out
    out["ok"] = True
    out["coeff"] = best_co
    if model_valid(best_co, angle, axis):
        out["inliers"] = np.nonzero(within(best_co, pts, thr))[0]
    return out


def plane_loop(p, cloud):
    """od.cpp:376-399: while (size > keep * nr) { segment; break if no inliers; extract the rest in order }.
    optimize_coefficients must be 0 (the refined model is not restated).  Returns the oracle's plane() fields plus
    `segments` (every segment_once result, the breaking one included)."""
    assert not p.optimize_coefficients, "ransac_ref restates the loop without optimizeModelCoefficients"
    cloud = np.ascontiguousarray(cloud, F32)
    nr = len(cloud)
    rem = cloud
    src = np.arange(nr, dtype=np.int32)
    pass_points = np.zeros(MAX_PASSES, np.int32)
    pass_inliers = np.zeros(MAX_PASSES, np.int32)
    pass_coeff = np.zeros((MAX_PASSES, 4), F32)
    last_coeff = np.zeros(4, F32)
    last_inliers = np.zeros(0, np.int32)
    n_passes, warnings, segments = 0, 0, []
    while float(len(rem)) > float(p.plane_keep_fraction) * float(nr):
        seg = segment_once(p, rem)
        segments.append(seg)
        last_coeff = seg["coeff"]
        last_inliers = seg["inliers"].astype(np.int32)
        if len(seg["inliers"]) == 0:
            warnings |= WARN_PLANE_BREAK
            break
        if n_passes < MAX_PASSES:
            pass_points[n_passes] = len(rem)
            pass_inliers[n_passes] = len(seg["inliers"])
            pass_coeff[n_passes] = seg["coeff"]
        n_passes += 1
        keep = np.ones(len(rem), bool)
        keep[seg["inliers"]] = False
        rem, src = rem[keep], src[keep]
    return dict(remaining=rem, src=src, n_passes=n_passes, pass_points=pass_points, pass_inliers=pass_inliers,
                pass_coeff=pass_coeff, last_coeff=last_coeff, inliers=last_inliers, warnings=warnings,
                segments=segments)
