"""CPU: the oracle's RANSAC plane loop at the parameters the defaults never reach, against the independent numpy
restatement tests/ransac_ref.py.  With optimize_coefficients = 0 the two agree bit for bit (coefficients, inlier
indices, iterations, pass counts, warnings); with optimize_coefficients = 1 the oracle's refined models are checked
by invariants: each pass removes exactly the points the float32 predicate selects with the reported coefficients, and
a refined normal is the smallest-eigenvalue eigenvector of the RANSAC inliers' covariance."""
import math

import numpy as np
import pytest

import oracle_lib as O
import ransac_ref as R
from pointcloud_obstacle_processing_b200 import synth

F32 = np.float32
RAMP_DEG = 29.0


def scene(seed, n, noise=0.01):
    """floor z = 0, two walls (x = 8, y = -12), a 29 degree ramp and clutter; shuffled, [n, 4] float32"""
    rng = np.random.default_rng(seed)
    m = [int(n * f) for f in (0.42, 0.2, 0.1, 0.14)]
    floor = np.stack([rng.uniform(-20, 20, m[0]), rng.uniform(-20, 20, m[0]), rng.normal(0, noise, m[0])], 1)
    wall_x = np.stack([8 + rng.normal(0, noise, m[1]), rng.uniform(-20, 20, m[1]), rng.uniform(0, 4, m[1])], 1)
    wall_y = np.stack([rng.uniform(-20, 20, m[2]), -12 + rng.normal(0, noise, m[2]), rng.uniform(0, 3, m[2])], 1)
    t = math.radians(RAMP_DEG)
    u = rng.uniform(0, 8, m[3])
    ramp = np.stack([-15 + u * math.cos(t), rng.uniform(0, 10, m[3]), u * math.sin(t)], 1)
    ramp += rng.normal(0, noise, (m[3], 1)) * np.array([-math.sin(t), 0, math.cos(t)])
    rest = n - sum(m)
    clutter = np.stack([rng.uniform(-20, 20, rest), rng.uniform(-20, 20, rest), rng.uniform(0, 3, rest)], 1)
    pts = np.concatenate([floor, wall_x, wall_y, ramp, clutter])[rng.permutation(n)]
    return np.concatenate([pts, np.ones((n, 1))], 1).astype(F32)


def collinear_scene(seed, n, frac_line=0.9):
    """mostly exactly collinear points ((p1-p0)/(p2-p0) has equal components): samples are redrawn, many times"""
    rng = np.random.default_rng(seed)
    n_line = int(n * frac_line)
    t = rng.integers(-2000, 2000, n_line).astype(F32) / F32(64.0)
    rest = np.concatenate([rng.uniform(-30, 30, size=(n - n_line, 2)), rng.normal(size=(n - n_line, 1)) * 0.05], 1)
    pts = np.concatenate([np.stack([t, t, t], 1), rest])[rng.permutation(n)]
    return np.concatenate([pts, np.ones((n, 1))], 1).astype(F32)


def tiny(n, seed=3):
    rng = np.random.default_rng(seed)
    return np.concatenate([rng.uniform(-5, 5, (n, 3)), np.ones((n, 1))], 1).astype(F32)


def base_params():
    return synth.params(2)


def with_params(**kw):
    p = base_params()
    for k, v in kw.items():
        setattr(p, k, v)
    return p


# One value at a time from the config-2 parameters, then the combinations that change the loop the most.
# (name, overrides); optimize_coefficients is set by the tests.
GRID = (
    [(f"iter{v}", dict(plane_max_iterations=v)) for v in (0, 1, 3, 4, 5, 8, 9, 63)]
    + [(f"prob{v}", dict(plane_probability=v)) for v in (1e-6, 0.5, 1 - 1e-9)]
    + [(f"angle{v}", dict(plane_segment_angle=v)) for v in (-1, 0, 1)]
    + [("angle1_axis_x", dict(plane_segment_angle=1, plane_axis=(1.0, 0.0, 0.0))),
       ("angle1_axis_z2", dict(plane_segment_angle=1, plane_axis=(0.0, 0.0, 2.0))),
       ("angle1_axis_xy", dict(plane_segment_angle=1, plane_axis=(0.6, -0.8, 0.0)))]
    + [(f"keep{v}", dict(plane_keep_fraction=v)) for v in (-0.5, 0.0, 0.95, 1.0, 2.0)]
    + [(f"seed{v}", dict(ransac_seed=v)) for v in (0, 1, 2 ** 32 - 1)]
    + [("iter63_prob_hi", dict(plane_max_iterations=63, plane_probability=1 - 1e-9)),
       ("iter1_angle1", dict(plane_max_iterations=1, plane_segment_angle=1)),
       ("keep0_angle1_axis_x", dict(plane_keep_fraction=0.0, plane_segment_angle=1, plane_axis=(1.0, 0.0, 0.0)))]
)
GRID_IDS = [g[0] for g in GRID]


def rng_table_params():
    """a zero threshold keeps every count at 0, so the adaptive k never stops the loop before max_iterations: on a
    cloud that is 99 % one line, 64 good samples take about 6 400 random numbers"""
    return with_params(optimize_coefficients=0, plane_max_iterations=63, plane_segment_dist_thres=0.0)


def clouds():
    """the clouds every grid case runs on: a 20 000-point and a 3 000-point scene, a collinear-heavy cloud, 300
    points, 3 points and 2 points"""
    return {"scene20k": scene(8, 20000), "scene3k": scene(11, 3000), "collinear": collinear_scene(7, 4000),
            "scene300": scene(8, 300), "three": tiny(3), "two": tiny(2)}


_CLOUDS = None


def cloud_set():
    global _CLOUDS
    if _CLOUDS is None:
        _CLOUDS = clouds()
    return _CLOUDS


def assert_plane_equal(a, b, what):
    """two plane() results bit for bit: pass counts, recorded passes, last selection, remaining cloud, warnings"""
    assert a["n_passes"] == b["n_passes"], f"{what}: n_passes {a['n_passes']} vs {b['n_passes']}"
    assert a["warnings"] == b["warnings"], f"{what}: warnings {a['warnings']} vs {b['warnings']}"
    for k in ("pass_points", "pass_inliers"):
        assert np.array_equal(a[k], b[k]), f"{what}: {k} {a[k]} vs {b[k]}"
    for k in ("pass_coeff", "last_coeff", "remaining"):
        x, y = np.asarray(a[k], F32), np.asarray(b[k], F32)
        assert x.shape == y.shape and np.array_equal(x.view(np.uint32), y.view(np.uint32)), f"{what}: {k} differ"
    assert np.array_equal(a["src"], b["src"]), f"{what}: remaining src idx"
    assert np.array_equal(a["inliers"], b["inliers"]), f"{what}: last inliers"


def pass_inputs(cloud, result, p):
    """the input of every pass of a plane() result, rebuilt from the recorded coefficients: apply the float32
    predicate with pass_coeff[k] and remove what it selects, order kept"""
    cur, out = cloud, []
    for k in range(min(result["n_passes"], R.MAX_PASSES)):
        out.append(cur)
        sel = R.within(result["pass_coeff"][k], cur, p.plane_segment_dist_thres)
        assert int(sel.sum()) == result["pass_inliers"][k], f"pass {k}: predicate selects {int(sel.sum())}"
        cur = cur[~sel]
    return out, cur


@pytest.mark.parametrize("case", GRID, ids=GRID_IDS)
def test_oracle_plane_matches_restatement(case):
    name, kw = case
    p = with_params(optimize_coefficients=0, **kw)
    for cname, cloud in cloud_set().items():
        what = f"{name} / {cname}"
        ref = R.plane_loop(p, cloud)
        o = O.plane(p, cloud)
        assert_plane_equal(o, ref, what)
        # every pass, the breaking one included: iterations, model and inlier count of segment_once
        cur = cloud
        for k, seg in enumerate(ref["segments"]):
            s = O.segment_once(p, cur)
            assert s["ok"] == seg["ok"], f"{what} pass {k}: ok"
            assert s["iterations"] == seg["iterations"], f"{what} pass {k}: iterations {s['iterations']} vs {seg['iterations']}"
            assert np.array_equal(s["ransac_coeff"].view(np.uint32), seg["coeff"].view(np.uint32)), f"{what} pass {k}"
            assert s["n_ransac_inliers"] == len(seg["inliers"]), f"{what} pass {k}"
            keep = np.ones(len(cur), bool)
            keep[seg["inliers"]] = False
            cur = cur[keep]


def test_restatement_limits():
    """the cases the issue's numbers rest on: max_iterations = 0 never draws (PCL's skip limit 10 * 0), the loop
    breaks at once; keep = 0 runs until RANSAC finds no plane; a perpendicular axis that only the walls satisfy
    takes more passes than the result records"""
    c = cloud_set()["scene20k"]
    r = R.plane_loop(with_params(optimize_coefficients=0, plane_max_iterations=0), c)
    assert r["n_passes"] == 0 and r["warnings"] == R.WARN_PLANE_BREAK
    assert r["segments"][0]["iterations"] == 0 and r["segments"][0]["rnd_used"] == 0
    r = R.plane_loop(with_params(optimize_coefficients=0, plane_keep_fraction=0.0), c)
    assert r["warnings"] == R.WARN_PLANE_BREAK and r["n_passes"] > R.MAX_PASSES
    r = R.plane_loop(with_params(optimize_coefficients=0, plane_segment_angle=1, plane_axis=(1.0, 0.0, 0.0)), c)
    assert r["n_passes"] > R.MAX_PASSES
    r = R.plane_loop(rng_table_params(), collinear_scene(7, 4000, 0.99))
    assert max(s["rnd_used"] for s in r["segments"]) > 4096


def test_grid_cases_change_the_result():
    """a parameter that changes nothing on these clouds would pin nothing: every case differs from the defaults on at
    least one cloud"""
    for opt in (0, 1):
        default = {k: O.plane(with_params(optimize_coefficients=opt), c) for k, c in cloud_set().items()}
        for name, kw in GRID:
            if name.startswith("angle") and name in ("angle-1", "angle0"):
                continue  # eps <= 0 never rejects, like the default 20 rad: the same result is the expected one
            p = with_params(optimize_coefficients=opt, **kw)
            changed = False
            for k, c in cloud_set().items():
                try:
                    assert_plane_equal(O.plane(p, c), default[k], "")
                except AssertionError:
                    changed = True
                    break
            assert changed, f"{name} (optimize {opt}) gives the default result on every cloud"


def _eig_check(p, cur, seg, coeff, what):
    """coeff is the RANSAC model (refinement reverted or skipped) or the smallest-eigenvalue eigenvector of the
    RANSAC inliers' covariance"""
    if np.array_equal(coeff.view(np.uint32), seg["coeff"].view(np.uint32)):
        return
    assert R.model_valid(coeff, p.plane_segment_angle, list(p.plane_axis)), what + ": refined model fails the angle test"
    x = cur[seg["inliers"], :3].astype(np.float64)
    assert len(x) >= 4, what
    w, v = np.linalg.eigh(np.cov(x.T, bias=True))
    if (w[1] - w[0]) < 1e-6 * max(w[2], 1e-30):
        return  # eigengap too small for the normal to be determined to 1e-6
    nrm = v[:, 0] * np.sign(np.dot(v[:, 0], coeff[:3]))
    assert np.max(np.abs(nrm - coeff[:3])) <= 1e-6, f"{what}: normal {coeff[:3]} vs eigh {nrm}"


@pytest.mark.parametrize("case", GRID, ids=GRID_IDS)
def test_oracle_refined_plane_invariants(case):
    name, kw = case
    p = with_params(optimize_coefficients=1, **kw)
    for cname, cloud in cloud_set().items():
        if cname == "scene20k" and name.startswith(("keep0", "keep-")):
            continue  # (100+ passes: the 3 000-point scene covers the case)
        what = f"{name} / {cname}"
        o = O.plane(p, cloud)
        inputs, rest = pass_inputs(cloud, o, p)
        if o["n_passes"] <= R.MAX_PASSES:
            assert np.array_equal(rest.view(np.uint32), o["remaining"].view(np.uint32)), what + ": remaining cloud"
        for k, cur in enumerate(inputs):
            seg = R.segment_once(p, cur)  # the RANSAC step does not depend on optimize_coefficients
            assert seg["ok"], what
            _eig_check(p, cur, seg, o["pass_coeff"][k], f"{what} pass {k}")
