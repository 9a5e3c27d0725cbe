"""GPU: the RANSAC, SOR and VoxelGrid parameters that the default-parameter tests never set, on every plane-loop tier
(k_plane_loop<512>, <1024>, <1024, windows>), against the oracle, against the independent restatement
tests/ransac_ref.py (optimize_coefficients = 0, coefficients bit for bit) and against invariants that come from
neither: a replay of the recorded passes must rebuild the device's remaining cloud."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle_lib as O
import ransac_ref as R
from parity_util import assert_bits_equal, compare_frames, compare_plane
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi
from test_gpu_fuzz import fuzz_case
from test_oracle_kat import numpy_voxel_keys
from test_oracle_params import GRID, GRID_IDS, collinear_scene, rng_table_params, scene, tiny, with_params

pytestmark = pytest.mark.gpu

POOL = ThreadPoolExecutor(8)
# plane-stage inputs of the three tiers: <512> up to 65 536 points, <1024> up to 131 072, windows above
TIERS = {"small": 20000, "large": 100000, "windows": 200000}
# the windowed tier runs the cases that change the loop's shape the most (the others are the same code per pass)
WINDOW_CASES = {"iter0", "iter1", "iter63", "prob1e-06", "angle1_axis_x", "keep0.0", "keep1.0"}


@pytest.fixture(scope="module")
def tier_clouds():
    return {t: scene(40 + i, n) for i, (t, n) in enumerate(TIERS.items())}


def grid_clouds(tier_clouds):
    """the tiers plus, on the small tier, a 3 000-point scene on which a probability near 1 changes the result and a
    300-point scene on which 63 iterations do (the tier scenes are decided by their first hypotheses)"""
    return dict(tier_clouds, scene3k=scene(11, 3000), scene300=scene(8, 300))


@pytest.fixture(scope="module")
def tier_ops(tier_clouds):
    ops = {t: ObstacleProcessor(synth.params(2), len(c)) for t, c in tier_clouds.items()}
    ops["scene3k"] = ops["scene300"] = ops["small"]
    yield ops
    for t in TIERS:
        ops[t].close()


def plane_invariants(p, cloud, g, what):
    """checks that do not come from the oracle: replaying the recorded passes from the input (float32 predicate with
    pass_coeff[k], inliers removed in order) reproduces every pass' count and, when all passes are recorded, the
    remaining cloud and the last selection; every recorded model passes the angle test; the remaining cloud is the
    input minus the inliers, in order"""
    n_rec = min(g["n_passes"], R.MAX_PASSES)
    assert np.all(g["pass_inliers"][n_rec:] == 0) and np.all(g["pass_points"][n_rec:] == 0), what + "unrecorded passes"
    cur = cloud
    for k in range(n_rec):
        assert g["pass_points"][k] == len(cur), f"{what}pass {k}: points {g['pass_points'][k]} vs {len(cur)}"
        assert R.model_valid(g["pass_coeff"][k], p.plane_segment_angle, list(p.plane_axis)), f"{what}pass {k}: angle"
        sel = R.within(g["pass_coeff"][k], cur, p.plane_segment_dist_thres)
        assert int(sel.sum()) == g["pass_inliers"][k] > 0, f"{what}pass {k}: predicate {int(sel.sum())} vs {g['pass_inliers'][k]}"
        last = np.nonzero(sel)[0]
        cur = cur[~sel]
    if g["n_passes"] <= R.MAX_PASSES:
        assert_bits_equal(g["remaining"], cur, what + "replayed remaining cloud")
        if g["n_passes"] and not g["warnings"] & abi.WARN_PLANE_BREAK:
            assert_bits_equal(g["inliers"], last.astype(np.int32), what + "last pass' inliers")
    src = g["src"]
    assert np.all(np.diff(src) > 0) if len(src) > 1 else True, what + "remaining order"
    assert_bits_equal(g["remaining"], cloud[src], what + "remaining = input[src]")
    assert len(cloud) - len(src) >= g["pass_inliers"].sum(), what + "inliers removed"


def check_plane_case(p, clouds, ops, what):
    oracle = {t: POOL.submit(O.plane, p, c) for t, c in clouds.items()}
    ref = {t: POOL.submit(R.plane_loop, p, c) for t, c in clouds.items()} if not p.optimize_coefficients else {}
    default = {t: POOL.submit(O.plane, with_params(optimize_coefficients=p.optimize_coefficients), c)
               for t, c in clouds.items()}
    changed = False
    for t, c in clouds.items():
        ops[t].set_params(p)
        g = ops[t].segment_plane_and_extract_indices(c)
        o = oracle[t].result()
        compare_plane(g, o, f"{what} {t} vs oracle: ")
        if t in ref:
            r = ref[t].result()
            compare_plane(g, r, f"{what} {t} vs ransac_ref: ")
            assert_bits_equal(g["pass_coeff"], r["pass_coeff"], f"{what} {t} vs ransac_ref: pass_coeff")
            assert_bits_equal(g["last_coeff"], r["last_coeff"], f"{what} {t} vs ransac_ref: last_coeff")
        plane_invariants(p, c, g, f"{what} {t}: ")
        d = default[t].result()
        changed |= (o["n_passes"] != d["n_passes"] or o["warnings"] != d["warnings"]
                    or not np.array_equal(o["pass_inliers"], d["pass_inliers"])
                    or not np.array_equal(o["pass_coeff"], d["pass_coeff"]) or len(o["remaining"]) != len(d["remaining"]))
    return changed


@pytest.mark.parametrize("opt", [0, 1])
@pytest.mark.parametrize("case", GRID, ids=GRID_IDS)
def test_plane_parameter_grid(case, opt, tier_clouds, tier_ops):
    name, kw = case
    p = with_params(optimize_coefficients=opt, **kw)
    clouds = {t: c for t, c in grid_clouds(tier_clouds).items() if t != "windows" or name in WINDOW_CASES}
    changed = check_plane_case(p, clouds, tier_ops, f"{name} opt={opt}")
    if name not in ("angle-1", "angle0"):  # (eps <= 0 never rejects, like the default 20 rad)
        assert changed, f"{name} opt={opt}: the oracle gives the default-parameter result on every tier"


def test_plane_max_iterations_zero_breaks_without_a_model(tier_clouds, tier_ops):
    """PCL stops computeModel after max_skip = 10 * max_iterations skipped samples: with max_iterations = 0 no sample
    is drawn, no model is found and the loop breaks on its first pass, leaving the cloud as it was"""
    for opt in (0, 1):
        p = with_params(optimize_coefficients=opt, plane_max_iterations=0)
        for t, c in tier_clouds.items():
            tier_ops[t].set_params(p)
            g = tier_ops[t].segment_plane_and_extract_indices(c)
            assert g["n_passes"] == 0 and g["warnings"] == abi.WARN_PLANE_BREAK, (t, g["n_passes"], g["warnings"])
            assert_bits_equal(g["remaining"], c, f"{t}: remaining cloud")
            assert len(g["inliers"]) == 0 and not g["last_coeff"].any(), t


def _batch(clouds):
    cap = max(max(len(c) for c in clouds), 1)
    batch = np.zeros((len(clouds), cap, 4), np.float32)
    counts = np.array([len(c) for c in clouds], np.int32)
    for f, c in enumerate(clouds):
        batch[f, :len(c)] = c
    return batch, counts


def _plane_only(p):
    p = p.copy()
    p.enable_crop = p.enable_voxel = p.enable_sor = 0
    p.outputs = abi.OUT_ALL
    return p


def check_batch(op, p, batch, counts, what):
    res = op.process_batch(batch, counts)
    oracle = list(POOL.map(lambda f: O.process(p, batch[f, :counts[f]]), range(len(counts))))
    for f in range(len(counts)):
        compare_frames(res[f], oracle[f], p, f"{what} frame {f}: ")
    return oracle


BATCH_CASES = {
    "angle1_axis_x": dict(plane_segment_angle=1, plane_axis=(1.0, 0.0, 0.0)),
    "angle1_axis_x_opt0": dict(plane_segment_angle=1, plane_axis=(1.0, 0.0, 0.0), optimize_coefficients=0),
    "keep0": dict(plane_keep_fraction=0.0),
    "iter0": dict(plane_max_iterations=0),
    "iter1_angle1_opt0": dict(plane_max_iterations=1, plane_segment_angle=1, optimize_coefficients=0),
    "prob_hi_keep0.95": dict(plane_probability=1 - 1e-9, plane_keep_fraction=0.95),
}


@pytest.fixture(scope="module")
def batch_frames(tier_clouds):
    """one wave of every tier, an empty and a 2-point frame, and scenes that need different numbers of passes"""
    return _batch([tier_clouds["small"], tier_clouds["large"], tier_clouds["windows"], np.zeros((0, 4), np.float32),
                   tiny(2), scene(11, 3000), scene(8, 20000), collinear_scene(7, 4000), scene(12, 40000),
                   scene(13, 300)])


@pytest.mark.parametrize("case", list(BATCH_CASES), ids=list(BATCH_CASES))
def test_plane_parameters_batched(case, batch_frames):
    """max_batch = 16: two lanes of 8 frames; 10 frames = two waves"""
    p = _plane_only(with_params(**BATCH_CASES[case]))
    batch, counts = batch_frames
    with ObstacleProcessor(p, batch.shape[1], max_batch=16) as op:
        oracle = check_batch(op, p, batch, counts, case)
    passes = [o.n_plane_passes for o in oracle]
    assert len(set(passes)) >= {"iter0": 1, "prob_hi_keep0.95": 2}.get(case, 3), passes
    if case in ("angle1_axis_x", "keep0"):
        assert max(passes) > R.MAX_PASSES, passes


def test_plane_stage_reading_the_cropped_or_staged_input(batch_frames):
    """crop on with voxel and SOR off: the plane stage reads the cropped cloud, which must not be the ping-pong cloud
    its first pass writes.  Crop, voxel and SOR off: it reads the input staging, which a repeat of the stage (a wave
    whose large frames only the repeat runs) reads again after the first run's passes"""
    batch, counts = batch_frames
    pc = _plane_only(with_params())
    pc.enable_crop = 1
    pc.x_min, pc.x_max, pc.y_min, pc.y_max, pc.z_min, pc.z_max = -30.0, 30.0, -30.0, 30.0, -5.0, 10.0
    for p in (pc, _plane_only(with_params())):
        for idx in ([0], [0, 2], [0, 1, 5, 6]):
            with ObstacleProcessor(p, batch.shape[1], max_batch=len(idx)) as op:
                oracle = check_batch(op, p, batch[idx], counts[idx], f"crop={p.enable_crop} frames {idx}")
            assert min(o.n_plane_passes for o in oracle) >= 3


def test_set_params_changes_the_plane_loop(batch_frames):
    """pcop_set_params between two batched calls on a 2-lane handle: max_iterations, probability, angle and
    optimize_coefficients of the second call are the new ones"""
    batch, counts = batch_frames
    p1 = _plane_only(with_params())
    p2 = _plane_only(with_params(plane_max_iterations=3, plane_probability=0.5, plane_segment_angle=1,
                                 plane_axis=(1.0, 0.0, 0.0), optimize_coefficients=0))
    with ObstacleProcessor(p1, batch.shape[1], max_batch=16) as op:
        o1 = check_batch(op, p1, batch, counts, "first")
        op.set_params(p2)
        o2 = check_batch(op, p2, batch, counts, "second")
    assert [o.n_plane_passes for o in o1] != [o.n_plane_passes for o in o2]


def _random_plane_params(p, seed):
    rng = np.random.default_rng(5000 + seed)
    p.plane_max_iterations = int(rng.choice([0, 1, 3, 4, 5, 8, 9, 50, 63]))
    p.plane_probability = float(rng.choice([1e-6, 0.5, 0.99, 1 - 1e-9]))
    p.plane_segment_angle = int(rng.choice([-1, 0, 1, 20]))
    ax = [(0.0, 0.0, 1.0), (1.0, 0.0, 0.0), (0.0, 0.0, 2.0), (0.3, 0.4, 0.87)][int(rng.integers(4))]
    p.plane_axis = ax
    p.plane_keep_fraction = float(rng.choice([-0.5, 0.0, 0.3, 0.95, 1.0, 2.0]))
    p.ransac_seed = int(rng.choice([0, 1, 12345, 2 ** 32 - 1]))
    p.optimize_coefficients = int(rng.integers(2))
    return p


@pytest.mark.parametrize("seed", range(64))
def test_fuzz_pipeline_plane_parameters(seed):
    p, cloud = fuzz_case(seed)
    p = _random_plane_params(p, seed)
    with ObstacleProcessor(p, max(len(cloud), 1)) as op:
        g = op.process(cloud)
    o = O.process(p, cloud)
    compare_frames(g, o, p, f"seed {seed} (n={len(cloud)}, iter={p.plane_max_iterations} prob={p.plane_probability} "
                            f"angle={p.plane_segment_angle} keep={p.plane_keep_fraction} opt={p.optimize_coefficients}): ")


@pytest.mark.parametrize("n", [4000, 100000])
@pytest.mark.parametrize("frac_line", [0.5, 0.99])
def test_rng_table_exhaustion(n, frac_line):
    """the device precomputes 4096 random numbers per pass (DESIGN §5): it sets PCOP_WARN_RNG_TABLE_EXHAUSTED exactly
    when the pass needs more, and otherwise equals the oracle"""
    p = rng_table_params()
    cloud = collinear_scene(9, n, frac_line)
    with ObstacleProcessor(p, n) as op:
        g = op.segment_plane_and_extract_indices(cloud)
    ref = R.plane_loop(p, cloud)
    exhausted = max(s["rnd_used"] for s in ref["segments"]) > 4096
    assert exhausted == (frac_line > 0.9)
    assert bool(g["warnings"] & abi.WARN_RNG_TABLE_EXHAUSTED) == exhausted
    o = O.plane(p, cloud)
    if exhausted:  # the generator stops at the table's end: fewer hypotheses, the same zero counts
        g["warnings"] &= ~abi.WARN_RNG_TABLE_EXHAUSTED
    compare_plane(g, o, f"n={n} line={frac_line}: ")


# ---- VoxelGrid overflow along the path a user takes: a crop box too large for the fused crop + voxel plan ---------
def _wide_params():
    p = synth.params(1)
    p.x_min, p.x_max, p.y_min, p.y_max, p.z_min, p.z_max = -1000.0, 1000.0, -1000.0, 1000.0, -50.0, 50.0
    p.downsample_size = 0.01
    p.enable_sor = 0
    p.outputs = abi.OUT_ALL
    return p


def _survivors(seed, n, extent):
    """n points: 85 % inside the box (a floor and blobs spread over `extent` metres), 15 % outside it"""
    rng = np.random.default_rng(seed)
    m = int(n * 0.85)
    xy = rng.uniform(-extent / 2, extent / 2, (m, 2))
    z = np.where(rng.random(m) < 0.6, rng.normal(0, 0.01, m), rng.uniform(0, 2, m))
    inside = np.concatenate([xy, z[:, None]], 1)
    out = rng.uniform(-1000, 1000, (n - m, 3))
    out[:, 2] = rng.choice([-80.0, 90.0], n - m)
    pts = np.concatenate([inside, out])[rng.permutation(n)]
    return np.concatenate([pts, np.ones((n, 1))], 1).astype(np.float32)


def _check_voxel_frame(p, cloud, g, overflow, what):
    o = O.process(p, cloud)
    compare_frames(g, o, p, what)
    assert bool(g.warnings & abi.WARN_VOXEL_OVERFLOW_FALLBACK) == overflow, what + "overflow warning"
    c = cloud[g.crop_kept_idx]
    if overflow:
        assert g.n_voxel == g.n_crop
        assert_bits_equal(g.voxel_centroids, c, what + "fallback centroids = cropped points")
        assert not g.voxel_keys.any(), what + "fallback keys"
    else:
        keys, div = numpy_voxel_keys(p, c)
        assert div.prod() < 2 ** 31
        assert_bits_equal(g.voxel_keys, np.unique(keys), what + "keys vs numpy")


def test_voxel_overflow_with_a_wide_crop_box():
    """compact survivors (10 m): the grid fits; survivors over 800 m: 80 000 x 80 000 x 200 cells overflow 2^31,
    PCL's "leaf size is too small" fallback passes the cropped cloud through; single frames and one batched call whose
    waves mix both kinds over two lanes"""
    p = _wide_params()
    frames = [(_survivors(s, 30000, 10.0), False) for s in (1, 2)] + [(_survivors(s, 30000, 800.0), True) for s in (3, 4)]
    with ObstacleProcessor(p, 30000) as op:
        for f, (cloud, overflow) in enumerate(frames):
            _check_voxel_frame(p, cloud, op.process(cloud), overflow, f"single {f}: ")
    order = [0, 2, 1, 3, 2, 0, 3, 1, 2, 3, 0]
    batch, counts = _batch([frames[i][0] for i in order])
    with ObstacleProcessor(p, batch.shape[1], max_batch=16) as op:
        res = op.process_batch(batch, counts)
    for f, i in enumerate(order):
        _check_voxel_frame(p, frames[i][0], res[f], frames[i][1], f"batched {f}: ")


def test_downsample_cloud_overflow_and_non_finite():
    """pcop_voxel on an overflowing cloud (output = input, keys 0), and crop-off + voxel-on frames with a +-inf
    coordinate (the bounds are infinite: the fallback)"""
    p = _wide_params()
    cloud = _survivors(5, 20000, 800.0)
    cloud = cloud[(np.abs(cloud[:, 2]) < 50)]
    with ObstacleProcessor(p, len(cloud)) as op:
        g_pts, g_keys, g_w = op.downsample_cloud(cloud)
    o_pts, o_keys, o_w = O.voxel(p, cloud)
    assert g_w == o_w and g_w & abi.WARN_VOXEL_OVERFLOW_FALLBACK
    assert_bits_equal(g_keys, o_keys, "keys")
    assert_bits_equal(g_pts, o_pts, "centroids")
    assert_bits_equal(g_pts, cloud, "centroids = input")
    p2 = synth.params(1)
    p2.enable_crop = 0
    p2.enable_sor = 0
    p2.outputs = abi.OUT_ALL
    clouds = []
    for k, v in enumerate((np.inf, -np.inf)):
        c = _survivors(6 + k, 5000, 10.0)
        c[100 + k, k] = v
        clouds.append(c)
    with ObstacleProcessor(p2, 5000) as op:
        for k, c in enumerate(clouds):
            compare_frames(op.process(c), O.process(p2, c), p2, f"inf {k}: ")
    batch, counts = _batch(clouds)
    with ObstacleProcessor(p2, 5000, max_batch=2) as op:
        res = op.process_batch(batch, counts)
    for k, c in enumerate(clouds):
        compare_frames(res[k], O.process(p2, c), p2, f"inf batched {k}: ")


# ---- StatisticalOutlierRemoval edges ------------------------------------------------------------------------------
def _sor_cloud():
    p = synth.params(1)
    cloud, _ = O.crop(p, synth.frame(1, 0))
    cloud, _, _ = O.voxel(p, cloud)
    return cloud[:5000].copy()


@pytest.mark.parametrize("std", [0.0, -0.5])
def test_stage_sor_zero_and_negative_multiplier(std):
    p = synth.params(1)
    p.statistical_outlier_stdDevThres = std
    cloud = _sor_cloud()
    with ObstacleProcessor(p, len(cloud)) as op:
        g_pts, g_idx, g_w = op.remove_statistical_outliers(cloud)
    o_pts, o_idx, o_w, _, _ = O.sor(p, cloud)
    assert g_w == o_w
    assert_bits_equal(g_idx, o_idx, "sor kept_idx")
    assert_bits_equal(g_pts, o_pts, "sor points")
    assert 0 < len(o_idx) < len(cloud)


@pytest.mark.parametrize("mean_k", [8, 31])
def test_sor_both_knn_kernels(mean_k):
    """one cloud as a single frame (B * grid_cap <= 32768: the warp-per-point k-NN kernel) and as 8 copies in one
    batch (above 32768: the serial kernel); both keep the oracle's indices"""
    p = synth.params(1)
    p.enable_crop = p.enable_voxel = p.enable_plane = 0
    p.enable_sor = 1
    p.statistical_outlier_meanK = mean_k
    p.outputs = abi.OUT_ALL
    cloud = _sor_cloud()
    o = O.process(p, cloud)
    with ObstacleProcessor(p, len(cloud)) as op:
        compare_frames(op.process(cloud), o, p, "single: ")
    batch, counts = _batch([cloud] * 8)
    with ObstacleProcessor(p, len(cloud), max_batch=8) as op:
        res = op.process_batch(batch, counts)
    for f in range(8):
        compare_frames(res[f], o, p, f"batched {f}: ")
    assert o.n_sor < len(cloud)
