"""GPU parity: the CUDA library (through the C ABI) against the CPU oracle on identical inputs."""
import numpy as np
import pytest

import oracle_lib as O
from parity_util import assert_bits_equal, assert_close, compare_frames
from pointcloud_obstacle_processing_b200 import ObstacleProcessor, synth
from pointcloud_obstacle_processing_b200 import _ctypes_abi as abi

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["fused", "generic"])
def ece_path(request, monkeypatch):
    """Euclidean clustering has two device paths: the fused shared-memory kernel for small clouds and the generic
    multi-kernel path.  PCOP_ECE_SMALL_MAX=0 forces the generic one (read when the handle is created)."""
    if request.param == "generic":
        monkeypatch.setenv("PCOP_ECE_SMALL_MAX", "0")
    else:
        monkeypatch.delenv("PCOP_ECE_SMALL_MAX", raising=False)
    return request.param


@pytest.fixture(params=["voxpart", "voxlsd", "voxgeneric"])
def vox_path(request, monkeypatch):
    """crop + VoxelGrid has two fused fast paths (keys relative to the crop box: the partition path and the LSD-sort
    path it falls back to) and the generic two-stage path; PCOP_VOXEL_FUSED=lsd / =0 (read when the handle is created)
    force the second / third."""
    if request.param == "voxgeneric":
        monkeypatch.setenv("PCOP_VOXEL_FUSED", "0")
    elif request.param == "voxlsd":
        monkeypatch.setenv("PCOP_VOXEL_FUSED", "lsd")
    else:
        monkeypatch.delenv("PCOP_VOXEL_FUSED", raising=False)
    return request.param


def all_outputs(p):
    p = p.copy()
    p.outputs = abi.OUT_ALL
    return p


@pytest.fixture(scope="module")
def frames():
    return {c: synth.frame(c, 0) for c in (1, 2, 3)}


@pytest.mark.parametrize("config", [1, 2, 3])
def test_stage_crop(config, frames):
    p = synth.params(config)
    cloud = frames[config]
    with ObstacleProcessor(p, len(cloud)) as op:
        g_pts, g_idx = op.crop(cloud)
    o_pts, o_idx = O.crop(p, cloud)
    assert_bits_equal(g_idx, o_idx, "kept_idx")
    assert_bits_equal(g_pts, o_pts, "cropped points")


@pytest.mark.parametrize("config", [1, 2, 3])
def test_stage_voxel(config, frames):
    p = synth.params(config)
    cloud, _ = O.crop(p, frames[config])
    with ObstacleProcessor(p, len(cloud)) as op:
        g_pts, g_keys, g_w = op.downsample_cloud(cloud)
    o_pts, o_keys, o_w = O.voxel(p, cloud)
    assert g_w == o_w
    assert_bits_equal(g_keys, o_keys, "voxel keys")
    assert_bits_equal(g_pts, o_pts, "voxel centroids")


@pytest.mark.parametrize("mean_k", [15, 1, 31, 40])  # (the warp-per-point kernel holds up to 32 neighbours; 40 takes the serial one)
def test_stage_sor(frames, mean_k):
    p = synth.params(1)
    p.statistical_outlier_meanK = mean_k
    cloud, _ = O.crop(p, frames[1])
    cloud, _, _ = O.voxel(p, cloud)
    with ObstacleProcessor(p, len(cloud)) as op:
        g_pts, g_idx, g_w = op.remove_statistical_outliers(cloud)
    o_pts, o_idx, o_w, dist, thr = O.sor(p, cloud)
    print("SOR margin min|d - thr| =", np.min(np.abs(dist.astype(np.float64) - thr)), "removed", len(cloud) - len(o_idx))
    assert g_w == o_w
    assert_bits_equal(g_idx, o_idx, "sor kept_idx")
    assert_bits_equal(g_pts, o_pts, "sor points")


def test_stage_sor_with_non_finite_points(frames):
    p = synth.params(1)
    cloud, _ = O.crop(p, frames[1])
    cloud, _, _ = O.voxel(p, cloud)
    cloud = cloud[:3000].copy()
    rng = np.random.default_rng(7)
    bad = rng.choice(len(cloud), 12, replace=False)
    cloud[bad[:4], 1] = np.nan
    cloud[bad[4:8], 2] = np.inf
    cloud[bad[8:], 0] = -np.inf
    with ObstacleProcessor(p, len(cloud)) as op:
        g_pts, g_idx, g_w = op.remove_statistical_outliers(cloud)
    o_pts, o_idx, o_w, dist, thr = O.sor(p, cloud)
    assert g_w == o_w
    assert_bits_equal(g_idx, o_idx, "sor kept_idx")
    assert_bits_equal(g_pts, o_pts, "sor points")


@pytest.mark.parametrize("config,index", [(1, 0), (2, 0), (2, 1), (3, 0), (3, 1), (4, 0)])
def test_stage_plane(config, index):
    """plane inputs of 8 684 (small tier), 56 424 and about 56 000, 129 789 (large tier), 132 404 (windows) and 999 976
    points (windows, 13 passes)"""
    p = synth.params(config)
    cloud, _ = O.crop(p, synth.frame(config, index))
    cloud, _, _ = O.voxel(p, cloud)
    with ObstacleProcessor(p, len(cloud)) as op:
        g = op.segment_plane_and_extract_indices(cloud)
    o = O.plane(p, cloud)
    assert g["n_passes"] == o["n_passes"]
    assert_bits_equal(g["pass_points"], o["pass_points"], "pass_points")
    assert_bits_equal(g["pass_inliers"], o["pass_inliers"], "pass_inliers")
    assert_close(g["pass_coeff"], o["pass_coeff"], "pass_coeff")
    assert_close(g["last_coeff"], o["last_coeff"], "last_coeff")
    assert_bits_equal(g["inliers"], o["inliers"], "last inliers")
    assert_bits_equal(g["src"], o["src"], "remaining src idx")
    assert_bits_equal(g["remaining"], o["remaining"], "remaining cloud")
    assert g["warnings"] == o["warnings"]


@pytest.mark.parametrize("config", [1, 2, 3])
def test_stage_cluster_and_centroid(config, frames, ece_path):
    p = synth.params(config)
    of = O.process(p, frames[config])
    cloud = of.remaining_cloud
    with ObstacleProcessor(p, max(len(cloud), 1)) as op:
        g_off, g_idx = op.extract_euclidian_clusters(cloud)
        g_obs = op.centroid_radius(cloud, of.cluster_offsets, of.cluster_indices)
    assert_bits_equal(g_off, of.cluster_offsets, "cluster offsets")
    assert_bits_equal(g_idx, of.cluster_indices, "cluster indices")
    assert_close(g_obs, of.obstacles, "obstacles")


@pytest.mark.parametrize("config", [1, 2])
def test_pipeline_voxel_paths(config, frames, vox_path):
    """default outputs (no cropped cloud requested: the fused path does not materialise it) and all outputs"""
    for outputs in (None, abi.OUT_ALL):
        p = synth.params(config)
        if outputs is not None:
            p.outputs = outputs
        cloud = frames[config]
        with ObstacleProcessor(p, len(cloud)) as op:
            g = op.process(cloud)
        o = O.process(p, cloud)
        compare_frames(g, o, p, f"config{config}/{vox_path}: ")


def _voxel_only(p):
    p = p.copy()
    p.enable_sor = p.enable_plane = p.enable_cluster = 0
    p.outputs = abi.OUT_CROP | abi.OUT_VOXEL
    return p


def _check_voxel(p, clouds, counts=None, max_batch=None):
    clouds = np.ascontiguousarray(clouds, np.float32)
    B = clouds.shape[0]
    counts = np.full(B, clouds.shape[1], np.int32) if counts is None else counts
    with ObstacleProcessor(p, clouds.shape[1], max_batch=max_batch or B) as op:
        res = op.process_batch(clouds, counts)
    for f in range(B):
        o = O.process(p, clouds[f, :counts[f]])
        assert res[f].n_crop == o.n_crop and res[f].n_voxel == o.n_voxel, (f, res[f].n_crop, o.n_crop, res[f].n_voxel, o.n_voxel)
        assert_bits_equal(res[f].voxel_keys, o.voxel_keys, f"frame {f} voxel keys")
        assert_bits_equal(res[f].voxel_centroids, o.voxel_centroids, f"frame {f} voxel centroids")
    return res


def test_voxel_partition_path_long_runs_and_big_buckets(vox_path):
    """voxels with far more than 8 points (ordered by the whole block), more than 64 of them in one group (the list
    overflows), and a bucket above 4096 points (the frame goes to the LSD path); centroids must stay bit-exact because
    every voxel is summed in ascending original index"""
    p = _voxel_only(synth.params(2))
    rng = np.random.default_rng(123)
    n = 40000
    frames_ = []
    # frame 0: 27 voxels x ~110 points inside a 0.3 m cube + background
    a = np.concatenate([rng.uniform(0.0, 0.3, size=(3000, 3)) + [5.0, 5.0, 0.0], rng.uniform(-30, 30, size=(n - 3000, 3)) * [1, 1, 0.03]])
    # frame 1: 125 voxels x 240 points: long runs everywhere, bucket far above 4096 points
    b = np.concatenate([rng.uniform(0.0, 0.5, size=(30000, 3)) + [-3.0, 2.0, -1.0], rng.uniform(-30, 30, size=(n - 30000, 3)) * [1, 1, 0.03]])
    # frame 2: all points in ONE voxel
    c = rng.uniform(0.01, 0.09, size=(n, 3)) + [1.0, 1.0, 0.0]
    # frame 3: ~700 voxels x 12 points in a thin slab (more than 64 long runs per group)
    d = np.concatenate([rng.uniform(0.0, 1.0, size=(9000, 3)) * [2.6, 2.6, 0.1] + [10.0, -8.0, 0.2], rng.uniform(-30, 30, size=(n - 9000, 3)) * [1, 1, 0.03]])
    for q in (a, b, c, d):
        q = q.astype(np.float32)
        frames_.append(_cloud(q[rng.permutation(n)]))
    _check_voxel(p, np.stack(frames_))


def test_voxel_partition_path_more_groups_than_the_grid_covers():
    """the reduce grid is sized from the frames seen so far; a later wave with many more groups is detected on the
    device and repeated with the worst-case grid"""
    p = _voxel_only(synth.params(2))
    rng = np.random.default_rng(124)
    n = 120000
    dense = (rng.uniform(-2, 2, size=(n, 3)) * [1, 1, 0.2]).astype(np.float32)     # few buckets, few groups
    spread = (rng.uniform(-39.9, 39.9, size=(n, 3)) * [1, 1, 0.05]).astype(np.float32)
    spread[:, 2] = rng.uniform(-2.4, 1.4, size=n)                                    # every bucket occupied
    with ObstacleProcessor(p, n, max_batch=2) as op:
        for cloud in (dense, dense, spread, spread, dense):
            c4 = _cloud(cloud)
            g = op.process(c4)
            o = O.process(p, c4)
            assert g.n_voxel == o.n_voxel
            assert_bits_equal(g.voxel_keys, o.voxel_keys, "voxel keys")
            assert_bits_equal(g.voxel_centroids, o.voxel_centroids, "voxel centroids")


def test_pipeline_survivor_with_nan_yz_redone_by_generic_path(frames):
    """the reference's crop only NaN-tests x (od.cpp:197): a survivor with NaN y or z reaches VoxelGrid; the fused
    fast path declines such a frame and the wave is redone by the generic path"""
    p = all_outputs(synth.params(2))
    n = synth.points_per_frame(2)
    clouds = synth.frames(2, 200, 3).copy()
    o_plain = O.process(p, clouds[1])
    keep = np.flatnonzero(np.isin(np.arange(n), o_plain.crop_kept_idx))
    clouds[1, keep[100], 1] = np.nan
    clouds[1, keep[5000], 2] = np.nan
    counts = np.full(3, n, np.int32)
    with ObstacleProcessor(p, n, max_batch=3) as op:
        res = op.process_batch(clouds, counts)
    for f in range(3):
        o = O.process(p, clouds[f])
        compare_frames(res[f], o, p, f"frame{f}: ")
    assert res[1].n_crop == o_plain.n_crop


@pytest.mark.parametrize("config", [1, 2, 3, 4])
def test_pipeline(config, frames, ece_path):
    p = all_outputs(synth.params(config))
    cloud = frames[config] if config in frames else synth.frame(config, 0)
    with ObstacleProcessor(p, len(cloud)) as op:
        g = op.process(cloud)
    o = O.process(p, cloud)
    compare_frames(g, o, p, f"config{config}: ")
    assert o.n_clusters > 0


@pytest.mark.parametrize("small_max", [None, 0, 4500])
def test_batch_mixed_sizes(small_max, monkeypatch):
    """frames of different sizes (ragged batch), more frames than one wave; small_max = 4500 routes the frames of one
    wave to different clustering paths"""
    if small_max is not None:
        monkeypatch.setenv("PCOP_ECE_SMALL_MAX", str(small_max))
    p = all_outputs(synth.params(2))
    n = synth.points_per_frame(2)
    B = 5
    clouds = synth.frames(2, 10, B)
    counts = np.array([n, n - 1777, 50000, 0, 3], np.int32)
    with ObstacleProcessor(p, n, max_batch=2) as op:
        res = op.process_batch(clouds, counts)
    for f in range(B):
        o = O.process(p, clouds[f, :counts[f]])
        compare_frames(res[f], o, p, f"frame{f}: ")


def _cloud(xyz):
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    return np.concatenate([xyz, np.ones((len(xyz), 1), np.float32)], axis=1)


def test_cluster_large_extent_falls_back_to_point_scan(ece_path):
    """extent / tolerance too large for 1024 clique cells per axis -> per-point neighbour scan path"""
    p = synth.params(1)
    p.euc_cluster_tolerance = 0.05
    p.euc_min_cluster_size = 2
    p.euc_max_cluster_size = 100000
    rng = np.random.default_rng(21)
    blobs = [rng.normal(size=(300, 3)) * 0.05 + c for c in ([0, 0, 0], [90, 5, 1], [-40, 70, 2], [10, -80, 0])]
    cloud = _cloud(np.concatenate(blobs))
    with ObstacleProcessor(p, len(cloud)) as op:
        g_off, g_idx = op.extract_euclidian_clusters(cloud)
    o_off, o_idx = O.cluster_bruteforce(p, cloud)
    assert_bits_equal(g_off, o_off, "offsets")
    assert_bits_equal(g_idx, o_idx, "indices")
    assert len(o_off) > 4


def test_cluster_non_finite_points_are_singletons(ece_path):
    p = synth.params(1)
    p.euc_cluster_tolerance = 0.2
    p.euc_min_cluster_size = 1
    p.euc_max_cluster_size = 100000
    rng = np.random.default_rng(22)
    pts = rng.normal(size=(500, 3)).astype(np.float32) * 0.3
    pts[7, 1] = np.nan
    pts[100, 2] = np.inf
    pts[101, 0] = -np.inf
    pts[300] = [np.nan, np.nan, np.nan]
    cloud = _cloud(pts)
    with ObstacleProcessor(p, len(cloud)) as op:
        g_off, g_idx = op.extract_euclidian_clusters(cloud)
    o_off, o_idx = O.cluster_bruteforce(p, cloud)
    assert_bits_equal(g_off, o_off, "offsets")
    assert_bits_equal(g_idx, o_idx, "indices")


@pytest.mark.parametrize("seed,tol,n", [(31, 0.05, 4000), (32, 0.11, 4000), (33, 0.3, 2500), (34, 1.0, 1500)])
def test_cluster_random_against_bruteforce(seed, tol, n, ece_path):
    p = synth.params(1)
    p.euc_cluster_tolerance = tol
    p.euc_min_cluster_size = 2
    p.euc_max_cluster_size = 100000
    rng = np.random.default_rng(seed)
    centers = rng.uniform(-3, 3, size=(15, 3))
    pts = centers[rng.integers(0, 15, n)] + rng.normal(size=(n, 3)) * 0.12
    cloud = _cloud(np.concatenate([pts, rng.uniform(-4, 4, size=(n // 8, 3))]))
    with ObstacleProcessor(p, len(cloud)) as op:
        g_off, g_idx = op.extract_euclidian_clusters(cloud)
    o_off, o_idx = O.cluster_bruteforce(p, cloud)
    assert_bits_equal(g_off, o_off, "offsets")
    assert_bits_equal(g_idx, o_idx, "indices")


def test_cluster_fused_kernel_capacity_edge(monkeypatch):
    """clouds just below / above the fused kernel's capacity take different paths and must agree with the oracle"""
    p = synth.params(1)
    p.euc_cluster_tolerance = 0.08
    p.euc_min_cluster_size = 3
    p.euc_max_cluster_size = 100000
    rng = np.random.default_rng(41)
    for n in (8960, 8961):
        centers = rng.uniform(-5, 5, size=(40, 3))
        pts = centers[rng.integers(0, 40, n)] + rng.normal(size=(n, 3)) * 0.15
        cloud = _cloud(pts)
        with ObstacleProcessor(p, len(cloud)) as op:
            g_off, g_idx = op.extract_euclidian_clusters(cloud)
            g_obs = op.centroid_radius(cloud, g_off, g_idx)
        o_off, o_idx = O.cluster_bruteforce(p, cloud)
        assert_bits_equal(g_off, o_off, "offsets")
        assert_bits_equal(g_idx, o_idx, "indices")
        assert len(o_off) > 10


def test_cluster_drops_oversize_and_undersize(ece_path):
    """components outside [min, max] are dropped whole (SURVEY 8a-6.3); ties in size are ordered by smallest index"""
    p = synth.params(1)
    p.euc_cluster_tolerance = 0.1
    p.euc_min_cluster_size = 10
    p.euc_max_cluster_size = 200
    rng = np.random.default_rng(42)
    sizes = [500, 200, 200, 199, 10, 10, 9, 1, 1]
    blobs = [rng.uniform(-0.2, 0.2, size=(s, 3)) * [1, 1, 0.2] + [3.0 * k, 0, 0] for k, s in enumerate(sizes)]
    pts = np.concatenate(blobs)
    pts = pts[rng.permutation(len(pts))]
    cloud = _cloud(pts)
    with ObstacleProcessor(p, len(cloud)) as op:
        g_off, g_idx = op.extract_euclidian_clusters(cloud)
    o_off, o_idx = O.cluster_bruteforce(p, cloud)
    assert_bits_equal(g_off, o_off, "offsets")
    assert_bits_equal(g_idx, o_idx, "indices")


@pytest.mark.parametrize("n_groups,per_group", [(40, 20), (300, 12), (1500, 4)])
def test_cluster_many_small_clusters(n_groups, per_group, ece_path):
    """cluster counts on both sides of the fused kernel's thresholds (member listing by warp scans up to 128
    clusters, root ranking by counting up to 1024 clusters, bitonic sorts beyond)"""
    p = synth.params(1)
    p.euc_cluster_tolerance = 0.05
    p.euc_min_cluster_size = 2
    p.euc_max_cluster_size = 100000
    rng = np.random.default_rng(50 + n_groups)
    side = int(np.ceil(np.sqrt(n_groups)))
    centers = np.array([[0.5 * (g % side), 0.5 * (g // side), 0.0] for g in range(n_groups)])
    sizes = rng.integers(max(per_group - 3, 1), per_group + 4, n_groups)
    pts = np.concatenate([centers[g] + rng.uniform(-0.02, 0.02, size=(sizes[g], 3)) for g in range(n_groups)])
    pts = pts[rng.permutation(len(pts))]
    cloud = _cloud(pts)
    with ObstacleProcessor(p, len(cloud)) as op:
        g_off, g_idx = op.extract_euclidian_clusters(cloud)
        g_obs = op.centroid_radius(cloud, g_off, g_idx)
    o_off, o_idx = O.cluster_bruteforce(p, cloud)
    assert_bits_equal(g_off, o_off, "offsets")
    assert_bits_equal(g_idx, o_idx, "indices")
    assert_close(g_obs, O.centroid_radius(cloud, o_off, o_idx), "obstacles")
    assert len(o_off) - 1 >= n_groups * 0.8


def test_batch_over_two_lanes():
    """max_batch = 16 gives two lanes of 8 frames; 20 frames = three waves dealt round-robin to the lanes
    (one host thread and stream per lane)"""
    p = all_outputs(synth.params(2))
    n = synth.points_per_frame(2)
    B = 20
    clouds = synth.frames(2, 100, B)
    counts = np.full(B, n, np.int32)
    counts[3] = 70000
    counts[17] = 0
    with ObstacleProcessor(p, n, max_batch=16) as op:
        for _ in range(2):  # second call reuses the lanes' buffers
            res = op.process_batch(clouds, counts)
    for f in range(B):
        o = O.process(p, clouds[f, :counts[f]])
        compare_frames(res[f], o, p, f"frame{f}: ")


def _compare_plane(p, cloud):
    with ObstacleProcessor(p, len(cloud)) as op:
        g = op.segment_plane_and_extract_indices(cloud)
    o = O.plane(p, cloud)
    assert g["n_passes"] == o["n_passes"]
    assert_bits_equal(g["pass_points"], o["pass_points"], "pass_points")
    assert_bits_equal(g["pass_inliers"], o["pass_inliers"], "pass_inliers")
    assert_close(g["pass_coeff"], o["pass_coeff"], "pass_coeff")
    assert_bits_equal(g["inliers"], o["inliers"], "last inliers")
    assert_bits_equal(g["src"], o["src"], "remaining src idx")
    assert_bits_equal(g["remaining"], o["remaining"], "remaining cloud")
    assert g["warnings"] == o["warnings"]
    return o


def _planes_cloud(rng, n, fracs, noise=0.01):
    """planes of decreasing size (fractions of n) plus uniform clutter: the loop of od.cpp:379 needs one pass per plane
    until at most 30 % of the cloud is left"""
    parts = []
    for k, fr in enumerate(fracs):
        m = int(n * fr)
        uv = rng.uniform(-20, 20, size=(m, 2))
        nrm = rng.normal(size=3)
        nrm /= np.linalg.norm(nrm)
        e1 = np.cross(nrm, [1.0, 0.3, 0.2])
        e1 /= np.linalg.norm(e1)
        e2 = np.cross(nrm, e1)
        parts.append(uv[:, :1] * e1 + uv[:, 1:] * e2 + nrm * (3.0 * k) + rng.normal(size=(m, 1)) * noise * nrm)
    rest = n - sum(len(q) for q in parts)
    parts.append(rng.uniform(-25, 25, size=(rest, 3)))
    pts = np.concatenate(parts).astype(np.float32)
    return pts[rng.permutation(len(pts))]


@pytest.mark.parametrize("n,fracs", [(30000, (0.35, 0.25, 0.15, 0.1)), (9000, (0.3, 0.2, 0.12, 0.1, 0.08)),
                                     (100000, (0.4, 0.2, 0.15)), (66000, (0.35, 0.25, 0.15, 0.1)),
                                     (150000, (0.4, 0.25, 0.15)), (1000000, (0.4, 0.2, 0.15))])
def test_plane_multi_pass(n, fracs):
    """several passes inside one launch: the second and later passes generate their hypotheses in the kernel and
    reload the cloud that the previous pass wrote (66 000 points: the large tier from the first pass on; 150 000 and
    1 000 000: windows in the first passes)"""
    p = synth.params(2)
    rng = np.random.default_rng(77 + n)
    o = _compare_plane(p, _cloud(_planes_cloud(rng, n, fracs)))
    assert o["n_passes"] >= 3, o["n_passes"]


def _collinear_cloud(rng, n, frac_line):
    """a share of exactly collinear points ((p1-p0)/(p2-p0) has equal components) in a flat clutter: samples drawn from
    the line fail isSampleGood and are redrawn"""
    n_line = int(n * frac_line)
    t = rng.integers(-2000, 2000, n_line).astype(np.float32) / 64.0
    line = np.stack([t, t, t], axis=1)
    rest = np.concatenate([rng.uniform(-30, 30, size=(n - n_line, 2)), rng.normal(size=(n - n_line, 1)) * 0.05], axis=1)
    pts = np.concatenate([line, rest]).astype(np.float32)
    return pts[rng.permutation(n)]


@pytest.mark.parametrize("case", ["n131073", "n150000", "n300000", "collinear", "no_plane"])
def test_plane_large_frames_in_windows(case):
    """frames above 8 x 16384 points: each CTA of the large tier walks its part of the frame in windows of its slice.
    131073 points: CTAs 0-6 own 18432 points (a full window and a 2048-point one), CTA 7 owns 2049 in one window;
    300000 points: later passes reload windows that other CTAs wrote in the same launch; redraws of collinear samples;
    a cloud whose RANSAC finds no plane (the loop breaks on its first pass)"""
    p = synth.params(2)
    rng = np.random.default_rng(5)
    if case == "n131073":
        pts, min_passes = _planes_cloud(rng, 131073, (0.45, 0.3)), 2
    elif case == "n150000":
        pts, min_passes = _planes_cloud(rng, 150000, (0.45, 0.3)), 2
    elif case == "n300000":
        pts, min_passes = _planes_cloud(rng, 300000, (0.4, 0.2, 0.15)), 3
    elif case == "collinear":
        pts, min_passes = _collinear_cloud(rng, 140000, 0.5), 0
    else:  # a zero threshold: no point is closer than 0 to any plane, the loop breaks on its first pass
        p.plane_segment_dist_thres = 0.0
        pts, min_passes = rng.uniform(-50, 50, size=(140000, 3)).astype(np.float32), 0
    o = _compare_plane(p, _cloud(pts))
    assert o["n_passes"] >= min_passes, o["n_passes"]
    if case == "no_plane":
        assert o["n_passes"] == 0 and o["warnings"] & abi.WARN_PLANE_BREAK, o


def test_plane_batch_with_large_and_windowed_frames():
    """one wave through pcop_process_batch: a small-tier frame, a large-tier frame in one window per CTA, a frame in
    several windows, an empty frame, and frames that need different numbers of passes"""
    p = all_outputs(synth.params(2))
    p.enable_crop = 0
    p.enable_voxel = 0
    rng = np.random.default_rng(23)
    clouds = [_planes_cloud(rng, 20000, (0.8,)), _planes_cloud(rng, 100000, (0.35, 0.3, 0.2)),
              _planes_cloud(rng, 200000, (0.4, 0.25, 0.15)), np.zeros((0, 3), np.float32),
              _planes_cloud(rng, 150000, (0.5, 0.25))]
    cap = max(len(c) for c in clouds)
    batch = np.zeros((len(clouds), cap, 4), np.float32)
    counts = np.array([len(c) for c in clouds], np.int32)
    for f, c in enumerate(clouds):
        batch[f, :len(c), :3] = c
        batch[f, :len(c), 3] = 1.0
    with ObstacleProcessor(p, cap, max_batch=len(clouds)) as op:
        res = op.process_batch(batch, counts)
    passes = []
    for f in range(len(clouds)):
        o = O.process(p, batch[f, :counts[f]])
        compare_frames(res[f], o, p, f"frame{f}: ")
        passes.append(o.n_plane_passes)
    assert len(set(passes)) >= 3, passes


def test_plane_batch_frames_with_different_pass_counts():
    """frames of one wave leave the loop after different numbers of passes (each cluster runs its own loop); also
    empty and tiny frames, and a frame whose RANSAC finds no plane"""
    p = all_outputs(synth.params(2))
    p.enable_crop = 0
    p.enable_voxel = 0
    rng = np.random.default_rng(11)
    clouds = [_planes_cloud(rng, 20000, (0.8,)), _planes_cloud(rng, 20000, (0.35, 0.3, 0.2)),
              _planes_cloud(rng, 15000, (0.3, 0.2, 0.15, 0.1)), np.zeros((0, 3), np.float32),
              rng.uniform(-5, 5, size=(2, 3)).astype(np.float32), _planes_cloud(rng, 20000, (0.5, 0.25)),
              np.repeat(rng.uniform(-5, 5, size=(1, 3)), 50, axis=0).astype(np.float32)]
    cap = max(len(c) for c in clouds)
    batch = np.zeros((len(clouds), cap, 4), np.float32)
    counts = np.array([len(c) for c in clouds], np.int32)
    for f, c in enumerate(clouds):
        batch[f, :len(c), :3] = c
        batch[f, :len(c), 3] = 1.0
    with ObstacleProcessor(p, cap, max_batch=len(clouds)) as op:
        res = op.process_batch(batch, counts)
    passes = []
    for f in range(len(clouds)):
        o = O.process(p, batch[f, :counts[f]])
        compare_frames(res[f], o, p, f"frame{f}: ")
        passes.append(o.n_plane_passes)
    assert len(set(passes)) >= 3, passes


@pytest.mark.parametrize("n", [6000, 100000])
@pytest.mark.parametrize("frac_line", [0.5, 0.9, 1.0])
def test_plane_collinear_samples_redrawn(frac_line, n):
    """samples that fail isSampleGood are redrawn (consuming random numbers): the hypothesis generator's parallel
    fast path must hand such frames to the sequential replay; an all-collinear cloud exhausts the 1000 redraws.
    6 000 points: small tier; 100 000: large tier, where later passes generate in the kernel from the cloud it wrote"""
    p = synth.params(2)
    rng = np.random.default_rng(61)
    pts = _collinear_cloud(rng, n, frac_line)
    o = _compare_plane(p, _cloud(pts))
    print("passes", o["n_passes"], "warnings", o["warnings"])


def _rigid(yaw, pitch, roll, t):
    cy, sy, cp, sp, cr, sr = np.cos(yaw), np.sin(yaw), np.cos(pitch), np.sin(pitch), np.cos(roll), np.sin(roll)
    R = np.array([[cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr],
                  [sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr],
                  [-sp, cp * sr, cp * cr]])
    m = np.eye(4)
    m[:3, :3] = R
    m[:3, 3] = t
    return m.astype(np.float32)


@pytest.mark.parametrize("is_dense", [False, True])
def test_transform_stage(is_dense, frames):
    """od.cpp:696 pcl_ros::transformPointCloud: bit-exact against the oracle, NaN holes included"""
    cloud = frames[3][:50000].copy()  # depth-camera frame: 10 % NaN pixels
    m = _rigid(0.7, -0.15, 0.05, [0.4, -2.0, 1.3])
    with ObstacleProcessor(synth.params(3), len(cloud)) as op:
        g = op.transform(cloud, m, is_dense=is_dense)
    assert_bits_equal(g, O.transform(cloud, m, is_dense=is_dense), "transformed cloud")


def test_accumulate_then_process_matches_oracle_on_concatenated_world_cloud():
    """od.cpp:691-701: accumulate_count clouds are transformed into the world frame and concatenated, the next callback
    runs the pipeline on the concatenation and empties the accumulator"""
    p = all_outputs(synth.params(1))
    base = synth.frame(1, 0)
    rng = np.random.default_rng(7)
    parts, mats = [], []
    for k in range(4):  # four sensor poses looking at the same arena: world cloud = T_k^-1 applied ... here simply T_k
        m = _rigid(0.02 * k, 0.01 * k, -0.015 * k, [0.01 * k, -0.02 * k, 0.005 * k])
        sub = base[rng.permutation(len(base))[:7000]]
        parts.append(sub)
        mats.append(m)
    world = np.concatenate([O.transform(c, m, is_dense=False) for c, m in zip(parts, mats)])
    with ObstacleProcessor(p, len(world)) as op:
        for c, m in zip(parts, mats):
            total = op.accumulate(c, m, is_dense=False)
        assert total == len(world) == op.accumulated_count
        g = op.process_accumulated()
        assert op.accumulated_count == 0
        with pytest.raises(Exception):
            op.accumulate(np.zeros((len(world) + 1, 4), np.float32))  # capacity
    o = O.process(p, world)
    compare_frames(g, o, p, "accumulated: ")
    assert o.n_clusters > 0


def _make_pointcloud2(xyz, point_step, offs, seed=3):
    n = len(xyz)
    rng = np.random.default_rng(seed)
    buf = rng.integers(0, 256, size=(n, point_step), dtype=np.uint8)
    for a, off in enumerate(offs):
        buf[:, off:off + 4] = np.ascontiguousarray(xyz[:, a], np.float32).view(np.uint8).reshape(n, 4)
    return buf.reshape(-1)


@pytest.mark.parametrize("point_step,offs", [(16, (0, 4, 8)), (32, (0, 4, 8)), (22, (1, 9, 14))])
def test_pointcloud2_ingest(point_step, offs, frames):
    """od.cpp:688-689 (wire decode) and the fused decode + transform + append (od.cpp:688-697) against the oracle"""
    cloud = frames[3][:60000]
    buf = _make_pointcloud2(cloud[:, :3], point_step, offs)
    m = _rigid(-0.4, 0.2, 0.1, [1.0, 0.5, -0.25])
    with ObstacleProcessor(synth.params(3), 2 * len(cloud)) as op:
        g = op.pointcloud2_to_xyz(buf, len(cloud), point_step, *offs)
        o = O.pointcloud2_to_xyz(buf, len(cloud), point_step, *offs)
        assert_bits_equal(g, o, "decoded cloud")
        # fused ingest twice (two callbacks), then the accumulated cloud must be the two transformed clouds in order
        op.accumulate_pointcloud2(buf, len(cloud), point_step, *offs, transform=m, is_dense=False)
        total = op.accumulate_pointcloud2(buf, len(cloud), point_step, *offs, transform=None, is_dense=False)
        assert total == 2 * len(cloud)
        p = all_outputs(synth.params(3))
        p.enable_crop = p.enable_voxel = p.enable_sor = p.enable_plane = p.enable_cluster = 0
        p.outputs = abi.OUT_REMAINING
        op.set_params(p)
        acc = op.process_accumulated().remaining_cloud
    want = np.concatenate([O.transform(o, m, is_dense=False), o])
    assert_bits_equal(acc, want, "accumulated cloud")


@pytest.mark.parametrize("config", [1, 2])
def test_occupancy_grid(config, frames):
    """od.cpp:175-269 (the occupancy grid's initial data set): counts, row averages and cells, bit-exact"""
    p = synth.params(config)
    if config == 2:
        p.block_size = 0.5
    cloud = frames[config]
    with ObstacleProcessor(p, len(cloud)) as op:
        g_grid, g_counts, g_avg = op.occupancy_grid(cloud)
        op.accumulate(cloud[:len(cloud) // 2])
        op.accumulate(cloud[len(cloud) // 2:])
        a_grid, a_counts, a_avg = op.occupancy_grid(None)  # the accumulated cloud
    o_grid, o_counts, o_avg = O.occupancy_grid(p, cloud)
    for g, o, what in ((g_counts, o_counts, "counts"), (g_avg, o_avg, "row averages"), (g_grid, o_grid, "cells"),
                       (a_counts, o_counts, "counts (accumulated)"), (a_grid, o_grid, "cells (accumulated)")):
        assert_bits_equal(g, o, what)
    assert o_counts.sum() > 1000 and (o_grid == 100).any() and (o_grid == 0).any()


def test_device_resident_results_match_host_results():
    """outputs | OUT_DEVICE: the result pointers are device pointers (for a consumer on the GPU); downloaded, every
    array equals the host-result run; 20 frames on two lanes"""
    p = synth.params(2)
    p.outputs = abi.OUT_ALL
    pd = p.copy()
    pd.outputs = abi.OUT_ALL | abi.OUT_DEVICE
    n = synth.points_per_frame(2)
    B = 20
    clouds = synth.frames(2, 300, B)
    counts = np.full(B, n, np.int32)
    with ObstacleProcessor(p, n, max_batch=16) as op:
        host = op.process_batch(clouds, counts)
    with ObstacleProcessor(pd, n, max_batch=16) as op:
        res = op.process_batch_raw(clouds.ctypes.data, n, counts)
        for f in range(B):
            r, hf = res[f], host[f]
            assert r.n_clusters == hf.n_clusters and r.n_remaining == hf.n_remaining and r.n_voxel == hf.n_voxel
            assert_bits_equal(op.download(r.remaining_cloud, r.n_remaining * 4, np.float32).reshape(-1, 4), hf.remaining_cloud, "remaining")
            assert_bits_equal(op.download(r.remaining_src_idx, r.n_remaining, np.int32), hf.remaining_src_idx, "remaining src")
            assert_bits_equal(op.download(r.cluster_offsets, r.n_clusters + 1, np.int32), hf.cluster_offsets, "offsets")
            assert_bits_equal(op.download(r.cluster_indices, r.n_cluster_points, np.int32), hf.cluster_indices, "indices")
            assert_bits_equal(op.download(r.obstacles, r.n_clusters * 4, np.float32).reshape(-1, 4), hf.obstacles, "obstacles")
            assert_bits_equal(op.download(r.voxel_keys, r.n_voxel, np.uint32), hf.voxel_keys, "voxel keys")
            assert_bits_equal(op.download(r.crop_kept_idx, r.n_crop, np.int32), hf.crop_kept_idx, "crop kept")


def test_batch_from_device_memory_matches_host_input():
    """pcop_process_batch takes host or device frames (the bench's `value` runs on frames resident in HBM)"""
    torch = pytest.importorskip("torch")
    p = synth.params(2)
    n = synth.points_per_frame(2)
    B = 12
    clouds = synth.frames(2, 400, B)
    counts = np.full(B, n, np.int32)
    counts[5] = 90000
    with ObstacleProcessor(p, n, max_batch=16) as op:
        host = op.process_batch(clouds, counts)
        dev = torch.from_numpy(clouds).to("cuda:0")
        res = op.process_batch_raw(dev.data_ptr(), n, counts)
        from pointcloud_obstacle_processing_b200.result import Frame
        for f in range(B):
            g = Frame.from_c(res[f])
            assert g.n_clusters == host[f].n_clusters and g.n_remaining == host[f].n_remaining
            assert_bits_equal(g.cluster_indices, host[f].cluster_indices, "indices")
            assert_bits_equal(g.remaining_cloud, host[f].remaining_cloud, "remaining")
            assert_bits_equal(g.obstacles, host[f].obstacles, "obstacles")


def test_batch_parity_on_64_frames():
    """BASELINE configs[4] (frame batches): 64 distinct HDL-64 frames through one pcop_process_batch call on two lanes,
    every frame checked against the oracle (counts, index sets bit-exact, obstacles within 1e-5)"""
    from concurrent.futures import ThreadPoolExecutor
    p = synth.params(2)  # default outputs: remaining cloud, clusters, obstacles
    n = synth.points_per_frame(2)
    B = 64
    clouds = synth.frames(2, 1000, B)
    with ObstacleProcessor(p, n, max_batch=B) as op:
        res = op.process_batch(clouds)
    with ThreadPoolExecutor(8) as ex:
        oracle = list(ex.map(lambda f: O.process(p, clouds[f]), range(B)))
    for f in range(B):
        compare_frames(res[f], oracle[f], p, f"frame{f}: ")
    assert sum(o.n_clusters for o in oracle) > 10 * B


@pytest.mark.parametrize("seed,opacity", [(1, 0), (2, 50), (3, 77), (4, -5)])
def test_occupancy_shadows_synthetic(seed, opacity):
    """od.cpp:467-672, 817-833 on synthetic clusters and an arbitrary sensor pose: start / end cells, line counts and
    every grid cell bit-exact against the oracle"""
    from shadow_util import rigid, shadow_scene
    p = synth.params(1)
    p.grid_opacity = opacity
    cloud, offsets, indices = shadow_scene(seed, n_clusters=12, noise=2000)
    sw, ws = rigid(0.3 * seed, 0.5, 0.1, [5.2, 1.9, 1.1])
    with ObstacleProcessor(p, len(cloud)) as op:
        grid0, _, _ = op.occupancy_grid(cloud)
        g_grid, g_rec, g_warn = op.handle_shadow_casting(grid0, cloud, offsets, indices, ws, sw)
    o_grid, o_rec, o_warn = O.occupancy_shadows(p, grid0, cloud, offsets, indices, ws, sw)
    assert_bits_equal(g_rec, o_rec, "shadow records")
    assert_bits_equal(g_grid, o_grid, "grid cells")
    assert g_warn == o_warn == 0
    assert (o_rec[:, 4] > 0).sum() >= 5 and (o_grid == 100).sum() > 500


@pytest.mark.parametrize("config", [1, 2])
def test_occupancy_grid_product_of_a_frame(config, frames):
    """the node's published product for one frame: initial data set (od.cpp:727), pipeline, shadows + marks
    (od.cpp:817-833) chained on the device library, against the same chain on the oracle"""
    from shadow_util import rigid
    p = synth.params(config)
    p.grid_opacity = 40
    if config == 2:
        p.block_size = 0.25
    cloud = frames[config]
    sw, ws = rigid(0.1, 0.45, 0.0, [p.x_max + 0.8, 0.5 * (p.y_min + p.y_max), 1.2])
    with ObstacleProcessor(p, len(cloud)) as op:
        grid0, _, _ = op.occupancy_grid(cloud)
        fr = op.process(cloud)
        g_grid, g_rec, g_warn = op.handle_shadow_casting(grid0, fr.remaining_cloud, fr.cluster_offsets, fr.cluster_indices,
                                                         ws, sw)
    o_grid0, _, _ = O.occupancy_grid(p, cloud)
    ofr = O.process(p, cloud)
    o_grid, o_rec, o_warn = O.occupancy_shadows(p, o_grid0, ofr.remaining_cloud, ofr.cluster_offsets, ofr.cluster_indices,
                                                ws, sw)
    assert fr.n_clusters == ofr.n_clusters and fr.n_clusters > 0
    assert_bits_equal(g_rec, o_rec, "shadow records")
    assert_bits_equal(g_grid, o_grid, "grid cells")
    assert g_warn == o_warn
    assert (o_grid == 100).sum() > 0 and (o_rec[:, 4] > 0).any()


def test_occupancy_shadows_degenerate_and_device_inputs():
    """NaN members, the 2^20-step cap of the cell search, a fan too long to draw (warning), no clusters, empty cloud;
    then the same call with every array resident on the device (PCOP_OUT_DEVICE consumers)"""
    torch = pytest.importorskip("torch")
    import ctypes as C
    from shadow_util import rigid, shadow_scene
    p = synth.params(1)
    p.grid_opacity = 33
    cloud, offsets, indices = shadow_scene(5)
    eye = np.eye(4, dtype=np.float32)
    sw, ws = rigid(0.2, 0.4, 0.0, [5.0, 2.0, 1.0])
    far_sw, _ = rigid(0.0, 0.0, 0.0, [-3.0e6, 3.0e6, 0.0])
    bad = cloud.copy()
    bad[indices[offsets[0]], 1] = np.nan
    bad[indices[offsets[1] + 1], 0] = np.nan
    tall = np.array([[1e-6, -1.0, 1.0, 1.0], [0.5, 1.2, 0.2, 1.0], [0.6, 1.1, 0.1, 1.0]], np.float32)
    cases = [
        ("no clusters", cloud, np.zeros(1, np.int32), np.zeros(0, np.int32), ws, sw),
        ("nan members", bad, offsets, indices, ws, sw),
        ("far pose", cloud, offsets, indices, eye, far_sw),
        ("fan too long", tall, np.array([0, 3], np.int32), np.arange(3, dtype=np.int32), eye, eye),
        ("empty cloud", np.zeros((0, 4), np.float32), np.zeros(1, np.int32), np.zeros(0, np.int32), ws, sw),
    ]
    with ObstacleProcessor(p, len(cloud)) as op:
        grid0, _, _ = op.occupancy_grid(cloud)
        for what, cl, off, idx, m_ws, m_sw in cases:
            g_grid, g_rec, g_warn = op.handle_shadow_casting(grid0, cl, off, idx, m_ws, m_sw)
            o_grid, o_rec, o_warn = O.occupancy_shadows(p, grid0, cl, off, idx, m_ws, m_sw)
            assert_bits_equal(g_rec, o_rec, what + ": shadow records")
            assert_bits_equal(g_grid, o_grid, what + ": grid cells")
            assert g_warn == o_warn, what
            if what == "fan too long":
                assert g_warn == 16
        # device-resident inputs and grid
        d_cloud = torch.from_numpy(cloud).cuda()
        d_off = torch.from_numpy(offsets).cuda()
        d_idx = torch.from_numpy(indices).cuda()
        d_grid = torch.from_numpy(grid0.copy()).cuda()
        rec = np.zeros((len(offsets) - 1, 6), np.int32)
        warn = C.c_uint32(0)
        op._check(op._lib.pcop_occupancy_shadows(op._h, d_cloud.data_ptr(), len(cloud), d_off.data_ptr(), d_idx.data_ptr(),
                                                 len(offsets) - 1, ws.ctypes.data_as(C.c_void_p), sw.ctypes.data_as(C.c_void_p),
                                                 d_grid.data_ptr(), rec.ctypes.data_as(C.c_void_p), C.byref(warn)))
        o_grid, o_rec, _ = O.occupancy_shadows(p, grid0, cloud, offsets, indices, ws, sw)
        assert_bits_equal(d_grid.cpu().numpy(), o_grid, "device-resident grid")
        assert_bits_equal(rec, o_rec, "device-resident records")


def test_bench_size_batch_is_position_independent():
    """BASELINE configs[4] at the bench's call size: 1024 frames in ONE pcop_process_batch call (4 lanes, uneven waves,
    early remaining-cloud copy).  The batch is 24 distinct frames laid out in a pseudo-random order; every copy must
    give exactly the arrays its source frame gives in a 24-frame call (itself checked against the oracle): a frame's
    result may not depend on its position, its wave, its lane or its neighbours."""
    import zlib
    from concurrent.futures import ThreadPoolExecutor
    p = synth.params(2)  # default outputs: remaining cloud + source indices, clusters, obstacles
    n = synth.points_per_frame(2)
    D, B = 24, 1024
    src = synth.frames(2, 2000, D)

    def digest(fr):
        parts = [np.int32([fr.n_crop, fr.n_voxel, fr.n_remaining, fr.n_clusters, fr.n_cluster_points, fr.warnings]),
                 fr.remaining_cloud, fr.remaining_src_idx, fr.cluster_offsets, fr.cluster_indices, fr.obstacles]
        crc = 0
        for a in parts:
            crc = zlib.crc32(np.ascontiguousarray(a).tobytes(), crc)
        return crc

    with ObstacleProcessor(p, n, max_batch=D) as op:
        small = op.process_batch(src)
    with ThreadPoolExecutor(8) as ex:
        oracle = list(ex.map(lambda f: O.process(p, src[f]), range(D)))
    for f in range(D):
        compare_frames(small[f], oracle[f], p, f"source frame {f}: ")
    want = [digest(fr) for fr in small]
    order = np.random.default_rng(77).integers(0, D, B)
    batch = np.ascontiguousarray(src[order])
    with ObstacleProcessor(p, n, max_batch=B) as op:
        for rep in range(2):  # the second call reuses every lane's buffers
            res = op.process_batch(batch)
            got = [digest(fr) for fr in res]
            bad = [f for f in range(B) if got[f] != want[order[f]]]
            assert not bad, f"call {rep}: {len(bad)} of {B} frames differ from their source frame, first {bad[:5]}"


def test_pointcloud2_staging_growth_keeps_the_other_buffers(frames):
    """a PointCloud2 message larger than the raw staging buffer makes the library grow that buffer; the occupancy,
    shadow and result buffers of the same handle must survive it (round-1 finding: they were freed with it)"""
    from shadow_util import rigid
    p = all_outputs(synth.params(2))
    p.grid_opacity = 40
    p.block_size = 0.25
    n = synth.points_per_frame(2)
    clouds = synth.frames(2, 300, 4)
    sw, ws = rigid(0.1, 0.45, 0.0, [p.x_max + 0.8, 0.5 * (p.y_min + p.y_max), 1.2])
    with ObstacleProcessor(p, n, max_batch=4) as op:
        for rnd, npts in enumerate((4000, 30000, 90000)):  # each message more than 1.25x the previous one
            grid, counts, row_avg = op.occupancy_grid(clouds[0])
            og, oc, oa = O.occupancy_grid(p, clouds[0])
            assert_bits_equal(grid, og, "grid")
            res = op.process_batch(clouds)
            r0 = res[0]
            sg, rec, w = op.handle_shadow_casting(grid, r0.remaining_cloud, r0.cluster_offsets, r0.cluster_indices, ws, sw)
            osg, orec, ow = O.occupancy_shadows(p, og, r0.remaining_cloud, r0.cluster_offsets, r0.cluster_indices, ws, sw)
            assert_bits_equal(sg, osg, f"shadow grid, round {rnd}")
            data = _make_pointcloud2(clouds[1][:npts, :3], 32, (0, 4, 8), seed=rnd)
            op.accumulate_reset()
            assert op.accumulate_pointcloud2(data, npts, 32, 0, 4, 8) == npts
            g = op.process_accumulated()
            o = O.process(p, clouds[1][:npts])
            compare_frames(g, o, p, f"accumulated, round {rnd}: ")
            for f in range(4):
                compare_frames(res[f], O.process(p, clouds[f]), p, f"round {rnd} frame {f}: ")


def test_python_wrappers_reject_device_results():
    p = synth.params(2)
    p.outputs = abi.OUT_DEFAULT | abi.OUT_DEVICE
    with ObstacleProcessor(p, 1000) as op:
        with pytest.raises(ValueError):
            op.process(np.zeros((10, 4), np.float32))


def test_no_device_allocation_after_the_first_call():
    """every buffer is allocated by pcop_create (the pinned result buffer grows once): repeated calls of the same shape
    must not change the free device memory (cudaMemGetInfo)"""
    import torch
    p = synth.params(2)
    n = synth.points_per_frame(2)
    clouds = synth.frames(2, 500, 24)
    counts = np.full(24, n, np.int32)
    with ObstacleProcessor(p, n, max_batch=24) as op:
        op.process_batch_raw(clouds.ctypes.data, n, counts)
        torch.cuda.synchronize()
        free0, _ = torch.cuda.mem_get_info()
        for _ in range(3):
            op.process_batch_raw(clouds.ctypes.data, n, counts)
            op.process_batch_raw(clouds.ctypes.data, n, counts[:1])
        torch.cuda.synchronize()
        free1, _ = torch.cuda.mem_get_info()
    assert free1 == free0, (free0, free1)


def test_batch_larger_than_max_batch_runs_in_waves():
    """a call may hold more frames than max_batch (the handle's wave buffers): it is processed in as many waves as it
    takes; results of all frames stay valid until the next call"""
    p = synth.params(2)
    n = synth.points_per_frame(2)
    B = 40
    clouds = synth.frames(2, 600, B)
    with ObstacleProcessor(p, n, max_batch=16) as op:
        res = op.process_batch(clouds)
    for f in (0, 7, 16, 23, 39):
        compare_frames(res[f], O.process(p, clouds[f]), p, f"frame{f}: ")


@pytest.mark.parametrize("point_step,offs", [(16, (0, 4, 8)), (32, (0, 4, 8)), (22, (1, 9, 14)), (12, (8, 0, 4))])
def test_pointcloud2_egress(point_step, offs, frames):
    """pcl::toROSMsg of the debug publishers (od.cpp:290-294): the PointCloud2 payload of a cloud, bit for bit; the
    reference's own layout (16, 0, 4, 8) is the PointXYZ array itself, padding float included"""
    p = all_outputs(synth.params(2))
    cloud = frames[2]
    with ObstacleProcessor(p, len(cloud)) as op:
        fr = op.process(cloud)
        for c in (fr.voxel_centroids, fr.remaining_cloud, cloud[:1], cloud[:0]):
            g = op.cloud_to_pointcloud2(c, point_step, *offs)
            o = O.xyz_to_pointcloud2(c, point_step, *offs)
            assert_bits_equal(g, o, f"PointCloud2 payload ({len(c)} points)")
        if point_step == 16:
            assert g.tobytes() == np.ascontiguousarray(cloud[:0]).tobytes()
            rt = op.pointcloud2_to_xyz(op.cloud_to_pointcloud2(fr.remaining_cloud), fr.n_remaining, 16, 0, 4, 8)
            assert_bits_equal(rt, fr.remaining_cloud, "egress -> ingest round trip")


def test_pointcloud2_egress_from_device_results():
    """a result array left on the GPU (outputs | OUT_DEVICE) serialised without a detour through the host"""
    p = synth.params(2)
    cloud = synth.frame(2, 3)
    with ObstacleProcessor(p, len(cloud)) as op:
        host = op.process(cloud)
    pd = p.copy()
    pd.outputs = abi.OUT_DEFAULT | abi.OUT_DEVICE
    with ObstacleProcessor(pd, len(cloud)) as op:
        res = op.process_batch_raw(np.ascontiguousarray(cloud).ctypes.data, len(cloud), np.array([len(cloud)], np.int32))
        import ctypes as C
        ptr = C.cast(res[0].remaining_cloud, C.c_void_p).value
        g = op.cloud_to_pointcloud2(None, device_ptr=ptr, n=res[0].n_remaining)
    assert_bits_equal(g, O.xyz_to_pointcloud2(host.remaining_cloud, 16, 0, 4, 8), "payload of the device-resident remaining cloud")


@pytest.mark.parametrize("config,batch,check", [(3, 6, (0, 3, 5)), (4, 3, (0, 2))])
def test_batch_of_large_frames_through_the_generic_paths(config, batch, check):
    """BASELINE configs[2] / [3] batched, as bench.py runs them: remaining clouds far above the fused clustering kernel's
    8960 points (generic clustering after one speculative miss), dense voxel buckets (LSD voxel path after one declined
    wave), a plane input above the resident kernel's small tier; two calls, so that the second one runs with the
    handle's adapted choices"""
    p = all_outputs(synth.params(config))
    clouds = synth.frames(config, 20, batch)
    with ObstacleProcessor(p, clouds.shape[1], max_batch=batch) as op:
        first = op.process_batch(clouds)
        res = op.process_batch(clouds)
    for f in check:
        o = O.process(p, clouds[f])
        compare_frames(first[f], o, p, f"config {config} first call frame {f}: ")
        compare_frames(res[f], o, p, f"config {config} second call frame {f}: ")
