"""Comparison helpers shared by the GPU parity tests."""
import numpy as np

REL_TOL = 1e-5  # north_star: centroids, plane coefficients and radii within 1e-5 relative


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_bits_equal(a, b, what):
    a = np.asarray(a)
    b = np.asarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    if a.dtype.kind == "f":
        same = (bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))  # NaN payload / sign is not part of the contract
    else:
        same = a == b
    if not same.all():
        bad = np.argwhere(~same)
        raise AssertionError(f"{what}: {len(bad)} of {a.size} elements differ, first at {bad[0].tolist()}: "
                             f"{a[tuple(bad[0])]!r} vs {b[tuple(bad[0])]!r}")


def assert_close(a, b, what, rel=REL_TOL):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    if a.size == 0:
        return
    scale = np.maximum(np.abs(a), np.abs(b))
    with np.errstate(invalid="ignore"):
        err = np.abs(a - b)  # (inf - inf = NaN: equal infinities are caught by a == b)
        ok = (a == b) | (np.isfinite(a) & np.isfinite(b) & (err <= rel * np.maximum(scale, 1e-30))) | (np.isnan(a) & np.isnan(b))
    if not ok.all():
        bad = np.argwhere(~ok)
        raise AssertionError(f"{what}: {len(bad)} elements beyond rel {rel}, first {bad[0].tolist()}: "
                             f"{a[tuple(bad[0])]} vs {b[tuple(bad[0])]}")


def compare_frames(g, o, params, what=""):
    """g: GPU Frame, o: oracle Frame.  Integer/index outputs bit-exact; floats bit-exact where the design makes
    them so (voxel centroids, remaining cloud), else within REL_TOL (plane coefficients, obstacles)."""
    for k in ("n_input", "n_crop", "n_voxel", "n_sor", "n_remaining", "n_clusters", "n_cluster_points",
              "n_plane_passes", "n_plane_inliers", "warnings"):
        assert getattr(g, k) == getattr(o, k), f"{what}{k}: gpu {getattr(g, k)} vs oracle {getattr(o, k)}"
    assert g.plane_pass_points == o.plane_pass_points, what + "plane_pass_points"
    assert g.plane_pass_inliers == o.plane_pass_inliers, what + "plane_pass_inliers"
    assert_close(g.plane_pass_coeff, o.plane_pass_coeff, what + "plane_pass_coeff")
    assert_close(g.plane_coeff, o.plane_coeff, what + "plane_coeff")
    if g.crop_kept_idx is not None:
        assert_bits_equal(g.crop_kept_idx, o.crop_kept_idx, what + "crop_kept_idx")
    if g.voxel_keys is not None:
        assert_bits_equal(g.voxel_keys, o.voxel_keys, what + "voxel_keys")
        assert_bits_equal(g.voxel_centroids, o.voxel_centroids, what + "voxel_centroids")
    if g.sor_kept_idx is not None:
        assert_bits_equal(g.sor_kept_idx, o.sor_kept_idx, what + "sor_kept_idx")
    if g.plane_inlier_idx is not None:
        assert_bits_equal(g.plane_inlier_idx, o.plane_inlier_idx, what + "plane_inlier_idx")
    if g.remaining_cloud is not None:
        assert_bits_equal(g.remaining_src_idx, o.remaining_src_idx, what + "remaining_src_idx")
        assert_bits_equal(g.remaining_cloud, o.remaining_cloud, what + "remaining_cloud")
    if g.cluster_offsets is not None:
        assert_bits_equal(g.cluster_offsets, o.cluster_offsets, what + "cluster_offsets")
        assert_bits_equal(g.cluster_indices, o.cluster_indices, what + "cluster_indices")
    if g.obstacles is not None:
        assert_close(g.obstacles, o.obstacles, what + "obstacles")


def compare_plane(g, o, what=""):
    """two segment_plane_and_extract_indices results (dicts of pcop_plane's outputs): counts and indices bit-exact,
    the remaining cloud bit-exact, coefficients within REL_TOL"""
    assert g["n_passes"] == o["n_passes"], f"{what}n_passes: {g['n_passes']} vs {o['n_passes']}"
    assert_bits_equal(g["pass_points"], o["pass_points"], what + "pass_points")
    assert_bits_equal(g["pass_inliers"], o["pass_inliers"], what + "pass_inliers")
    assert_close(g["pass_coeff"], o["pass_coeff"], what + "pass_coeff")
    assert_close(g["last_coeff"], o["last_coeff"], what + "last_coeff")
    assert_bits_equal(g["inliers"], o["inliers"], what + "last inliers")
    assert_bits_equal(g["src"], o["src"], what + "remaining src idx")
    assert_bits_equal(g["remaining"], o["remaining"], what + "remaining cloud")
    assert g["warnings"] == o["warnings"], f"{what}warnings: {g['warnings']} vs {o['warnings']}"
