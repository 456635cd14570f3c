"""Pins the CPU oracle to every known-answer test the reference holds for the KNN path.

Each test restates a reference unit test (file:line given) on the same hand-built input and checks
the oracle against the reference's own assertions.  The Rust reference itself cannot be built here
(no cargo/rustc), so these are the strongest pins available; exact KNN lists / masks on realistic
inputs are pinned by the oracle alone (see oracle/pcr_oracle.h).
"""
import math
import os

import numpy as np
import pytest

# The reference's data/ fixtures, restated as far as its tests pin them (tests/golden/reference_data/README.md)
REF_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_data")


def cloud(x, y=None, z=None):
    if y is None:
        return np.asarray(x, np.float32).reshape(-1, 3)
    return np.stack([np.asarray(x, np.float32), np.asarray(y, np.float32), np.asarray(z, np.float32)], 1)


# ---- crates/spatial/src/kdtree.rs:166-269 -----------------------------------------------------------
def test_knn_returns_expected_neighbors(oracle):  # :173-183
    t = oracle.Tree(cloud([0, 1, 2, 10], [0] * 4, [0] * 4))
    idx, dist = t.knn([0.2, 0, 0], 2)
    assert list(idx) == [0, 1] and dist[0] <= dist[1]


def test_radius_search_finds_points(oracle):  # :186-192
    t = oracle.Tree(cloud([0, 0.5, 2], [0] * 3, [0] * 3))
    assert list(t.radius_search([0, 0, 0], 0.75)) == [0, 1]


def test_knn_edge_cases(oracle):  # :194-243
    empty = oracle.Tree(np.zeros((0, 3), np.float32))
    assert len(empty.knn([0, 0, 0], 5)[0]) == 0
    one = oracle.Tree(cloud([1], [2], [3]))
    assert len(one.knn([0, 0, 0], 0)[0]) == 0
    assert len(one.knn([np.nan, 0, 0], 1)[0]) == 0
    assert len(empty.radius_search([0, 0, 0], 10.0)) == 0
    assert len(oracle.Tree(cloud([0], [0], [0])).radius_search([0, 0, 0], -1.0)) == 0
    three = oracle.Tree(cloud([0, 1, 2], [0] * 3, [0] * 3))
    assert len(three.knn([0, 0, 0], 100)[0]) == 3


def test_knn_distances_are_sorted(oracle):  # :246-253
    t = oracle.Tree(cloud([0, 3, 1, 7, 2], [0] * 5, [0] * 5))
    _, dist = t.knn([0.5, 0, 0], 5)
    assert (np.diff(dist) >= 0).all()


def test_radius_search_exact_boundary(oracle):  # :255-269
    t = oracle.Tree(cloud([1, 5], [0, 0], [0, 0]))
    idx = t.radius_search([0, 0, 0], 1.0)
    assert 0 in idx and 1 not in idx


def test_adversarial_kdtree(oracle):  # tests/test_adversarial.rs:84-143
    one = oracle.Tree(cloud([1], [2], [3]))
    idx, dist = one.knn([1, 2, 3], 1)
    assert list(idx) == [0] and dist[0] == 0
    for q in ([np.inf, 0, 0], [np.nan, np.nan, np.nan], [-np.inf, 0, 0]):
        assert len(one.knn(q, 1)[0]) == 0 and len(one.radius_search(q, 1.0)) == 0
    assert len(one.radius_search([1, 2, 3], 0.0)) == 0
    assert len(one.radius_search([1, 2, 3], np.inf)) == 0


def test_find_correspondences(oracle):  # crates/registration/src/correspondence.rs:47-113
    c = cloud([0, 1, 2], [0] * 3, [0] * 3)
    si, ti, dd = oracle.Tree(c).find_correspondences(c)
    assert list(si) == list(ti) == [0, 1, 2] and (np.abs(dd) < 1e-6).all()
    src = cloud([0, 1, 10], [0] * 3, [0] * 3)
    si, ti, dd = oracle.Tree(c).find_correspondences(src, 3.0)
    assert list(si) == [0, 1]
    assert len(oracle.Tree(cloud([1], [2], [3])).find_correspondences(np.zeros((0, 3), np.float32))[0]) == 0
    assert len(oracle.Tree(np.zeros((0, 3), np.float32)).find_correspondences(cloud([1], [2], [3]))[0]) == 0


# ---- crates/filters/src/statistical_outlier.rs:71-146 ------------------------------------------------
def test_sor_removes_outliers(oracle):  # :78-101
    v = [0.0, 0.1, -0.1, 0.05, -0.05, 100.0]
    keep, _, _ = oracle.sor(cloud(v, v, v), 4, 1.0)
    assert list(keep) == [1, 1, 1, 1, 1, 0]


def test_sor_keeps_inliers(oracle):  # :104-124
    g = np.arange(3, dtype=np.float32)
    pts = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    keep, _, _ = oracle.sor(pts, 5, 3.0)
    assert keep.sum() == 27


def test_sor_degenerate(oracle):  # :127-146
    assert len(oracle.sor(np.zeros((0, 3), np.float32), 5, 1.0)[0]) == 0
    assert list(oracle.sor(cloud([1], [2], [3]), 5, 1.0)[0]) == [1]
    assert list(oracle.sor(cloud([1, 2], [3, 4], [5, 6]), 0, 1.0)[0]) == [0, 0]


# ---- crates/filters/src/radius_outlier.rs:26-61, tests/test_adversarial.rs:185-193 -------------------
def test_ror(oracle):
    keep = oracle.ror(cloud([0, 0.1, 0.2, 100], [0] * 4, [0] * 4), 0.5, 2)
    assert list(keep) == [1, 1, 1, 0]
    assert oracle.ror(cloud([0, 0.1, 0.2, 0.3, 0.4], [0] * 5, [0] * 5), 1.0, 2).sum() == 5
    assert list(oracle.ror(cloud([0], [0], [0]), 1.0, 2)) == [0]


# ---- crates/normals/src/estimate.rs:240-492 ----------------------------------------------------------
def _plane(axis, n=10, spacing=1.0, offset=0.0):
    i, j = np.divmod(np.arange(n * n), n)
    pert = offset + np.arange(n * n, dtype=np.float32) * np.float32(1e-7)
    a, b = i.astype(np.float32) * np.float32(spacing), j.astype(np.float32) * np.float32(spacing)
    return cloud(a, b, pert) if axis == 2 else cloud(a, pert, b)


def test_normals_of_planes(oracle):  # :307-350
    n = oracle.normals(_plane(2), 10)
    assert (np.abs(n[:, 2]) > 0.9).all()
    n = oracle.normals(_plane(1), 10)
    assert (np.abs(n[:, 1]) > 0.9).all()


def test_normals_of_sphere(oracle):  # :353-384
    n_lat = n_lon = 20
    pts = []
    for i in range(1, n_lat):
        th = np.float32(np.pi) * np.float32(i) / np.float32(n_lat)
        for j in range(n_lon):
            ph = np.float32(2.0 * np.pi) * np.float32(j) / np.float32(n_lon)
            pts.append([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)])
    pts = np.asarray(pts, np.float32)
    n = oracle.normals(pts, 15)
    dots = np.sum(n * (-pts), axis=1)
    assert (dots > 0.8).mean() > 0.85


def test_normals_unit_length_and_degenerate(oracle):  # :387-453, tests/test_adversarial.rs:197-211
    n = oracle.normals(_plane(2, 5), 5)
    assert np.allclose(np.linalg.norm(n, axis=1), 1.0, atol=1e-5)
    assert oracle.normals(np.zeros((0, 3), np.float32), 10).shape == (0, 3)
    assert oracle.normals(cloud([1], [2], [3]), 5).shape == (1, 3)
    assert oracle.normals(cloud([1], [2], [3]), 0).shape == (0, 3)
    i = np.arange(20, dtype=np.float32)
    line = oracle.normals(cloud(i, i * np.float32(1e-7), i * np.float32(2e-7)), 5)
    assert np.isfinite(line).all()
    assert np.isfinite(oracle.normals(cloud([1, 1], [1, 1], [1, 1]), 5)).all()


def test_normals_viewpoint(oracle):  # :456-492
    pts = _plane(2, 10, 1.0, 5.0)
    above = oracle.normals(pts, 10, (5.0, 5.0, 100.0))
    below = oracle.normals(pts, 10, (5.0, 5.0, -100.0))
    for t in (44, 45, 55, 54):
        assert above[t, 2] > 0.9 and below[t, 2] < -0.9


# ---- data fixtures (SURVEY 8c: expected values by inspection) ------------------------------------------
def test_reference_data_fixtures(oracle):
    bunny = oracle.read_pcd_ascii(os.path.join(REF_DATA, "bunny.pcd"))
    assert bunny.tolist() == [[0.0, 0.0, 0.0]]
    # config 1: SOR(k=10, std 1.0) keeps the single point; normals k=20 -> exactly (0, 0, 1)
    assert list(oracle.sor(bunny, 10, 1.0)[0]) == [1]
    assert oracle.normals(bunny, 20).tolist() == [[0.0, 0.0, 1.0]]
    assert oracle.read_pcd_ascii(os.path.join(REF_DATA, "two_scans.pcd")).tolist() == [[0, 0, 0], [1, 1, 1]]
    p = oracle.read_pcd_ascii(os.path.join(REF_DATA, "plane_with_noise.pcd"))
    assert p.shape == (3, 3) and abs(p[1, 2] - 1.01) < 1e-6


# ---- crates/registration/src/icp.rs:300-599 ----------------------------------------------------------
CUBE = cloud([0, 1, 0, 1, 0, 1, 0, 1], [0, 0, 1, 1, 0, 0, 1, 1], [0, 0, 0, 0, 1, 1, 1, 1])
I3 = np.eye(3, dtype=np.float32)


def test_icp_identity(oracle):  # :326-344, :428-434
    r = oracle.icp_point_to_point(CUBE, CUBE)
    assert np.allclose(r.rotation, I3, atol=1e-4) and np.allclose(r.translation, 0, atol=1e-4)
    assert r.rmse < 1e-4 and abs(r.fitness - 1.0) < 1e-6 and r.converged


@pytest.mark.xfail(strict=True, reason=(
    "icp.rs:347-371 `known_translation` as the reference states it (shift exactly 1.0): iteration 1 pairs every source with the "
    "face x = 1 and moves the cube by 0.5; in iteration 2 the sources at x = 1.5 are EXACTLY equidistant from the target faces "
    "x = 1 and x = 2 (a 4-way tie per point).  Under the (d^2, index) order this engine and its oracle define -- north_star: "
    "'KNN index sets bit-exact under a (distance, index) tie-break' -- the lower index wins, the pairing does not change and ICP "
    "stalls at rmse 0.5; the reference passes only through kiddo's unspecified traversal order.  Kept verbatim so that a "
    "maintainer running the reference's own suite sees the one red test and its cause; the intent is pinned tie-free below."))
def test_icp_known_translation_as_in_the_reference(oracle):
    tgt = oracle.apply_transform(CUBE, I3, [1.0, 0, 0])
    r = oracle.icp_point_to_point(CUBE, tgt, 100, 1e-8)
    assert r.converged
    assert r.rmse < 1e-3
    assert np.allclose(r.translation, [1.0, 0, 0], atol=0.05)


def test_icp_known_translation_tie_free(oracle):
    # icp.rs:347-371 shifts by exactly 1.0, which makes the second iteration an exact 4-way tie
    # (sources at x = 1.5 between target faces x = 1 and x = 2): its outcome rests on kiddo's
    # unspecified tie order.  A shift below 0.5 has unique nearest neighbours and pins the intent.
    tgt = oracle.apply_transform(CUBE, I3, [0.3, 0, 0])
    r = oracle.icp_point_to_point(CUBE, tgt, 100, 1e-8)
    assert r.converged and r.rmse < 1e-3 and np.allclose(r.translation, [0.3, 0, 0], atol=0.05)


def test_icp_known_rotation_small_angle_z(oracle):  # :374-425
    a = np.float32(np.pi / 6)
    sx = [i * 0.25 - 5.0 for i in range(40)] + [0.0] * 20
    sy = [0.0] * 40 + [i * 0.25 for i in range(20)]
    src = cloud(sx, sy, [0.0] * 60)
    R = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]], np.float32)
    tgt = oracle.apply_transform(src, R, [0, 0, 0])
    r = oracle.icp_point_to_point(src, tgt, 200, 1e-10)
    assert r.converged and r.rmse < 0.05
    out = oracle.apply_transform(src, r.rotation, r.translation)
    assert np.abs(out - tgt).max() < 0.15
    assert abs(r.rotation[0, 0] - np.cos(a)) < 0.1 and abs(r.rotation[0, 1] + np.sin(a)) < 0.1
    assert abs(r.rotation[1, 0] - np.sin(a)) < 0.1 and abs(r.rotation[2, 2] - 1.0) < 0.1


def test_icp_empty_and_limits(oracle):  # :444-513, tests/test_adversarial.rs:236-247
    e = np.zeros((0, 3), np.float32)
    r = oracle.icp_point_to_point(e, e)
    assert np.allclose(r.rotation, I3) and r.num_iterations == 0 and r.converged
    r = oracle.icp_point_to_point(e, CUBE)
    assert r.num_iterations == 0 and not r.converged
    assert oracle.icp_point_to_point(CUBE, CUBE, max_iterations=0).num_iterations == 0
    src = cloud(np.arange(10), [0] * 10, [0] * 10)
    tgt = cloud(np.arange(10) + 0.1, [0] * 10, [0] * 10)
    tight = oracle.icp_point_to_point(src, tgt, 1, 1e-8, 0.01)
    loose = oracle.icp_point_to_point(src, tgt, 1, 1e-8, math.inf)
    assert tight.fitness <= loose.fitness


def test_transform_algebra(oracle):  # :516-599
    out = oracle.apply_transform(CUBE, I3, [0, 0, 0])
    assert np.allclose(out, CUBE, atol=1e-6)
    out = oracle.apply_transform(cloud([1, 2], [3, 4], [5, 6]), I3, [10, 20, 30])
    assert np.allclose(out, [[11, 23, 35], [12, 24, 36]], atol=1e-6)
    R, t = oracle.compose((I3, [1, 0, 0]), (I3, [0, 2, 0]))
    assert np.allclose(t, [1, 2, 0], atol=1e-6)
    Rz = np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1]], np.float32)
    R, t = oracle.compose((Rz, [0, 0, 0]), (I3, [1, 0, 0]))
    p = oracle.apply_transform(cloud([1], [0], [0]), R, t)
    assert np.allclose(p, [[1, 1, 0]], atol=1e-5)
    p = oracle.apply_transform(cloud([1], [0], [0]), Rz, [0, 0, 0])
    assert np.allclose(p, [[0, 1, 0]], atol=1e-6)


# ---- crates/registration/src/icp_plane.rs:238-436 -----------------------------------------------------
def _flat_plane(grid=10):
    i, j = np.divmod(np.arange(grid * grid), grid)
    return cloud(i.astype(np.float32) - grid / 2.0, j.astype(np.float32) - grid / 2.0,
                 np.arange(grid * grid, dtype=np.float32) * np.float32(1e-7))


def test_plane_icp_identity(oracle):  # :263-272
    c = _flat_plane()
    r = oracle.icp_point_to_plane(c, c, oracle.normals(c, 10))
    assert r.converged and r.rmse < 1e-4
    assert np.allclose(r.rotation, I3, atol=1e-3) and np.allclose(r.translation, 0, atol=1e-3)


def test_plane_icp_translation_along_normal(oracle):  # :275-300
    tgt = _flat_plane()
    src = oracle.apply_transform(tgt, I3, [0, 0, 0.2])
    r = oracle.icp_point_to_plane(src, tgt, oracle.normals(tgt, 10), 200, 1e-10)
    assert r.rmse < 0.05 and abs(r.translation[2] + 0.2) < 0.1


def test_plane_icp_small_rotation(oracle):  # :327-380
    pts = []
    for i in range(1, 15):
        th = np.float32(np.pi / 2) * np.float32(i) / np.float32(15)
        for j in range(30):
            ph = np.float32(2 * np.pi) * np.float32(j) / np.float32(30)
            pts.append([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)])
    tgt = np.asarray(pts, np.float32)
    a = np.float32(0.1)
    R = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]], np.float32)
    src = oracle.apply_transform(tgt, R, [0, 0, 0])
    r = oracle.icp_point_to_plane(src, tgt, oracle.normals(tgt, 10), 200, 1e-10)
    assert r.rmse < 0.1
    out = oracle.apply_transform(src, r.rotation, r.translation)
    assert np.linalg.norm(out - tgt, axis=1).max() < 0.2


def test_plane_icp_empty_and_mismatch(oracle):  # :381-406
    e = np.zeros((0, 3), np.float32)
    r = oracle.icp_point_to_plane(e, e, e)
    assert np.allclose(r.rotation, I3) and r.num_iterations == 0
    c = cloud([0, 1], [0, 0], [0, 0])
    with pytest.raises(ValueError):
        oracle.icp_point_to_plane(c, c, np.zeros((3, 3), np.float32))


def test_hemisphere_registration(oracle):  # tests/real_world_pipeline.rs:191-255 (PCG64 instead of ChaCha12)
    from pointclouds_rs_b200 import scenes

    tgt = scenes.hemisphere(500, 99, 5.0)
    src = oracle.apply_transform(tgt, scenes.rot_z(0.05), [0.3, -0.2, 0.1])
    r = oracle.icp_point_to_point(src, tgt, 100, 1e-6)
    assert r.converged and r.rmse < 0.5 and np.abs(np.array(r.translation) + [0.3, -0.2, 0.1]).max() < 1.0
    r = oracle.icp_point_to_plane(src, tgt, oracle.normals(tgt, 15), 100, 1e-6)
    assert r.converged and r.rmse < 0.5


# ---- crates/filters/src/voxel_downsample.rs (input preparation of config 2) ---------------------------
def test_voxel_downsample(oracle):
    from pointclouds_rs_b200 import scenes

    pts = cloud([0.1, 0.2, 1.1, 1.3, -0.4], [0.1, 0.3, 0.1, 0.2, 0.0], [0.0, 0.0, 0.0, 0.0, 0.0])
    out = oracle.voxel_downsample(pts, 1.0)
    assert out.shape == (3, 3)  # keys (-1,0,0), (0,0,0), (1,0,0) in key order
    assert np.allclose(out[0], [-0.4, 0, 0]) and np.allclose(out[1], [0.15, 0.2, 0]) and np.allclose(out[2], [1.2, 0.15, 0])
    with pytest.raises(ValueError):
        oracle.voxel_downsample(pts, 0.0)
    big = scenes.kitti_scene(5, (4000, 200, 50, 100))
    for v in (0.05, 0.5):
        a, b = oracle.voxel_downsample(big, v), scenes.voxel_downsample_np(big, v)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
