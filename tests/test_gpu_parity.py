"""Parity of the CUDA path (through the C ABI) with the CPU oracle -- the tests proper.

Bars (BASELINE.json north_star): KNN index lists and distances bit-exact under (d^2, index);
SOR mean distances, statistics and keep masks bit-exact; normals within 1e-4 rad; ICP transforms
within 1e-4.
"""
import math
import os

import numpy as np
import pytest

from pointclouds_rs_b200 import scenes

pytestmark = pytest.mark.gpu

T = max(1, min(16, os.cpu_count() or 1))


def _cloud(pcr, pts):
    return pcr.PointCloud.from_numpy(np.ascontiguousarray(pts, dtype=np.float32))


def lattice(n=10, spacing=1.0):
    g = np.arange(n, dtype=np.float32) * np.float32(spacing)
    return np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, 3).astype(np.float32)


SCENES = {
    "kitti20k": lambda: scenes.kitti_scene(3, (17_000, 850, 140, 1_160)),
    "cube20k": lambda: scenes.uniform_cube(20_000, 5),
    "lattice1000": lambda: lattice(10),
    "dupes": lambda: np.repeat(scenes.uniform_cube(500, 9, 0, 10), 7, axis=0),
    "line": lambda: np.stack([np.arange(300, dtype=np.float32), np.zeros(300, np.float32), np.zeros(300, np.float32)], 1),
    "tiny5": lambda: scenes.uniform_cube(5, 1, 0, 1),
    "plane_far_outlier": lambda: np.vstack([scenes.kitti_scene(4, (5_000, 10, 10, 10)), [[4000.0, -3000.0, 900.0]]]).astype(np.float32),
    **scenes.ADVERSARIAL,  # exact ties, duplicates, density ramps, far k-th neighbours, cell faces, flat grids
}


def _queries(pts, rng):
    own = pts[rng.integers(0, len(pts), min(len(pts), 1500))]
    fin = pts[np.isfinite(pts).all(1)]
    lo, hi = fin.min(0), fin.max(0)
    ext = rng.uniform(lo - 0.3 * (hi - lo) - 1, hi + 0.3 * (hi - lo) + 1, (400, 3)).astype(np.float32)
    far = np.array([[1e6, 1e6, 1e6], [-5e4, 0, 0], [0, 0, 1e-30]], np.float32)
    bad = np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf]], np.float32)
    return np.vstack([own, ext, far, bad]).astype(np.float32)


@pytest.mark.parametrize("scene", list(SCENES))
@pytest.mark.parametrize("k", [1, 2, 11, 12, 13, 20, 21, 22, 32, 33, 70])
def test_knn_bit_exact(pcr, oracle, scene, k):
    pts = SCENES[scene]()
    rng = np.random.default_rng(11)
    q = _queries(pts, rng)
    tree = pcr.KdTree(_cloud(pcr, pts), k_hint=k)
    idx, dist, cnt = tree.knn(q, k)
    o_idx, o_dist, o_cnt = oracle.Tree(pts).knn_batch(q, k, threads=T)
    assert np.array_equal(cnt, o_cnt)
    assert np.array_equal(idx, o_idx), f"first diff row {np.nonzero((idx != o_idx).any(1))[0][:5]}"
    assert np.array_equal(dist.view(np.uint32), o_dist.view(np.uint32))
    idx2, cnt2 = tree.knn_indices(q, k)
    assert np.array_equal(idx2, o_idx) and np.array_equal(cnt2, o_cnt)


def test_knn_nonfinite_points_are_not_indexed(pcr, oracle):
    pts = scenes.uniform_cube(3000, 2, 0, 10)
    pts[::17, 0] = np.nan
    pts[5::31, 2] = np.inf
    q = scenes.uniform_cube(500, 3, 0, 10)
    tree = pcr.KdTree(_cloud(pcr, pts), k_hint=8)
    idx, dist, cnt = tree.knn(q, 8)
    o_idx, o_dist, o_cnt = oracle.Tree(pts).knn_batch(q, 8)
    assert np.array_equal(idx, o_idx) and np.array_equal(dist.view(np.uint32), o_dist.view(np.uint32))
    assert tree.len() == 3000 and tree.info()["n_indexed"] == int(np.isfinite(pts).all(1).sum())


def test_knn_edge_cases(pcr):
    empty = pcr.KdTree(pcr.PointCloud())
    idx, dist, cnt = empty.knn(np.zeros((3, 3), np.float32), 5)  # kdtree.rs:194-201
    assert (cnt == 0).all() and (idx == 0xFFFFFFFF).all() and np.isinf(dist).all()
    one = pcr.KdTree(_cloud(pcr, [[1, 2, 3]]))
    idx, dist, cnt = one.knn(np.array([[0, 0, 0], [np.nan, 0, 0]], np.float32), 0)  # kdtree.rs:204-210
    assert (cnt == 0).all()
    idx, dist, cnt = one.knn(np.array([[0, 0, 0], [np.nan, 0, 0]], np.float32), 1)  # kdtree.rs:213-219
    assert list(cnt) == [1, 0] and idx[0, 0] == 0
    three = pcr.KdTree(_cloud(pcr, [[0, 0, 0], [1, 0, 0], [2, 0, 0]]))
    idx, dist, cnt = three.knn(np.zeros((1, 3), np.float32), 100)  # kdtree.rs:238-243
    assert cnt[0] == 3 and list(idx[0, :3]) == [0, 1, 2]
    # kdtree.rs:173-183
    col = pcr.KdTree(_cloud(pcr, [[0, 0, 0], [1, 0, 0], [2, 0, 0], [10, 0, 0]]))
    idx, dist, cnt = col.knn(np.array([[0.2, 0, 0]], np.float32), 2)
    assert list(idx[0]) == [0, 1] and dist[0, 0] <= dist[0, 1]


@pytest.mark.parametrize("scene,k,std", [("kitti20k", 10, 1.0), ("kitti20k", 20, 2.0), ("cube20k", 10, 1.0),
                                         ("lattice1000", 5, 3.0), ("dupes", 4, 1.0), ("plane_far_outlier", 10, 1.0),
                                         ("kitti20k", 40, 1.0)]
                         + [(name, k, 1.0) for name in scenes.ADVERSARIAL for k in (10, 20, 21, 31)])
def test_sor_bit_exact(pcr, oracle, scene, k, std):
    pts = SCENES[scene]()
    keep, kept, mean_d, stats = pcr.sor_mask(_cloud(pcr, pts), k, std, want_mean=True)
    o_keep, o_mean, o_stats = oracle.sor(pts, k, std, threads=T)
    assert np.array_equal(mean_d.view(np.uint32), o_mean.view(np.uint32))
    assert np.array_equal(stats.view(np.uint32), o_stats.view(np.uint32)), (stats, o_stats)
    assert np.array_equal(keep, o_keep) and kept == int(o_keep.sum())


def test_sor_full_frame_122k(pcr, oracle):
    pts = scenes.kitti_scene()  # BASELINE config 2
    assert len(pts) == 122_000
    keep, kept, mean_d, stats = pcr.sor_mask(_cloud(pcr, pts), 10, 1.0, want_mean=True)
    o_keep, o_mean, o_stats = oracle.sor(pts, 10, 1.0, threads=T)
    assert np.array_equal(mean_d.view(np.uint32), o_mean.view(np.uint32))
    assert np.array_equal(stats.view(np.uint32), o_stats.view(np.uint32))
    assert np.array_equal(keep, o_keep)


def test_sor_reference_known_answers(pcr):
    # statistical_outlier.rs:78-101
    v = [0.0, 0.1, -0.1, 0.05, -0.05, 100.0]
    c = _cloud(pcr, np.stack([v, v, v], 1))
    out = pcr.statistical_outlier_removal(c, 4, 1.0)
    assert len(out) == 5 and np.abs(out.to_numpy()).max() <= 0.2
    # :104-124
    assert len(pcr.statistical_outlier_removal(_cloud(pcr, lattice(3)), 5, 3.0)) == 27
    # :127-146
    assert len(pcr.statistical_outlier_removal(pcr.PointCloud(), 5, 1.0)) == 0
    single = pcr.statistical_outlier_removal(_cloud(pcr, [[1, 2, 3]]), 5, 1.0)
    assert len(single) == 1 and list(single.to_numpy()[0]) == [1, 2, 3]
    assert len(pcr.statistical_outlier_removal(_cloud(pcr, [[1, 3, 5], [2, 4, 6]]), 0, 1.0)) == 0
    with pytest.raises(ValueError):
        pcr.statistical_outlier_removal(_cloud(pcr, [[1, 3, 5], [2, 4, 6]]), 3, float("nan"))
    with pytest.raises(ValueError):
        pcr.statistical_outlier_removal(_cloud(pcr, [[1, 3, 5], [2, 4, 6]]), 3, -1.0)


def test_sor_with_nonfinite_points(pcr, oracle):
    pts = scenes.kitti_scene(8, (4_000, 200, 50, 100))
    pts[10] = [np.nan, 0, 0]
    pts[500] = [0, np.inf, 1]
    keep, kept, mean_d, stats = pcr.sor_mask(_cloud(pcr, pts), 10, 1.0, want_mean=True)
    o_keep, o_mean, o_stats = oracle.sor(pts, 10, 1.0)
    assert np.array_equal(mean_d.view(np.uint32), o_mean.view(np.uint32))
    assert np.array_equal(keep, o_keep) and keep[10] == 0 and keep[500] == 0


def _angles(a, b):
    """Angle between directions (sign-insensitive), robust near 0: atan2(|a x b|, |a . b|)."""
    a = a.astype(np.float64)
    b = b.astype(np.float64)
    return np.arctan2(np.linalg.norm(np.cross(a, b), axis=1), np.abs(np.sum(a * b, axis=1)))


@pytest.mark.parametrize("scene,k", [("kitti20k", 20), ("cube20k", 10), ("kitti20k", 15), ("cube20k", 40), ("dupes", 6)])
def test_normals_parity(pcr, oracle, scene, k):
    pts = SCENES[scene]()
    nrm = pcr.normals_array(_cloud(pcr, pts), k)
    o = oracle.normals(pts, k, threads=T)
    assert nrm.shape == o.shape
    ang = _angles(nrm, o)
    # tolerance from north_star: 1e-4 rad (modulo sign only where the orientation dot is ~0)
    assert np.nanmax(ang) < 1e-4, f"max angle {np.nanmax(ang)}, n>1e-4: {(ang > 1e-4).sum()}"
    same_sign = np.sum(nrm * o, axis=1) > 0
    assert same_sign.mean() > 0.9999
    ln = np.linalg.norm(nrm, axis=1)
    assert np.allclose(ln, 1.0, atol=1e-5)


def test_normals_reference_known_answers(pcr):
    # estimate.rs:307-350 planes, :401-453 degenerate, :456-492 viewpoint
    idx = np.arange(100, dtype=np.float32)
    i, j = np.divmod(np.arange(100), 10)
    xy = np.stack([i.astype(np.float32), j.astype(np.float32), idx * np.float32(1e-7)], 1)
    n = pcr.normals_array(_cloud(pcr, xy), 10)
    assert (np.abs(n[:, 2]) > 0.9).all()
    xz = np.stack([i.astype(np.float32), idx * np.float32(1e-7), j.astype(np.float32)], 1)
    n = pcr.normals_array(_cloud(pcr, xz), 10)
    assert (np.abs(n[:, 1]) > 0.9).all()
    assert pcr.normals_array(pcr.PointCloud(), 10).shape == (0, 3)
    assert pcr.normals_array(_cloud(pcr, [[1, 2, 3]]), 0).shape == (0, 3)
    one = pcr.normals_array(_cloud(pcr, [[0, 0, 0]]), 20)  # data/bunny.pcd: exactly (0,0,1)
    assert one.tolist() == [[0.0, 0.0, 1.0]]
    two = pcr.normals_array(_cloud(pcr, [[1, 1, 1], [1, 1, 1]]), 5)  # test_adversarial.rs:197-211
    assert np.isfinite(two).all()
    up = np.stack([i.astype(np.float32), j.astype(np.float32), 5 + idx * np.float32(1e-7)], 1)
    above = pcr.normals_array(_cloud(pcr, up), 10, (5.0, 5.0, 100.0))
    below = pcr.normals_array(_cloud(pcr, up), 10, (5.0, 5.0, -100.0))
    for t in (44, 45, 55, 54):
        assert above[t, 2] > 0.9 and below[t, 2] < -0.9
    withn = pcr.estimate_normals(_cloud(pcr, xy), 10)
    assert withn.normals_to_numpy().shape == (100, 3) and len(withn) == 100


def test_normals_nonfinite_points(pcr, oracle):
    pts = scenes.uniform_cube(2000, 4, 0, 5)
    pts[7] = [np.nan, 1, 1]
    nrm = pcr.normals_array(_cloud(pcr, pts), 8)
    o = oracle.normals(pts, 8)
    assert nrm[7].tolist() == [0.0, 0.0, 1.0] == o[7].tolist()
    ok = np.ones(len(pts), bool)
    ok[7] = False
    assert np.nanmax(_angles(nrm[ok], o[ok])) < 1e-4


@pytest.mark.parametrize("radius", [0.05, 0.5, 2.0])
def test_radius_parity(pcr, oracle, radius):
    pts = scenes.kitti_scene(6, (8_000, 400, 60, 140))
    rng = np.random.default_rng(5)
    q = _queries(pts, rng)
    tree = pcr.KdTree(_cloud(pcr, pts), k_hint=10)
    cnt = tree.radius_count(q, radius)
    otree = oracle.Tree(pts)
    assert np.array_equal(cnt, otree.radius_count_batch(q, radius, threads=T))
    off, idx = tree.radius_search(q, radius)
    assert np.array_equal(np.diff(off).astype(np.uint32), cnt)
    for j in list(range(0, 60)) + [len(q) - 1, len(q) - 4]:
        assert np.array_equal(idx[off[j]:off[j + 1]], otree.radius_search(q[j], radius))
    # kdtree.rs:106-112: r <= 0 / non-finite -> empty
    assert (tree.radius_count(q, 0.0) == 0).all() and (tree.radius_count(q, -1.0) == 0).all()
    assert (tree.radius_count(q, float("inf")) == 0).all()


def test_radius_exact_boundary(pcr):
    tree = pcr.KdTree(_cloud(pcr, [[1, 0, 0], [5, 0, 0]]))  # kdtree.rs:255-269
    off, idx = tree.radius_search(np.zeros((1, 3), np.float32), 1.0)
    assert list(idx) == [0]
    tree = pcr.KdTree(_cloud(pcr, [[0, 0, 0], [0.5, 0, 0], [2, 0, 0]]))  # kdtree.rs:186-192
    off, idx = tree.radius_search(np.zeros((1, 3), np.float32), 0.75)
    assert list(idx) == [0, 1]


def test_ror_parity(pcr, oracle):
    pts = scenes.kitti_scene(6, (8_000, 400, 60, 140))
    for r, mn in [(0.5, 5), (0.3, 2), (2.0, 40)]:
        keep, kept = pcr.ror_mask(_cloud(pcr, pts), r, mn)
        assert np.array_equal(keep, oracle.ror(pts, r, mn, threads=T)) and kept == int(keep.sum())
    # radius_outlier.rs:26-61 and tests/test_adversarial.rs:185-193
    c = _cloud(pcr, [[0, 0, 0], [0.1, 0, 0], [0.2, 0, 0], [100, 0, 0]])
    assert len(pcr.radius_outlier_removal(c, 0.5, 2)) == 3
    assert len(pcr.radius_outlier_removal(_cloud(pcr, [[0, 0, 0]]), 1.0, 2)) == 0
    assert len(pcr.radius_outlier_removal(pcr.PointCloud(), 1.0, 2)) == 0
    with pytest.raises(ValueError):
        pcr.radius_outlier_removal(c, 0.0, 2)


def test_apply_transform_bit_exact(pcr, oracle):
    pts = scenes.uniform_cube(5000, 12, -50, 50)
    R = scenes.rot_z(0.3)
    t = [0.5, -1.25, 3.0]
    out = pcr.apply_transform(_cloud(pcr, pts), R, t).to_numpy()
    ref = oracle.apply_transform(pts, R, t)
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))


def test_find_correspondences(pcr, oracle):
    tgt = scenes.hemisphere(3000, 3)
    src = oracle.apply_transform(tgt, scenes.rot_z(0.03), [0.1, 0.0, -0.05])
    tree = pcr.KdTree(_cloud(pcr, tgt), k_hint=1)
    for md in (math.inf, 0.12):
        si, ti, dd = tree.find_correspondences(_cloud(pcr, src), md)
        osi, oti, odd = oracle.Tree(tgt).find_correspondences(src, md, threads=T)
        assert np.array_equal(si, osi) and np.array_equal(ti, oti)
        assert np.array_equal(dd.view(np.uint32), odd.view(np.uint32))


def _check_icp(res, o, atol=1e-4, exact_iters=True):
    # The stopping test |prev_rmse - rmse| < tol is evaluated at the f32 noise floor once ICP has
    # converged, so the iteration at which it first holds may differ by a few when the per-iteration
    # arithmetic is not bit-identical (the engine reduces in f64 trees, the reference sequentially).
    if exact_iters:
        assert res.num_iterations == o.num_iterations, (res.num_iterations, o.num_iterations)
    else:
        assert abs(res.num_iterations - o.num_iterations) <= 4, (res.num_iterations, o.num_iterations)
    assert res.converged == o.converged
    assert np.allclose(np.array(res.rotation), o.rotation, atol=atol), (res.rotation, o.rotation)
    assert np.allclose(np.array(res.translation), o.translation, atol=atol), (res.translation, o.translation)
    assert abs(res.rmse - o.rmse) <= 1e-4 * max(1.0, abs(o.rmse))
    assert abs(res.fitness - o.fitness) < 1e-6


@pytest.mark.parametrize("n", [500, 6000])
def test_icp_parity_hemisphere(pcr, oracle, n):
    # tests/real_world_pipeline.rs:191-255 shape
    tgt = scenes.hemisphere(n, 99, 5.0)
    src = oracle.apply_transform(tgt, scenes.rot_z(0.05), [0.3, -0.2, 0.1])
    s, t = _cloud(pcr, src), _cloud(pcr, tgt)
    res = pcr.icp_point_to_point(s, t, max_iterations=100, tolerance=1e-6)
    o = oracle.icp_point_to_point(src, tgt, 100, 1e-6, threads=T)
    _check_icp(res, o, exact_iters=False)
    assert res.converged and res.rmse < 0.5
    tn = pcr.estimate_normals(t, 15)
    res = pcr.icp_point_to_plane(s, tn, max_iterations=100, tolerance=1e-6)
    o = oracle.icp_point_to_plane(src, tgt, oracle.normals(tgt, 15, threads=T), 100, 1e-6, threads=T)
    _check_icp(res, o, exact_iters=False)
    assert res.converged and res.rmse < 0.5


def test_icp_fixed_iterations(pcr, oracle):
    # BASELINE config 4 shape at reduced size: tolerance 0 -> exactly max_iterations iterations
    tgt = scenes.aerial_scene(42, 0.01)
    src = oracle.apply_transform(tgt, scenes.rot_z(0.05), [0.3, -0.2, 0.1])
    nrm = oracle.normals(tgt, 20, threads=T)
    t = _cloud(pcr, tgt)
    t.normals = nrm
    res = pcr.icp_point_to_plane(_cloud(pcr, src), t, max_iterations=30, tolerance=0.0)
    o = oracle.icp_point_to_plane(src, tgt, nrm, 30, 0.0, threads=T)
    assert res.num_iterations == 30 and not res.converged
    _check_icp(res, o)


def test_icp_reference_known_answers(pcr):
    cube = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0], [0, 0, 1], [1, 0, 1], [0, 1, 1], [1, 1, 1]], np.float32)
    c = _cloud(pcr, cube)
    r = pcr.icp_point_to_point(c, c)  # icp.rs:326-344
    assert np.allclose(r.rotation, np.eye(3), atol=1e-4) and np.allclose(r.translation, 0, atol=1e-4)
    assert r.rmse < 1e-4 and abs(r.fitness - 1.0) < 1e-6 and r.converged
    # icp.rs:347-371 (known_translation) shifts by exactly 1.0: at the second iteration the source
    # corners at x = 1.5 are EXACTLY equidistant (d^2 = 0.25) from the target faces x = 1 and x = 2,
    # so its outcome rests on kiddo's unspecified tie order.  With the engine's (d^2, index) rule
    # the tie goes to x = 1 and ICP legitimately stalls at rmse 0.5; the CPU oracle must agree.
    # The same test with a tie-free shift of 0.3 pins the intended behaviour (any shift >= 0.5 runs
    # into the same symmetric tie after the first centroid alignment).
    t = _cloud(pcr, cube + np.array([0.3, 0, 0], np.float32))
    r = pcr.icp_point_to_point(c, t, 100, 1e-8)
    assert r.converged and r.rmse < 1e-3 and np.allclose(r.translation, [0.3, 0, 0], atol=0.05)
    e = pcr.PointCloud()
    r = pcr.icp_point_to_point(e, e)  # icp.rs:444-455
    assert r.num_iterations == 0 and r.converged and np.allclose(r.rotation, np.eye(3))
    r = pcr.icp_point_to_point(e, c)  # icp.rs:458-468
    assert r.num_iterations == 0 and not r.converged
    r = pcr.icp_point_to_point(c, c, max_iterations=0)  # tests/test_adversarial.rs:236-247
    assert r.num_iterations == 0
    with pytest.raises(ValueError):  # icp_plane.rs:27-32 / registration.rs:66-71
        pcr.icp_point_to_plane(c, c)
    bad = _cloud(pcr, cube)
    bad.normals = np.zeros((3, 3), np.float32)
    with pytest.raises(ValueError):
        pcr.icp_point_to_plane(c, bad)


def test_icp_tie_dependent_reference_case(pcr, oracle):
    cube = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0], [0, 0, 1], [1, 0, 1], [0, 1, 1], [1, 1, 1]], np.float32)
    tgt = cube + np.array([1, 0, 0], np.float32)
    r = pcr.icp_point_to_point(_cloud(pcr, cube), _cloud(pcr, tgt), 100, 1e-8)
    o = oracle.icp_point_to_point(cube, tgt, 100, 1e-8)
    _check_icp(r, o)


def test_sor_many_far_outliers_use_coarser_levels(pcr, oracle):
    # outliers whose k-th neighbour is dozens of cells away exercise the level-1/2 grids
    rng = np.random.default_rng(3)
    dense = scenes.kitti_scene(9, (20_000, 500, 100, 0))
    far = rng.uniform(-400, 400, (300, 3)).astype(np.float32)
    pts = np.vstack([dense, far]).astype(np.float32)
    keep, kept, mean_d, stats = pcr.sor_mask(_cloud(pcr, pts), 10, 1.0, want_mean=True)
    o_keep, o_mean, o_stats = oracle.sor(pts, 10, 1.0, threads=T)
    assert np.array_equal(mean_d.view(np.uint32), o_mean.view(np.uint32))
    assert np.array_equal(keep, o_keep)
    nrm = pcr.normals_array(_cloud(pcr, pts), 20)
    assert np.nanmax(_angles(nrm, oracle.normals(pts, 20, threads=T))) < 1e-4
    tree = pcr.KdTree(_cloud(pcr, pts), 40)
    q = np.vstack([far, rng.uniform(-1000, 1000, (200, 3)).astype(np.float32)])
    for k in (3, 40):
        idx, dist, cnt = tree.knn(q, k)
        o_idx, o_dist, o_cnt = oracle.Tree(pts).knn_batch(q, k, threads=T)
        assert np.array_equal(idx, o_idx) and np.array_equal(dist.view(np.uint32), o_dist.view(np.uint32))


def test_batch_matches_single_frames(pcr, oracle):
    frames = [scenes.kitti_scene(s, (3_000 + 200 * s, 150, 30, 70 + s)) for s in range(5)]
    frames.insert(2, np.array([[1, 2, 3]], np.float32))      # one-point frame
    frames.insert(4, np.zeros((0, 3), np.float32))           # empty frame
    off = np.concatenate([[0], np.cumsum([len(f) for f in frames])])
    pts = np.vstack(frames)
    keep, nrm, kept = pcr.sor_normals_batch(pts, off, 10, 1.0, 20)
    for f, fr in enumerate(frames):
        sl = slice(off[f], off[f + 1])
        if len(fr) == 0:
            continue
        o_keep, _, _ = oracle.sor(fr, 10, 1.0, threads=T)
        assert np.array_equal(keep[sl], o_keep), f"frame {f}"
        assert kept[f] == o_keep.sum()
        sel = np.nonzero(o_keep)[0]
        o_n = oracle.normals(fr[sel], 20, threads=T)
        got = nrm[sl][sel]
        assert np.nanmax(_angles(got, o_n)) < 1e-4, f"frame {f}"
        assert (nrm[sl][o_keep == 0] == 0).all()


def test_batch_large_k_generic_path(pcr, oracle):
    # k > 32 runs the shared-memory top-k kernels on every level, with the tombstoned shared index
    frames = [scenes.kitti_scene(20 + s, (2_000, 100, 20, 40)) for s in range(2)]
    off = np.concatenate([[0], np.cumsum([len(f) for f in frames])])
    keep, nrm, kept = pcr.sor_normals_batch(np.vstack(frames), off, 35, 1.0, 40)
    for f, fr in enumerate(frames):
        sl = slice(off[f], off[f + 1])
        o_keep, _, _ = oracle.sor(fr, 35, 1.0, threads=T)
        assert np.array_equal(keep[sl], o_keep)
        sel = np.nonzero(o_keep)[0]
        assert np.nanmax(_angles(nrm[sl][sel], oracle.normals(fr[sel], 40, threads=T))) < 1e-4


# ---- fused SOR -> normals: one search, the normals from the SOR pass's neighbour lists ----------------
@pytest.mark.parametrize("k_sor,std,k_nrm", [(10, 1.0, 20), (20, 2.0, 15), (5, 0.0, 8), (31, 1.0, 10), (10, 0.3, 31), (3, 1.0, 1)])
def test_fused_lists_equal_the_two_step_path(pcr, oracle, k_sor, std, k_nrm):
    """K = max(k_sor, k_nrm) + 1 <= 32 takes the fused path.  std = 0 / 0.3 remove a third to a half of the points, so
    most lists lose more neighbours than their margin and the fallback search carries the result; the normals must be
    BIT-identical to estimate_normals on the filtered cloud (same kernels' arithmetic, same neighbour order)."""
    pts = np.vstack([scenes.kitti_scene(31, (6_000, 300, 60, 140)), [[np.nan, 0, 0], [1, np.inf, 2]]]).astype(np.float32)
    _fused_equals_two_step(pcr, oracle, pts, k_sor, std, k_nrm, check_angles=True)


@pytest.mark.parametrize("k_sor,std,k_nrm", [(10, 1.0, 20), (5, 0.0, 8), (31, 1.0, 10), (10, 0.3, 31), (3, 1.0, 1)])
@pytest.mark.parametrize("scene", ["tie_grid", "dup_cloud"])
def test_fused_lists_equal_the_two_step_path_on_ties(pcr, oracle, scene, k_sor, std, k_nrm):
    """The same on clouds where most lists depend on the index tie-break (exact d^2 ties, duplicate points): a shared
    wrong member would not cancel out, because the filtered cloud renumbers the points.  (The oracle's normals are not
    compared here: symmetric neighbourhoods leave the smallest eigenvector undetermined.)"""
    _fused_equals_two_step(pcr, oracle, scenes.ADVERSARIAL[scene](), k_sor, std, k_nrm, check_angles=False)


def _fused_equals_two_step(pcr, oracle, pts, k_sor, std, k_nrm, check_angles):
    off = np.array([0, len(pts)], np.uint64)
    keep, nrm, kept = pcr.sor_normals_batch(pts, off, k_sor, std, k_nrm)
    o_keep, _, _ = oracle.sor(pts, k_sor, std, threads=T)
    assert np.array_equal(keep, o_keep) and kept[0] == o_keep.sum()
    sel = np.nonzero(o_keep)[0]
    two_step = pcr.normals_array(_cloud(pcr, pts[sel]), k_nrm)      # a fresh search on the filtered cloud
    assert np.array_equal(nrm[sel].view(np.uint32), two_step.view(np.uint32))
    if check_angles:
        assert np.nanmax(_angles(nrm[sel], oracle.normals(pts[sel], k_nrm, threads=T))) < 1e-4
    assert (nrm[o_keep == 0] == 0).all()
    dev = pcr.DeviceCloud.from_numpy(pts).sor_normals(k_sor, std, k_nrm)
    assert np.array_equal(dev.to_numpy(), pts[sel], equal_nan=True) and np.array_equal(dev.normals_to_numpy().view(np.uint32), two_step.view(np.uint32))


@pytest.mark.parametrize("cap", [None, "5"])
@pytest.mark.parametrize("scene", ["dup_cloud", "wires"])
def test_fused_fallback_that_defers_keeps_its_counts(pcr, oracle, monkeypatch, scene, cap):
    """The fallback search of the fused path can defer queries to level 1.  Its own round trips must not clobber the
    fallback count and the kept count that ride along with its first one: a lost kept count made the device-resident
    form return an empty cloud, a lost fallback count skipped the queries beyond the blind pass's capacity."""
    if cap:
        monkeypatch.setenv("PCR_FALLBACK_CAP", cap)
    pts = scenes.ADVERSARIAL[scene]()
    for k_sor, std, k_nrm in ((10, 1.0, 20), (5, 0.0, 8)):
        o_keep, _, _ = oracle.sor(pts, k_sor, std, threads=T)
        sel = np.nonzero(o_keep)[0]
        two_step = pcr.normals_array(_cloud(pcr, pts[sel]), k_nrm)
        dev = pcr.DeviceCloud.from_numpy(pts).sor_normals(k_sor, std, k_nrm)
        assert np.array_equal(dev.to_numpy(), pts[sel], equal_nan=True), (k_sor, std, k_nrm)
        assert np.array_equal(dev.normals_to_numpy().view(np.uint32), two_step.view(np.uint32)), (k_sor, std, k_nrm)
        keep, nrm, kept = pcr.sor_normals_batch(pts, [0, len(pts)], k_sor, std, k_nrm)
        assert np.array_equal(keep, o_keep) and kept[0] == len(sel)
        assert np.array_equal(nrm[sel].view(np.uint32), two_step.view(np.uint32)), (k_sor, std, k_nrm)


def test_fused_fallback_beyond_the_blind_pass(pcr, monkeypatch):
    """The fallback pass is launched before its length is known, for a fixed capacity; what exceeds it runs afterwards.
    A capacity of 5 forces that second pass: the result must not change by a bit."""
    pts = scenes.kitti_scene(32, (6_000, 300, 60, 140))
    want = pcr.DeviceCloud.from_numpy(pts).sor_normals(10, 0.3, 20)
    monkeypatch.setenv("PCR_FALLBACK_CAP", "5")
    got = pcr.DeviceCloud.from_numpy(pts).sor_normals(10, 0.3, 20)
    assert np.array_equal(got.to_numpy(), want.to_numpy())
    assert np.array_equal(got.normals_to_numpy().view(np.uint32), want.normals_to_numpy().view(np.uint32))


def test_fused_lists_multi_frame_edge_cases(pcr, oracle):
    frames = [scenes.kitti_scene(40, (3_000, 150, 30, 70)), np.zeros((0, 3), np.float32), np.array([[1, 2, 3]], np.float32),
              scenes.uniform_cube(15, 4, 0, 1), np.repeat(scenes.uniform_cube(200, 5, 0, 3), 4, axis=0),
              scenes.kitti_scene(41, (2_000, 100, 20, 400))]
    off = np.concatenate([[0], np.cumsum([len(f) for f in frames])])
    keep, nrm, kept = pcr.sor_normals_batch(np.vstack(frames), off, 10, 1.0, 20)
    for f, fr in enumerate(frames):
        sl = slice(off[f], off[f + 1])
        if len(fr) == 0:
            continue
        o_keep, _, _ = oracle.sor(fr, 10, 1.0, threads=T)
        assert np.array_equal(keep[sl], o_keep), f"frame {f}"
        sel = np.nonzero(o_keep)[0]
        if len(sel):
            two_step = pcr.normals_array(_cloud(pcr, fr[sel]), 20)
            assert np.array_equal(nrm[sl][sel].view(np.uint32), two_step.view(np.uint32)), f"frame {f}"


def test_cell_size_cache_never_changes_results(pcr, oracle):
    """With pcr_ctx_set_frame_stream the context reuses the cell size of the previous probe for a cloud of the same size and extent.  Only speed may
    depend on it: a cloud with a very different density profile inside the same box must give the same bits."""
    rng = np.random.default_rng(3)
    n = 20_000
    flat = np.concatenate([rng.uniform(0, 40, (n, 2)), rng.normal(0, 0.02, (n, 1))], 1).astype(np.float32)
    blob = np.concatenate([rng.normal(20, 0.5, (n, 2)), rng.normal(0, 0.02, (n, 1))], 1).astype(np.float32)
    for arr in (flat, blob):  # same bounding box for both: the corners pin it
        arr[:4] = [[0, 0, -0.1], [40, 40, 0.1], [0, 40, 0], [40, 0, 0]]
    ctx = pcr.Context()
    ctx.set_frame_stream(True)
    first = pcr.sor_mask(_cloud(pcr, flat), 10, 1.0, ctx=ctx, want_mean=True)          # probes, fills the cache
    second = pcr.sor_mask(_cloud(pcr, blob), 10, 1.0, ctx=ctx, want_mean=True)         # same n and box: cached cell size
    fresh = pcr.sor_mask(_cloud(pcr, blob), 10, 1.0, ctx=pcr.Context(), want_mean=True)
    assert np.array_equal(second[0], fresh[0]) and np.array_equal(second[2].view(np.uint32), fresh[2].view(np.uint32))
    o_keep, o_mean, _ = oracle.sor(blob, 10, 1.0, threads=T)
    assert np.array_equal(second[0], o_keep) and np.array_equal(second[2].view(np.uint32), o_mean.view(np.uint32))
    assert np.array_equal(first[0], oracle.sor(flat, 10, 1.0, threads=T)[0])


@pytest.mark.parametrize("world", [2, 3, 8])
def test_query_shards_partition_the_cloud(pcr, oracle, world):
    """SURVEY 8e rows 1-2 on ONE GPU: with pcr_ctx_debug_set_shard a context plays one rank of a query-sharded call and
    returns that rank's part (zero bits where another rank writes).  The parts must be disjoint and their integer sum --
    what the NCCL merge computes -- must be the unsharded result bit for bit, for SOR mean distances, normals and the
    radius-outlier mask, with non-finite points (owned by rank 0) in the cloud."""
    pts = scenes.kitti_scene(11, (9_000, 450, 80, 170))
    pts[17] = [np.nan, 1, 2]
    pts[4000] = [3, -np.inf, 0]
    cloud = _cloud(pcr, pts)
    _, _, mean_full, _ = pcr.sor_mask(cloud, 10, 1.0, want_mean=True)
    nrm_full = pcr.normals_array(cloud, 20)
    ror_full, _ = pcr.ror_mask(cloud, 0.5, 5)
    assert np.array_equal(mean_full.view(np.uint32), oracle.sor(pts, 10, 1.0, threads=T)[1].view(np.uint32))
    mean_sum = np.zeros(len(pts), np.uint64)
    nrm_sum = np.zeros((len(pts), 3), np.uint64)
    mean_owners = np.zeros(len(pts), np.int32)
    nrm_owners = np.zeros(len(pts), np.int32)
    ror_or = np.zeros(len(pts), np.uint8)
    for r in range(world):
        ctx = pcr.Context()
        ctx.debug_set_shard(r, world)
        ctx.set_query_sharding(True)
        _, _, mean_r, _ = pcr.sor_mask(cloud, 10, 1.0, ctx=ctx, want_mean=True)
        nrm_r = pcr.normals_array(cloud, 20, ctx=ctx)
        ror_r, _ = pcr.ror_mask(cloud, 0.5, 5, ctx=ctx)
        ctx.close()
        mean_sum += mean_r.view(np.uint32)
        nrm_sum += nrm_r.view(np.uint32)
        mean_owners += mean_r.view(np.uint32) != 0
        nrm_owners += np.any(nrm_r.view(np.uint32) != 0, axis=1)
        ror_or |= ror_r
    assert mean_owners.max() <= 1 and nrm_owners.max() == 1 and nrm_owners.min() == 1  # (a unit normal is never all zero)
    assert np.array_equal(mean_sum.astype(np.uint32), mean_full.view(np.uint32))
    assert np.array_equal(nrm_sum.astype(np.uint32), nrm_full.view(np.uint32))
    assert np.array_equal(ror_or, ror_full)
