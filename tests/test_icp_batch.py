"""Batched ICP (pcr_icp_point_to_*_batch): many (source frame, target frame) pairs of one buffer in one call.

CPU tests: the Python layer rejects bad arguments with ValueError before it touches a device.
GPU tests: every pair against the CPU oracle (the ICP bar of test_gpu_parity.py) and against the single-pair call;
a pair's result bit for bit independent of the other pairs of the call and of repetition; the edge cases of the
single-pair call, all inside one batch.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest

import pointclouds_rs_b200 as P
from pointclouds_rs_b200 import _ffi, scenes

T = max(1, min(16, os.cpu_count() or 1))
gpu = pytest.mark.gpu


def _pack(frames):
    off = np.zeros(len(frames) + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in frames])
    pts = np.vstack([np.asarray(f, np.float32).reshape(-1, 3) for f in frames]) if frames else np.zeros((0, 3), np.float32)
    return np.ascontiguousarray(pts, np.float32), off


# ---- argument checks (no device needed) ------------------------------------------------------------------------

def _args():
    pts = np.zeros((10, 3), np.float32)
    return pts, [0, 4, 10], [[1, 0]]


@pytest.mark.parametrize("offsets", [[0, 6, 4, 10], [0, 4, 9], [1, 4, 10], [0, 4, 11], []])
def test_bad_offsets_raise(offsets):
    pts, _, pairs = _args()
    with pytest.raises(ValueError):
        P.icp_point_to_point_batch(pts, offsets, pairs)
    with pytest.raises(ValueError):
        P.icp_point_to_plane_batch(pts, offsets, pairs, np.zeros_like(pts))


@pytest.mark.parametrize("pairs", [[[0, 2]], [[2, 0]], [[-1, 0]]])
def test_pair_frame_id_out_of_range_raises(pairs):
    pts, off, _ = _args()
    with pytest.raises(ValueError):
        P.icp_point_to_point_batch(pts, off, pairs)


@pytest.mark.parametrize("pairs", [[0, 1], [[0, 1, 1]], np.zeros((2, 2, 2), np.int64), [[0.0, 1.0]]])
def test_pairs_of_the_wrong_shape_raise(pairs):
    pts, off, _ = _args()
    with pytest.raises(ValueError):
        P.icp_point_to_point_batch(pts, off, pairs)


@pytest.mark.parametrize("shape", [(9, 3), (10, 2), (30,)])
def test_normals_shape_mismatch_raises(shape):
    pts, off, pairs = _args()
    with pytest.raises(ValueError):
        P.icp_point_to_plane_batch(pts, off, pairs, np.zeros(shape, np.float32))
    with pytest.raises(ValueError):
        P.icp_point_to_plane_batch(pts, off, pairs, None)


@pytest.mark.parametrize("kw", [{"tolerance": -1e-3}, {"tolerance": math.nan}, {"max_correspondence_distance": -1.0},
                                {"max_correspondence_distance": math.nan}])
def test_bad_parameters_raise(kw):
    pts, off, pairs = _args()
    with pytest.raises(ValueError):
        P.icp_point_to_point_batch(pts, off, pairs, **kw)
    with pytest.raises(ValueError):
        P.icp_point_to_plane_batch(pts, off, pairs, np.zeros_like(pts), **kw)


# ---- GPU ----------------------------------------------------------------------------------------------------------

def _check_icp(res, o, atol=1e-4, exact_iters=True):
    # (as in test_gpu_parity.py) the stopping test |prev_rmse - rmse| < tol is evaluated at the f32 noise floor once ICP
    # has converged, so the iteration at which it first holds may differ by a few when the per-iteration arithmetic is not
    # bit-identical (the engine reduces in f64 trees, the reference sequentially).
    if exact_iters:
        assert res.num_iterations == o.num_iterations, (res.num_iterations, o.num_iterations)
    else:
        assert abs(res.num_iterations - o.num_iterations) <= 4, (res.num_iterations, o.num_iterations)
    assert res.converged == o.converged
    assert np.allclose(np.array(res.rotation), o.rotation, atol=atol), (res.rotation, o.rotation)
    assert np.allclose(np.array(res.translation), o.translation, atol=atol), (res.translation, o.translation)
    assert res.rmse == o.rmse or abs(res.rmse - o.rmse) <= 1e-4 * max(1.0, abs(o.rmse))  # (== : no correspondences, both inf)
    assert abs(res.fitness - o.fitness) < 1e-6


def _bits(r):
    return (np.float32(r.rotation).tobytes(), np.float32(r.translation).tobytes(), np.float32(r.rmse).tobytes(),
            np.float32(r.fitness).tobytes(), r.num_iterations, r.converged)


@pytest.fixture(scope="module")
def mixed(oracle):
    """~6 consecutive pairs of a 20 K-point sequence, hemisphere pairs of 500 and 6000 points, a reduced aerial pair."""
    frames, pairs = [], []
    seq = scenes.kitti_sequence(7, seed=5, counts=(17_600, 880, 145, 495))
    for i, f in enumerate(seq):
        frames.append(f)
        if i:
            pairs.append((i, i - 1))
    # a motion from which point-to-point converges within the 30 fixed iterations (7 and 17 in the oracle): after 30 of the
    # 68 iterations rot_z(0.05) needs, the 6000-point hemisphere is still moving along its nearly symmetric yaw mode, where
    # the engine and the reference (f64 vs f32 H, DESIGN section 3.4) are more than 1e-4 apart
    for tgt in (scenes.hemisphere(500, 99, 5.0), scenes.hemisphere(6000, 99, 5.0), scenes.aerial_scene(42, 0.01)):
        src = oracle.apply_transform(tgt, scenes.rot_z(0.01), [0.05, -0.03, 0.02])
        frames += [np.asarray(src, np.float32), tgt]
        pairs.append((len(frames) - 2, len(frames) - 1))
    pts, off = _pack(frames)
    # the same normals for both sides (the oracle's), as test_icp_fixed_iterations does
    nrm = np.zeros_like(pts)
    for f in range(len(frames)):
        b, e = int(off[f]), int(off[f + 1])
        nrm[b:e] = oracle.normals(pts[b:e], 15, threads=T)
    return pts, off, np.array(pairs, np.uint32), nrm


def _frame(pts, off, f):
    return pts[int(off[f]):int(off[f + 1])]


def _single(pcr, plane, pts, off, nrm, s, t, **kw):
    src = pcr.PointCloud.from_numpy(np.ascontiguousarray(_frame(pts, off, s)))
    tgt = pcr.PointCloud.from_numpy(np.ascontiguousarray(_frame(pts, off, t)))
    if plane:
        tgt.normals = np.ascontiguousarray(_frame(nrm, off, t))
        return pcr.icp_point_to_plane(src, tgt, **kw)
    return pcr.icp_point_to_point(src, tgt, **kw)


def _batch(pcr, plane, pts, off, pairs, nrm, **kw):
    if plane:
        return pcr.icp_point_to_plane_batch(pts, off, pairs, nrm, **kw)
    return pcr.icp_point_to_point_batch(pts, off, pairs, **kw)


@gpu
@pytest.mark.parametrize("plane", [False, True], ids=["p2p", "p2plane"])
@pytest.mark.parametrize("tol,iters,exact", [(0.0, 30, True), (1e-6, 100, False)])
def test_batch_matches_oracle(pcr, oracle, mixed, plane, tol, iters, exact):
    pts, off, pairs, nrm = mixed
    res = _batch(pcr, plane, pts, off, pairs, nrm, max_iterations=iters, tolerance=tol)
    assert len(res) == len(pairs)
    for j, ((s, t), r) in enumerate(zip(pairs, res)):
        if not plane and j == len(pairs) - 1:
            # the aerial pair: on this 500 m scene the single-pair call's point-to-point also departs from the reference by
            # more than 1e-4 (54 vs 17 iterations at tolerance 1e-6); test_batch_matches_single_calls holds the batch to it
            continue
        src, tgt = _frame(pts, off, s), _frame(pts, off, t)
        if plane:
            o = oracle.icp_point_to_plane(src, tgt, _frame(nrm, off, t), iters, tol, threads=T)
        else:
            o = oracle.icp_point_to_point(src, tgt, iters, tol, threads=T)
        _check_icp(r, o, exact_iters=exact)
        if tol == 0.0:
            assert r.num_iterations == iters and not r.converged


@gpu
@pytest.mark.parametrize("plane", [False, True], ids=["p2p", "p2plane"])
def test_batch_matches_single_calls(pcr, mixed, plane):
    pts, off, pairs, nrm = mixed
    for tol, iters, exact in ((0.0, 30, True), (1e-6, 100, False)):
        res = _batch(pcr, plane, pts, off, pairs, nrm, max_iterations=iters, tolerance=tol)
        for (s, t), r in zip(pairs, res):
            _check_icp(r, _single(pcr, plane, pts, off, nrm, s, t, max_iterations=iters, tolerance=tol), exact_iters=exact)


@gpu
@pytest.mark.parametrize("plane", [False, True], ids=["p2p", "p2plane"])
def test_pair_results_independent_and_reproducible(pcr, mixed, plane):
    pts, off, pairs, nrm = mixed
    kw = dict(max_iterations=40, tolerance=1e-6)
    full = [_bits(r) for r in _batch(pcr, plane, pts, off, pairs, nrm, **kw)]
    again = [_bits(r) for r in _batch(pcr, plane, pts, off, pairs, nrm, **kw)]
    assert full == again
    perm = np.random.default_rng(1).permutation(len(pairs))
    permuted = [_bits(r) for r in _batch(pcr, plane, pts, off, pairs[perm], nrm, **kw)]
    for j, p in enumerate(perm):
        assert permuted[j] == full[p]
    for p in range(len(pairs)):
        alone = _batch(pcr, plane, pts, off, pairs[p:p + 1], nrm, **kw)
        assert [_bits(alone[0])] == [full[p]], p
    # a pair listed twice in one call gets the same answer twice
    twice = _batch(pcr, plane, pts, off, np.vstack([pairs[:1], pairs[:1]]), nrm, **kw)
    assert _bits(twice[0]) == _bits(twice[1]) == full[0]


@gpu
@pytest.mark.parametrize("plane", [False, True], ids=["p2p", "p2plane"])
def test_edge_cases_in_one_batch(pcr, plane):
    empty = np.zeros((0, 3), np.float32)
    a = scenes.kitti_scene(21, (4_000, 200, 40, 60))
    b1, b2, b3 = (np.ascontiguousarray(a @ scenes.rot_z(r).T + np.float32(d), np.float32)
                  for r, d in ((0.02, 0.1), (-0.03, -0.15), (0.01, 0.05)))
    nonfinite = a.copy()
    nonfinite[::97] = np.nan
    nonfinite[5::211, 1] = np.inf
    nonfinite_src = np.ascontiguousarray(nonfinite @ scenes.rot_z(0.02).T + np.float32(0.1), np.float32)
    far = np.ascontiguousarray(a + np.float32(1000.0), np.float32)
    small_t = scenes.hemisphere(100, 7, 5.0)
    small_s = np.ascontiguousarray(small_t @ scenes.rot_z(0.04).T + np.float32([0.2, -0.1, 0.05]), np.float32)
    big_t = scenes.kitti_scene(22)[:100_000]
    big_s = np.ascontiguousarray(big_t @ scenes.rot_z(0.01).T + np.float32([0.3, 0.1, 0.0]), np.float32)
    frames = [empty, a, np.array([[1, 2, 3]], np.float32), np.array([[1.5, 2.5, 2.5]], np.float32), b1, b2, b3, nonfinite,
              nonfinite_src, far, small_t, small_s, big_t, big_s, empty]
    E, A, ONE1, ONE2, B1, B2, B3, NF, NFS, FAR, ST, SS, BT, BS, E2 = range(len(frames))
    pairs = np.array([(E, A), (A, E), (E, E2), (ONE2, ONE1), (A, A), (B1, A), (B2, A), (B3, A), (NFS, NF), (A, NF),
                      (FAR, A), (SS, ST), (BS, BT)], np.uint32)
    pts, off = _pack(frames)
    nrm = np.zeros_like(pts)
    for f in range(len(frames)):
        b, e = int(off[f]), int(off[f + 1])
        if e > b:
            nrm[b:e] = pcr.normals_array(pcr.PointCloud.from_numpy(np.ascontiguousarray(pts[b:e])), 15)
    kw = dict(max_iterations=60, tolerance=1e-6, max_correspondence_distance=5.0)
    res = _batch(pcr, plane, pts, off, pairs, nrm, **kw)
    for (s, t), r in zip(pairs, res):
        _check_icp(r, _single(pcr, plane, pts, off, nrm, s, t, **kw), exact_iters=False)
    eye = np.eye(3).tolist()
    # icp.rs:131-139: an empty side -> identity, 0 iterations, converged only when both are empty
    for j, conv in ((0, False), (1, False), (2, True)):
        assert res[j].num_iterations == 0 and res[j].converged == conv and res[j].rotation == eye and res[j].translation == [0, 0, 0]
    assert res[4].converged and np.allclose(res[4].rotation, eye, atol=1e-6) and np.allclose(res[4].translation, 0, atol=1e-6)
    assert res[10].num_iterations == 1 and not res[10].converged and res[10].fitness == 0.0  # nothing within 5 m
    assert res[11].num_iterations != res[12].num_iterations  # the 100-point and the 100 K-point pair finish at different passes
    # max_iterations = 0: the metrics of the initial alignment only
    kw0 = dict(kw, max_iterations=0)
    for (s, t), r in zip(pairs, _batch(pcr, plane, pts, off, pairs, nrm, **kw0)):
        o = _single(pcr, plane, pts, off, nrm, s, t, **kw0)
        assert r.num_iterations == 0 and r.rotation == eye and r.translation == [0, 0, 0]
        _check_icp(r, o)


@gpu
def test_errors(pcr):
    pts, off = _pack([scenes.hemisphere(300, 1), scenes.hemisphere(300, 2)])
    pairs = np.array([[1, 0]], np.uint32)
    lib, h = _ffi.load(), pcr.default_context()._h
    x, y, z = (np.ascontiguousarray(pts[:, i]) for i in range(3))
    prm = _ffi.IcpParams(10, 1e-5, math.inf)
    res = (_ffi.IcpResultC * 1)()
    f = lambda a: a.ctypes.data_as(_ffi.f32p)
    u64 = lambda a: a.ctypes.data_as(_ffi.u64p)
    u32 = lambda a: a.ctypes.data_as(_ffi.u32p)
    st = lib.pcr_icp_point_to_plane_batch(h, f(x), f(y), f(z), u64(off), 2, f(x), f(y), f(z), len(x) - 1, u32(pairs), 1, C.byref(prm), res)
    assert st == _ffi.PCR_ERR_NORMALS_MISMATCH
    bad = np.array([[2, 0]], np.uint32)
    st = lib.pcr_icp_point_to_point_batch(h, f(x), f(y), f(z), u64(off), 2, u32(bad), 1, C.byref(prm), res)
    assert st == _ffi.PCR_ERR_INVALID_ARG
    dec = np.array([0, 400, 300], np.uint64)
    st = lib.pcr_icp_point_to_point_batch(h, f(x), f(y), f(z), u64(dec), 2, u32(pairs), 1, C.byref(prm), res)
    assert st == _ffi.PCR_ERR_INVALID_ARG
    with pytest.raises(ValueError):
        pcr.icp_point_to_plane_batch(pts, off, pairs, np.zeros((len(pts) - 1, 3), np.float32))
    with pytest.raises(ValueError):
        pcr.icp_point_to_plane_batch(pts, off, pairs, None)
    with pytest.raises(ValueError):
        pcr.icp_point_to_point_batch(pts, off, [[0, 2]])
    assert pcr.icp_point_to_point_batch(pts, off, np.zeros((0, 2), np.uint32)) == []
