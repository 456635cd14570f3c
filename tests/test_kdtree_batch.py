"""Batch index (pcr_index_build_batch / KdTreeBatch): the KdTree queries of many frames in one call, query frame f searched
in index frame f only.

CPU tests: the Python layer rejects bad offsets, frame-count mismatches and bad shapes (ValueError) before any device work;
the new C symbols are declared and bound.
GPU tests: on a mixed batch (KITTI frames, an empty frame with queries, an all-NaN frame, a one-point frame, a frame below
the brute-force size, a lattice with exact ties, a query frame without queries, non-finite queries, k above a frame's size,
queries far outside their frame's box) every frame's KNN rows, radius counts, radius CSR and correspondences equal, bit for
bit, the single KdTree on that frame alone and the oracle; frames are independent of their neighbours and of their order;
two batch indexes stay valid across other calls on the context; the DeviceFrames build equals the numpy build; the
single-cloud calls reject a batch index; the C error codes; a KITTI sequence against the single calls.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest

import pointclouds_rs_b200 as P
from pointclouds_rs_b200 import _ffi, scenes
from oracle import oracle as O

gpu = pytest.mark.gpu

NEW_SYMBOLS = ("pcr_index_build_batch", "pcr_index_build_batch_dev", "pcr_knn_batch", "pcr_knn_batch_dev", "pcr_radius_count_batch",
               "pcr_radius_count_batch_dev", "pcr_radius_search_batch", "pcr_find_correspondences_batch")
KS = (1, 10, 32, 33, 64)
u32p = lambda a: a.ctypes.data_as(_ffi.u32p)  # noqa: E731
u64p = lambda a: a.ctypes.data_as(_ffi.u64p)  # noqa: E731
f32p = lambda a: a.ctypes.data_as(_ffi.f32p)  # noqa: E731


def _pack(frames):
    off = np.zeros(len(frames) + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in frames])
    pts = np.vstack([np.asarray(f, np.float32).reshape(-1, 3) for f in frames]) if frames else np.zeros((0, 3), np.float32)
    return np.ascontiguousarray(pts, np.float32), off


def _lattice():
    g = np.stack(np.meshgrid(np.arange(12), np.arange(10), np.arange(3), indexing="ij"), -1).reshape(-1, 3)
    return np.ascontiguousarray(g * 0.5, np.float32)


def _mixed():
    """(index frames, query frames): every edge case of the single calls, one frame each."""
    rng = np.random.default_rng(7)
    k0 = scenes.kitti_scene(seed=11, counts=(7_000, 350, 60, 150))
    k1 = scenes.kitti_scene(seed=12, counts=(5_000, 250, 40, 120))
    hemi = scenes.hemisphere(3_000, 5)
    hemi[rng.choice(3_000, 100, replace=False), rng.integers(0, 3, 100)] = np.nan
    lat = _lattice()
    small = scenes.hemisphere(50, 6)  # below the brute-force frame size
    index = [k0, np.zeros((0, 3), np.float32), np.full((40, 3), np.nan, np.float32), np.array([[1.0, 2.0, 3.0]], np.float32), small, lat,
             hemi, k1]

    def near(p, n, s):
        sel = p[rng.choice(len(p), n)]
        return (sel + rng.normal(0.0, s, sel.shape)).astype(np.float32)

    q0 = np.vstack([near(k0, 2_000, 0.05), near(k0, 40, 0.05) + np.float32(300.0),
                    np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf]], np.float32)])
    queries = [
        q0,
        rng.uniform(-5, 5, (10, 3)).astype(np.float32),        # empty index frame
        rng.uniform(-5, 5, (5, 3)).astype(np.float32),         # all-NaN index frame
        np.array([[1.0, 2.0, 3.0], [0, 0, 0], [1e4, 1e4, 1e4], [np.nan, 1, 1]], np.float32),
        near(small, 30, 0.2),
        np.vstack([lat[::7], lat[::11] + np.float32(0.25)]).astype(np.float32),  # exact ties
        np.zeros((0, 3), np.float32),                          # no queries
        np.vstack([near(k1, 1_500, 0.05), near(k1, 60, 1.0) + np.float32([60.0, -80.0, 30.0])]),  # far outside: coarser levels
    ]
    return index, queries


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _per_frame_single(frames, queries, k, ctx):
    """KdTree.knn of every frame alone"""
    return [P.KdTree(P.PointCloud.from_numpy(np.ascontiguousarray(f, np.float32)), ctx=ctx).knn(q, k) for f, q in zip(frames, queries)]


def _split_rows(arr, q_off, f):
    return arr[int(q_off[f]):int(q_off[f + 1])]


# ---- argument checks (no device needed) ------------------------------------------------------------------------

def test_new_symbols_are_declared_and_bound():
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(_ffi.__file__))), "include", "pcr_b200.h")).read()
    lib = _ffi.load()
    for name in NEW_SYMBOLS:
        assert name in _ffi.SIGNATURES and f"{name}(" in header
        assert getattr(lib, name).restype is C.c_int


@pytest.mark.parametrize("offsets", [[0, 6, 4, 10], [1, 4, 10], [0, 4, 11], [0, 4, 9], [], [0.0, 4.0, 10.0], [0]])
def test_bad_index_offsets_raise(offsets):
    with pytest.raises(ValueError):
        P.KdTreeBatch(np.zeros((10, 3), np.float32), offsets)


@pytest.mark.parametrize("points", [np.zeros((10, 2), np.float32), np.zeros(30, np.float32), np.zeros((10, 3, 1), np.float32)])
def test_bad_point_shapes_raise(points):
    with pytest.raises(ValueError):
        P.KdTreeBatch(points, [0, 10])


def _unbuilt(n_frames):
    """A KdTreeBatch without a device index: its query methods must reject bad arguments before reaching the library."""
    t = object.__new__(P.KdTreeBatch)
    t._h, t._off = None, np.zeros(n_frames + 1, np.uint64)
    return t


@pytest.mark.parametrize("q_off", [[0, 4], [0, 2, 2, 4], [0, 3, 1, 4], [1, 2, 4], [0, 2, 5], [0.0, 2.0, 4.0]])
def test_bad_query_offsets_raise(q_off):
    t = _unbuilt(2)
    q = np.zeros((4, 3), np.float32)
    for call in (lambda: t.knn(q, q_off, 3), lambda: t.knn_indices(q, q_off, 3), lambda: t.radius_count(q, q_off, 1.0),
                 lambda: t.radius_search(q, q_off, 1.0), lambda: t.find_correspondences(q, q_off)):
        with pytest.raises(ValueError):
            call()


def test_bad_query_shape_raises():
    t = _unbuilt(1)
    with pytest.raises(ValueError):
        t.knn(np.zeros((4, 2), np.float32), [0, 4], 1)


# ---- GPU ------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def mixed():
    index, queries = _mixed()
    pts, off = _pack(index)
    qpts, q_off = _pack(queries)
    ctx = P.Context()
    tree = P.KdTreeBatch(pts, off, k_hint=10, ctx=ctx)
    yield ctx, index, queries, tree, qpts, q_off
    tree.free()
    ctx.close()


@gpu
@pytest.mark.parametrize("k", KS)
def test_knn_parity_with_single_calls_and_oracle(mixed, k):
    ctx, index, queries, tree, qpts, q_off = mixed
    idx, dist, cnt = tree.knn(qpts, q_off, k)
    i2, c2 = tree.knn_indices(qpts, q_off, k)
    assert np.array_equal(idx, i2) and np.array_equal(cnt, c2)
    single = _per_frame_single(index, queries, k, ctx)
    for f, (si, sd, sc) in enumerate(single):
        bi, bd, bc = (_split_rows(a, q_off, f) for a in (idx, dist, cnt))
        assert np.array_equal(bi, si), f"frame {f}: idx"
        assert np.array_equal(_bits(bd), _bits(sd)), f"frame {f}: dist bits"
        assert np.array_equal(bc, sc), f"frame {f}: counts"
        if len(queries[f]):
            oi, od, oc = O.Tree(index[f]).knn_batch(queries[f], k)
            assert np.array_equal(bi, oi) and np.array_equal(_bits(bd), _bits(od)) and np.array_equal(bc, oc), f"frame {f}: oracle"


@gpu
@pytest.mark.parametrize("r", [0.3, 2.0, 0.0, -1.0, math.nan])
def test_radius_parity_with_single_calls_and_oracle(mixed, r):
    ctx, index, queries, tree, qpts, q_off = mixed
    cnt = tree.radius_count(qpts, q_off, r)
    r_off, r_idx = tree.radius_search(qpts, q_off, r)
    assert np.array_equal(np.diff(r_off.astype(np.int64)), cnt.astype(np.int64))
    for f in range(len(index)):
        single = P.KdTree(P.PointCloud.from_numpy(index[f]), ctx=ctx)
        q = np.ascontiguousarray(queries[f])
        assert np.array_equal(_split_rows(cnt, q_off, f), single.radius_count(q, r)), f"frame {f}: counts"
        s_off, s_idx = single.radius_search(q, r)
        b, e = int(q_off[f]), int(q_off[f + 1])
        assert np.array_equal(r_off[b:e + 1] - r_off[b], s_off), f"frame {f}: CSR offsets"
        assert np.array_equal(r_idx[int(r_off[b]):int(r_off[e])], s_idx), f"frame {f}: CSR indices"
        if len(q):
            ot = O.Tree(index[f])
            assert np.array_equal(_split_rows(cnt, q_off, f), ot.radius_count_batch(q, r)), f"frame {f}: oracle counts"
            for j in range(0, len(q), 97):
                assert np.array_equal(r_idx[int(r_off[b + j]):int(r_off[b + j + 1])], ot.radius_search(q[j], r)), f"frame {f} query {j}"


@gpu
def test_radius_search_capacity_protocol(mixed):
    ctx, index, queries, tree, qpts, q_off = mixed
    lib = _ffi.load()
    x, y, z = (np.ascontiguousarray(qpts[:, j]) for j in range(3))
    nq = len(qpts)
    r_off, total = np.zeros(nq + 1, np.uint64), C.c_size_t()
    small = np.zeros(4, np.uint32)
    st = lib.pcr_radius_search_batch(tree._h, f32p(x), f32p(y), f32p(z), u64p(q_off), tree.n_frames, 2.0, u64p(r_off), u32p(small), 4,
                                     C.byref(total))
    assert st == _ffi.PCR_ERR_CAPACITY and total.value > 4
    full = np.zeros(total.value, np.uint32)
    st = lib.pcr_radius_search_batch(tree._h, f32p(x), f32p(y), f32p(z), u64p(q_off), tree.n_frames, 2.0, u64p(r_off), u32p(full),
                                     total.value, C.byref(total))
    assert st == _ffi.PCR_OK
    e_off, e_idx = tree.radius_search(qpts, q_off, 2.0)
    assert np.array_equal(r_off, e_off) and np.array_equal(full, e_idx)


@gpu
@pytest.mark.parametrize("max_d", [math.inf, 0.5])
def test_correspondences_parity_with_single_calls(mixed, max_d):
    ctx, index, queries, tree, qpts, q_off = mixed
    si, ti, dd, c_off = tree.find_correspondences(qpts, q_off, max_d)
    assert len(c_off) == len(index) + 1 and c_off[0] == 0
    for f in range(len(index)):
        single = P.KdTree(P.PointCloud.from_numpy(index[f]), ctx=ctx)
        a, b, d = single.find_correspondences(P.PointCloud.from_numpy(np.ascontiguousarray(queries[f])), max_d)
        lo, hi = int(c_off[f]), int(c_off[f + 1])
        assert np.array_equal(si[lo:hi], a) and np.array_equal(ti[lo:hi], b), f"frame {f}: pairs"
        assert np.array_equal(_bits(dd[lo:hi]), _bits(d)), f"frame {f}: dist bits"


@gpu
def test_frames_are_independent_and_calls_repeat(mixed):
    ctx, index, queries, tree, qpts, q_off = mixed
    k = 10
    ref = tree.knn(qpts, q_off, k)
    again = tree.knn(qpts, q_off, k)
    assert all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(ref, again))
    for order in (list(range(len(index)))[::-1], [7, 0, 5], [3]):
        pts, off = _pack([index[f] for f in order])
        qp, qo = _pack([queries[f] for f in order])
        t = P.KdTreeBatch(pts, off, ctx=ctx)
        idx, dist, cnt = t.knn(qp, qo, k)
        for j, f in enumerate(order):
            assert np.array_equal(_split_rows(idx, qo, j), _split_rows(ref[0], q_off, f)), f"frame {f} in {order}"
            assert np.array_equal(_bits(_split_rows(dist, qo, j)), _bits(_split_rows(ref[1], q_off, f)))
            assert np.array_equal(_split_rows(cnt, qo, j), _split_rows(ref[2], q_off, f))
        t.free()


@gpu
def test_two_batch_indexes_persist_across_other_calls(mixed):
    ctx, index, queries, tree, qpts, q_off = mixed
    seq = scenes.kitti_sequence(3, seed=3, counts=(6_000, 300, 50, 100))
    s_pts, s_off = _pack(seq)
    other = P.KdTreeBatch(s_pts, s_off, ctx=ctx)
    sq, sq_off = _pack([f[::3] + np.float32(0.02) for f in seq])
    a0 = tree.knn(qpts, q_off, 16)
    b0 = other.knn(sq, sq_off, 16)
    P.estimate_normals_batch(s_pts, s_off, 20, ctx=ctx)  # (transient indexes of the same context in between)
    a1 = tree.knn(qpts, q_off, 16)
    b1 = other.knn(sq, sq_off, 16)
    for x, y in zip(a0 + b0, a1 + b1):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))
    other.free()


@gpu
def test_from_device_frames_equals_numpy_build(mixed):
    ctx, index, queries, tree, qpts, q_off = mixed
    pts, off = _pack(index)
    frames = P.DeviceFrames.from_numpy(pts, off, ctx=ctx)
    t = P.KdTreeBatch.from_device_frames(frames, k_hint=10)
    assert t.n_frames == len(index) and len(t) == len(pts) and np.array_equal(t.offsets, off)
    for k in (1, 33):
        for x, y in zip(t.knn(qpts, q_off, k), tree.knn(qpts, q_off, k)):
            assert np.array_equal(x.view(np.uint32), y.view(np.uint32))
    assert np.array_equal(t.radius_count(qpts, q_off, 0.3), tree.radius_count(qpts, q_off, 0.3))
    t.free()
    frames.free()


@gpu
def test_single_cloud_calls_reject_a_batch_index(mixed):
    ctx, index, queries, tree, qpts, q_off = mixed
    lib = _ffi.load()
    q = np.zeros(3, np.float32)
    idx, dist, cnt = np.zeros(8, np.uint32), np.zeros(8, np.float32), np.zeros(8, np.uint32)
    off, total, m = np.zeros(2, np.uint64), C.c_size_t(), C.c_size_t()
    calls = {
        "pcr_knn_batch": lambda: lib.pcr_knn(tree._h, f32p(q), f32p(q), f32p(q), 1, 1, u32p(idx), f32p(dist), u32p(cnt)),
        "pcr_knn_batch_dev": lambda: lib.pcr_knn_dev(tree._h, None, None, None, 0, 1, None, None, None),
        "pcr_radius_count_batch": lambda: lib.pcr_radius_count(tree._h, f32p(q), f32p(q), f32p(q), 1, 1.0, u32p(cnt)),
        "pcr_radius_search_batch": lambda: lib.pcr_radius_search(tree._h, f32p(q), f32p(q), f32p(q), 1, 1.0, u64p(off), u32p(idx), 8,
                                                                 C.byref(total)),
        "pcr_find_correspondences_batch": lambda: lib.pcr_find_correspondences(tree._h, f32p(q), f32p(q), f32p(q), 1, 1.0, u32p(idx),
                                                                               u32p(cnt), f32p(dist), C.byref(m)),
    }
    for name, call in calls.items():
        assert call() == _ffi.PCR_ERR_INVALID_ARG, name
        assert name in _ffi.last_error(ctx._h), name


@gpu
@pytest.mark.parametrize("k", [1, 10, 33])
def test_batch_of_one_equals_single_call(mixed, k):
    ctx = mixed[0]
    pts = scenes.kitti_scene(seed=21, counts=(9_000, 400, 80, 200))
    q = (pts[::5] + np.float32(0.03)).astype(np.float32)
    t = P.KdTreeBatch(pts, [0, len(pts)], ctx=ctx)
    single = P.KdTree(P.PointCloud.from_numpy(pts), ctx=ctx)
    for x, y in zip(t.knn(q, [0, len(q)], k), single.knn(q, k)):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))
    assert np.array_equal(t.radius_count(q, [0, len(q)], 0.5), single.radius_count(q, 0.5))
    for x, y in zip(t.radius_search(q, [0, len(q)], 0.5), single.radius_search(q, 0.5)):
        assert np.array_equal(x, y)
    t.free()


@gpu
def test_c_error_codes(mixed):
    ctx, index, queries, tree, qpts, q_off = mixed
    lib = _ffi.load()
    x, y, z = (np.ascontiguousarray(qpts[:, j]) for j in range(3))
    nq, nf = len(qpts), tree.n_frames
    idx, dist, cnt = np.zeros(nq * 2, np.uint32), np.zeros(nq * 2, np.float32), np.zeros(nq, np.uint32)

    def knn(h=tree._h, off=q_off, n=nf, k=2, qx=x):
        return lib.pcr_knn_batch(h, f32p(qx) if qx is not None else None, f32p(y), f32p(z), u64p(off) if off is not None else None, n, k,
                                 u32p(idx), f32p(dist), u32p(cnt))

    assert knn() == _ffi.PCR_OK
    assert knn(h=None) == _ffi.PCR_ERR_INVALID_ARG
    assert knn(off=None) == _ffi.PCR_ERR_INVALID_ARG
    assert knn(qx=None) == _ffi.PCR_ERR_INVALID_ARG
    bad = q_off.copy()
    bad[0] = 1
    assert knn(off=bad) == _ffi.PCR_ERR_INVALID_ARG
    assert "query_offsets" in _ffi.last_error(ctx._h)
    bad = q_off.copy()
    bad[2], bad[3] = bad[3], bad[2] - 1
    assert knn(off=bad) == _ffi.PCR_ERR_INVALID_ARG
    assert knn(off=q_off[:-1].copy(), n=nf - 1) == _ffi.PCR_ERR_INVALID_ARG  # frame-count mismatch
    assert knn(k=_ffi.PCR_MAX_K + 1) == _ffi.PCR_ERR_UNSUPPORTED
    assert lib.pcr_radius_count_batch(tree._h, f32p(x), f32p(y), f32p(z), u64p(q_off), nf + 1, 1.0, u32p(cnt)) == _ffi.PCR_ERR_INVALID_ARG
    c_off = np.zeros(nf + 1, np.uint64)
    assert lib.pcr_find_correspondences_batch(tree._h, f32p(x), f32p(y), f32p(z), u64p(q_off), nf, 1.0, None, u32p(cnt), f32p(dist),
                                              u64p(c_off)) == _ffi.PCR_ERR_INVALID_ARG
    h = C.c_void_p()
    off0 = np.zeros(1, np.uint64)
    assert lib.pcr_index_build_batch(ctx._h, f32p(x), f32p(y), f32p(z), u64p(off0), 0, 0, C.byref(h)) == _ffi.PCR_ERR_INVALID_ARG
    assert lib.pcr_index_build_batch(ctx._h, None, None, None, u64p(np.array([0, 3], np.uint64)), 1, 0, C.byref(h)) == _ffi.PCR_ERR_INVALID_ARG
    assert not h.value


@gpu
@pytest.mark.parametrize("k", [1, 10])
def test_kitti_sequence_against_single_calls(k):
    ctx = P.Context()
    seq = scenes.kitti_sequence(8)
    pts, off = _pack(seq)
    vox, v_off = P.voxel_downsample_batch(pts, off, 0.2, ctx=ctx)
    frames = [vox[int(v_off[f]):int(v_off[f + 1])] for f in range(8)]
    i_pts, i_off = _pack(frames[:7])
    q_pts, q_off = _pack(frames[1:])
    t = P.KdTreeBatch(i_pts, i_off, k_hint=k, ctx=ctx)
    idx, dist, cnt = t.knn(q_pts, q_off, k)
    for f in range(7):
        si, sd, sc = P.KdTree(P.PointCloud.from_numpy(np.ascontiguousarray(frames[f])), ctx=ctx).knn(frames[f + 1], k)
        assert np.array_equal(_split_rows(idx, q_off, f), si), f"frame {f}"
        assert np.array_equal(_bits(_split_rows(dist, q_off, f)), _bits(sd)) and np.array_equal(_split_rows(cnt, q_off, f), sc)
    t.free()
    ctx.close()
