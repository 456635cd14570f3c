"""Device-resident frame batches (pcr_frames / DeviceFrames) and the batched radius outlier filter
(pcr_radius_outlier_batch): a pipeline over many frames as one upload, a chain of batch calls and one download.

CPU tests: the Python layer rejects bad arguments (ValueError; IndexError naming the frame of an index outside it) before
it touches a device.
GPU tests: every DeviceFrames filter and select / select_inverse equal, frame by frame and bit for bit, to the DeviceCloud
method on that frame alone, on a mixed batch (KITTI frames, empty, one-point, all-NaN and NaN-mixed frames, two identical
frames back to back), with and without normals carried; the batched radius filter against the oracle and the single call;
RANSAC with outliers, clustering and ICP against the raw batch calls; the obstacle pipeline and the odometry front end over
8 frames; independence of the other frames; the C error codes.
"""
import ctypes as C

import numpy as np
import pytest

import pointclouds_rs_b200 as P
from pointclouds_rs_b200 import _ffi, scenes
from oracle import oracle as O

gpu = pytest.mark.gpu


def _pack(frames):
    off = np.zeros(len(frames) + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in frames])
    pts = np.vstack([np.asarray(f, np.float32).reshape(-1, 3) for f in frames]) if frames else np.zeros((0, 3), np.float32)
    return np.ascontiguousarray(pts, np.float32), off


def _icp_bits(r):
    return (np.float32(r.rotation).tobytes(), np.float32(r.translation).tobytes(), np.float32(r.rmse).tobytes(),
            np.float32(r.fitness).tobytes(), r.num_iterations, r.converged)


def _mixed():
    """KITTI frames, the edge cases of the single calls, and two identical frames back to back (shared cells)."""
    rng = np.random.default_rng(5)
    k0 = scenes.kitti_scene(seed=11, counts=(7_000, 350, 60, 150))
    nan_mixed = scenes.hemisphere(500, 3)
    nan_mixed[rng.choice(500, 60, replace=False), rng.integers(0, 3, 60)] = np.nan
    nan_mixed[::97, 0] = np.inf
    return [
        k0,
        np.zeros((0, 3), np.float32),
        np.array([[1.0, 2.0, 3.0]], np.float32),
        np.full((40, 3), np.nan, np.float32),
        nan_mixed,
        scenes.hemisphere(800, 9),
        scenes.hemisphere(800, 9),
        np.array([[np.nan, 0.0, 0.0]], np.float32),
        scenes.kitti_scene(seed=12, counts=(5_000, 250, 40, 120)),
    ]


def _frames_equal(batch, clouds):
    """batch: DeviceFrames; clouds: one DeviceCloud per frame.  Coordinates and normals, bit for bit."""
    pts, off = batch.to_numpy()
    nrm = batch.normals_to_numpy()
    assert len(off) == len(clouds) + 1
    for f, cl in enumerate(clouds):
        b, e = int(off[f]), int(off[f + 1])
        assert pts[b:e].tobytes() == cl.to_numpy().tobytes(), f"frame {f}: points"
        if e > b:
            assert batch.has_normals() == cl.has_normals(), f"frame {f}: normals flag"
        if nrm is not None and e > b:
            assert nrm[b:e].tobytes() == cl.normals_to_numpy().tobytes(), f"frame {f}: normals"


# ---- argument checks (no device needed) ------------------------------------------------------------------------

@pytest.mark.parametrize("offsets", [[0, 6, 4, 10], [1, 4, 10], [0, 4, 11], [0, 4, 9], [], [0.0, 4.0, 10.0]])
def test_bad_offsets_raise(offsets):
    pts = np.zeros((10, 3), np.float32)
    with pytest.raises(ValueError):
        P.DeviceFrames.from_numpy(pts, offsets)
    with pytest.raises(ValueError):
        P.radius_outlier_removal_batch(pts, offsets, 1.0, 2)


def test_no_frame_raises():
    with pytest.raises(ValueError):
        P.DeviceFrames.from_numpy(np.zeros((0, 3), np.float32), [0])


@pytest.mark.parametrize("shape", [(10, 2), (30,), (2, 5, 3), (10, 4)])
def test_bad_point_shape_raises(shape):
    pts = np.zeros(shape, np.float32)
    with pytest.raises(ValueError):
        P.DeviceFrames.from_numpy(pts, [0, 4, 10])
    with pytest.raises(ValueError):
        P.radius_outlier_removal_batch(pts, [0, 4, 10], 1.0, 2)


@pytest.mark.parametrize("radius", [0.0, -1.0, float("nan"), float("inf")])
def test_bad_radius_raises(radius):
    with pytest.raises(ValueError):
        P.radius_outlier_removal_batch(np.zeros((10, 3), np.float32), [0, 4, 10], radius, 2)


def test_frame_lists_checked_on_the_host():
    off = np.array([0, 4, 4, 10], np.uint64)
    idx, l_off = P._frame_lists([[3, 0, 3], [], np.array([5, 1], np.int64)], off)
    assert idx.tolist() == [3, 0, 3, 5, 1] and l_off.tolist() == [0, 3, 3, 5]
    for bad in ([[0]], [[0], [], [0], [1]], "abc", None, [[[0]], [], []], [[0.5], [], []]):
        with pytest.raises(ValueError):
            P._frame_lists(bad, off)
    with pytest.raises(IndexError, match="frame 0"):
        P._frame_lists([[4], [], []], off)
    with pytest.raises(IndexError, match="frame 1"):
        P._frame_lists([[0], [0], []], off)
    with pytest.raises(IndexError, match="frame 2"):
        P._frame_lists([[0], [], [-1]], off)


# ---- GPU: filters and selection against the single-frame DeviceCloud --------------------------------------------

@pytest.fixture(scope="module")
def mixed(pcr):
    frames = _mixed()
    pts, off = _pack(frames)
    return frames, P.DeviceFrames.from_numpy(pts, off)


@gpu
def test_upload_download_and_frames(mixed):
    frames, batch = mixed
    pts, off = _pack(frames)
    got, got_off = batch.to_numpy()
    assert got.tobytes() == pts.tobytes() and np.array_equal(got_off, off)
    assert batch.n_frames == len(frames) and len(batch) == len(pts) and not batch.has_normals()
    for f, fr in enumerate(frames):
        assert batch.frame(f).to_numpy().tobytes() == fr.tobytes()
    with pytest.raises(IndexError):
        batch.frame(len(frames))


@gpu
@pytest.mark.parametrize("with_normals", [False, True])
def test_filters_equal_single_calls(mixed, with_normals):
    frames, batch = mixed
    if with_normals:
        batch = batch.estimate_normals(10, (0.5, -1.0, 2.0))
    singles = [batch.frame(f) for f in range(len(frames))]
    _frames_equal(batch, singles)
    _frames_equal(batch.voxel_downsample(0.3), [c.voxel_downsample(0.3) for c in singles])
    for k, s in ((8, 1.0), (20, 2.0), (0, 1.0)):
        _frames_equal(batch.statistical_outlier_removal(k, s), [c.statistical_outlier_removal(k, s) for c in singles])
    for r, m in ((0.5, 5), (2.0, 1), (0.3, 0)):
        _frames_equal(batch.radius_outlier_removal(r, m), [c.radius_outlier_removal(r, m) for c in singles])
    _frames_equal(batch.estimate_normals(15), [c.estimate_normals(15) for c in singles])
    _frames_equal(batch.sor_normals(10, 1.5, 12, (0.0, 0.0, 1.5)), [c.sor_normals(10, 1.5, 12, (0.0, 0.0, 1.5)) for c in singles])


@gpu
@pytest.mark.parametrize("with_normals", [False, True])
def test_select_equals_single_calls(mixed, with_normals):
    frames, batch = mixed
    if with_normals:
        batch = batch.estimate_normals(8)
    rng = np.random.default_rng(2)
    lists = [rng.integers(0, len(fr), rng.integers(0, 2 * len(fr) + 1)) if len(fr) else np.zeros(0, np.int64) for fr in frames]
    lists[5] = np.array([3, 3, 0, 799, 3], np.int64)  # order and duplicates kept
    singles = [batch.frame(f) for f in range(len(frames))]
    _frames_equal(batch.select(lists), [c.select(l) for c, l in zip(singles, lists)])
    inv = batch.select_inverse(lists)
    for f, (fr, l) in enumerate(zip(frames, lists)):
        rest = np.setdiff1d(np.arange(len(fr)), l)
        ref = singles[f].select(rest)
        b, e = int(inv.offsets[f]), int(inv.offsets[f + 1])
        assert inv.to_numpy()[0][b:e].tobytes() == ref.to_numpy().tobytes(), f"frame {f}"
        assert P.PointCloud.from_numpy(fr).select_inverse(l).to_numpy().tobytes() == ref.to_numpy().tobytes()
    with pytest.raises(IndexError, match="frame 2"):
        batch.select([[], [], [1], [], [], [], [], [], []])


# ---- GPU: batched radius outlier removal --------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("radius", [0.4, 2.0])
def test_radius_batch_against_oracle_and_single(pcr, radius):
    frames = _mixed()
    pts, off = _pack(frames)
    for m in (0, 1, 5, 10_000):
        keep, kept = pcr.radius_outlier_removal_batch(pts, off, radius, m)
        for f, fr in enumerate(frames):
            b, e = int(off[f]), int(off[f + 1])
            ref = O.ror(fr, radius, m)
            single, n_single = pcr.ror_mask(pcr.PointCloud.from_numpy(fr), radius, m) if len(fr) else (np.zeros(0, np.uint8), 0)
            assert np.array_equal(keep[b:e], ref), f"frame {f}, min_neighbors {m}"
            assert np.array_equal(keep[b:e], single) and int(kept[f]) == n_single


@gpu
@pytest.mark.parametrize("radius", [0.0, -1.0, float("nan")])
def test_radius_batch_nonpositive_radius(pcr, radius):
    """radius <= 0 or not finite: every count is 0, a point is kept iff min_neighbors == 0 (as the single call)."""
    pts, off = _pack(_mixed())
    lib, h = _ffi.load(), pcr.default_context()._h
    x, y, z = (np.ascontiguousarray(pts[:, j]) for j in range(3))
    for m in (0, 1):
        keep = np.full(len(pts), 7, np.uint8)
        kept = np.zeros(len(off) - 1, np.uint64)
        st = lib.pcr_radius_outlier_batch(h, x.ctypes.data_as(_ffi.f32p), y.ctypes.data_as(_ffi.f32p), z.ctypes.data_as(_ffi.f32p),
                                          off.ctypes.data_as(_ffi.u64p), len(off) - 1, radius, m, keep.ctypes.data_as(_ffi.u8p),
                                          kept.ctypes.data_as(_ffi.u64p))
        assert st == _ffi.PCR_OK
        assert np.all(keep == (1 if m == 0 else 0))
        assert np.array_equal(kept, np.diff(off) if m == 0 else np.zeros_like(kept))


@gpu
def test_radius_batch_aerial_tiles(pcr):
    tiles = [scenes.aerial_scene(seed=s, scale=0.02) for s in range(4)]
    pts, off = _pack(tiles)
    keep, kept = pcr.radius_outlier_removal_batch(pts, off, 2.0, 5)
    batch = P.DeviceFrames.from_numpy(pts, off).radius_outlier_removal(2.0, 5)
    got, g_off = batch.to_numpy()
    for f, t in enumerate(tiles):
        ref = O.ror(t, 2.0, 5)
        assert np.array_equal(keep[int(off[f]):int(off[f + 1])], ref) and int(kept[f]) == int(ref.sum())
        assert got[int(g_off[f]):int(g_off[f + 1])].tobytes() == t[ref.astype(bool)].tobytes()


# ---- GPU: RANSAC, clustering, ICP against the raw batch calls -----------------------------------------------------

@gpu
def test_ransac_with_outliers(mixed):
    frames, batch = mixed
    pts, off = _pack(frames)
    triples = [P.draw_plane_samples(len(fr), 200, [7, f]) for f, fr in enumerate(frames)]
    res, outl = batch.ransac_plane_samples(0.1, triples, outliers=True)
    models, inl, inl_off = P.ransac_plane_samples_batch(pts, off, 0.1, triples)
    o_pts, o_off = outl.to_numpy()
    for f, fr in enumerate(frames):
        assert np.float32(res[f].normal + [res[f].d]).tobytes() == models[f].tobytes(), f"frame {f}"
        assert res[f].inliers == inl[int(inl_off[f]):int(inl_off[f + 1])].tolist(), f"frame {f}"
        ref = P.PointCloud.from_numpy(fr).select_inverse(res[f].inliers).to_numpy()
        assert o_pts[int(o_off[f]):int(o_off[f + 1])].tobytes() == ref.tobytes(), f"frame {f}"
    assert [r.inliers for r in batch.ransac_plane_samples(0.1, triples)] == [r.inliers for r in res]
    seeded = batch.ransac_plane(0.1, 50, seed=3)
    ref_models, _, _ = P.ransac_plane_batch(pts, off, 0.1, 50, seed=3)
    assert np.float32([r.normal + [r.d] for r in seeded]).tobytes() == ref_models.tobytes()


@gpu
def test_cluster_equals_batch_call(mixed):
    frames, batch = mixed
    pts, off = _pack(frames)
    for thr, lo, hi in ((0.5, 1, 100_000), (1.0, 10, 400), (0.0, 1, 10)):
        assert batch.euclidean_cluster(thr, lo, hi) == P.euclidean_cluster_batch(pts, off, thr, lo, hi)


@gpu
def test_icp_equals_batch_call(pcr):
    seq = scenes.kitti_sequence(4, seed=8, counts=(8_800, 440, 70, 250))
    pts, off = _pack(seq)
    pairs = np.array([(1, 0), (2, 1), (3, 2), (0, 3), (2, 2)], np.uint32)
    kw = dict(max_iterations=20, tolerance=0.0)
    batch = P.DeviceFrames.from_numpy(pts, off)
    assert [_icp_bits(r) for r in batch.icp_point_to_point(pairs, **kw)] == \
        [_icp_bits(r) for r in pcr.icp_point_to_point_batch(pts, off, pairs, **kw)]
    with_n = batch.estimate_normals(12)
    nrm = pcr.estimate_normals_batch(pts, off, 12)
    assert [_icp_bits(r) for r in with_n.icp_point_to_plane(pairs, **kw)] == \
        [_icp_bits(r) for r in pcr.icp_point_to_plane_batch(pts, off, pairs, nrm, **kw)]
    with pytest.raises(ValueError):
        batch.icp_point_to_plane(pairs)
    with pytest.raises(ValueError):
        batch.icp_point_to_point([(0, 4)])


# ---- GPU: whole pipelines ---------------------------------------------------------------------------------------

@gpu
def test_obstacle_pipeline(pcr):
    """upload -> voxel 0.15 -> SOR (20, 2.0) -> RANSAC 0.15 with outliers -> cluster (0.8, 10, 20000) over 8 frames: the
    frame-by-frame single calls' clusters."""
    frames = [scenes.kitti_scene(seed=40 + s, counts=scenes.KITTI_COUNTS["frame80k"]) for s in range(8)]
    pts, off = _pack(frames)
    s = P.DeviceFrames.from_numpy(pts, off).voxel_downsample(0.15).statistical_outlier_removal(20, 2.0)
    s_off = s.offsets
    triples = [P.draw_plane_samples(int(s_off[f + 1] - s_off[f]), 500, [99, f]) for f in range(len(frames))]
    planes, rest = s.ransac_plane_samples(0.15, triples, outliers=True)
    batched = rest.euclidean_cluster(0.8, 10, 20_000)
    for f, fr in enumerate(frames):
        v = pcr.voxel_downsample(pcr.PointCloud.from_numpy(fr), 0.15)
        sc = pcr.statistical_outlier_removal(v, 20, 2.0)
        r = pcr.ransac_plane_samples(sc, 0.15, triples[f])
        assert np.float32(r.normal + [r.d]).tobytes() == np.float32(planes[f].normal + [planes[f].d]).tobytes(), f"frame {f}"
        assert batched[f] == pcr.euclidean_cluster(sc.select_inverse(r.inliers), 0.8, 10, 20_000), f"frame {f}"
    assert sum(len(c) for c in batched) > 0


@gpu
def test_odometry_front_end(pcr):
    """voxel 0.2 -> normals 15 -> point-to-plane ICP over consecutive pairs: the bits of the three raw batch calls."""
    seq = scenes.kitti_sequence(8, seed=3, counts=(17_600, 880, 145, 495))
    pts, off = _pack(seq)
    pairs = np.array([(i + 1, i) for i in range(len(seq) - 1)], np.uint32)
    kw = dict(max_iterations=30, tolerance=0.0)
    chained = P.DeviceFrames.from_numpy(pts, off).voxel_downsample(0.2).estimate_normals(15).icp_point_to_plane(pairs, **kw)
    vox, v_off = pcr.voxel_downsample_batch(pts, off, 0.2)
    nrm = pcr.estimate_normals_batch(vox, v_off, 15)
    raw = pcr.icp_point_to_plane_batch(vox, v_off, pairs, nrm, **kw)
    assert [_icp_bits(r) for r in chained] == [_icp_bits(r) for r in raw]


@gpu
def test_independence_and_repeatability(pcr):
    frames = _mixed()
    perm = np.random.default_rng(4).permutation(len(frames))

    def run(frs):
        b = P.DeviceFrames.from_numpy(*_pack(frs)).sor_normals(10, 1.5, 12).radius_outlier_removal(0.6, 3)
        pts, off = b.to_numpy()
        nrm = b.normals_to_numpy()
        return [(pts[int(off[f]):int(off[f + 1])].tobytes(), nrm[int(off[f]):int(off[f + 1])].tobytes()) for f in range(len(frs))]

    base = run(frames)
    assert run(frames) == base
    permuted = run([frames[i] for i in perm])
    assert [permuted[j] for j in np.argsort(perm)] == base


# ---- GPU: C error codes -----------------------------------------------------------------------------------------

@gpu
def test_errors(pcr):
    pts, off = _pack([scenes.hemisphere(300, 1), scenes.hemisphere(200, 2)])
    lib, h = _ffi.load(), pcr.default_context()._h
    x, y, z = (np.ascontiguousarray(pts[:, j]) for j in range(3))
    u32 = lambda a: a.ctypes.data_as(_ffi.u32p)
    u64 = lambda a: a.ctypes.data_as(_ffi.u64p)
    out = C.c_void_p(1234)
    assert lib.pcr_frames_upload(None, x.ctypes.data, y.ctypes.data, z.ctypes.data, u64(off), 2, C.byref(out)) == _ffi.PCR_ERR_INVALID_ARG
    assert lib.pcr_frames_upload(h, x.ctypes.data, y.ctypes.data, z.ctypes.data, u64(off), 2, None) == _ffi.PCR_ERR_INVALID_ARG
    bad = np.array([0, 400, 300], np.uint64)
    out = C.c_void_p(1234)
    assert lib.pcr_frames_upload(h, x.ctypes.data, y.ctypes.data, z.ctypes.data, u64(bad), 2, C.byref(out)) == _ffi.PCR_ERR_INVALID_ARG
    assert out.value is None
    fr = C.c_void_p()
    assert lib.pcr_frames_upload(h, x.ctypes.data, y.ctypes.data, z.ctypes.data, u64(off), 2, C.byref(fr)) == _ffi.PCR_OK
    try:
        assert lib.pcr_frames_count(fr) == 2 and lib.pcr_frames_len(fr) == 500
        got = np.zeros(3, np.uint64)
        assert lib.pcr_frames_offsets(fr, u64(got)) == _ffi.PCR_OK and np.array_equal(got, off)
        # a select index outside its frame: the message names the frame and the index, and no handle comes back
        idx = np.array([5, 250], np.uint32)
        i_off = np.array([0, 1, 2], np.uint64)
        sel = C.c_void_p(1234)
        assert lib.pcr_frames_select(fr, u32(idx), u64(i_off), 0, C.byref(sel)) == _ffi.PCR_ERR_INVALID_ARG
        assert sel.value is None
        assert "frame 1" in _ffi.last_error(h) and "250" in _ffi.last_error(h)
        assert lib.pcr_frames_select(fr, u32(idx), u64(i_off), 1, C.byref(sel)) == _ffi.PCR_ERR_INVALID_ARG
        assert lib.pcr_frames_select(None, u32(idx), u64(i_off), 0, C.byref(sel)) == _ffi.PCR_ERR_INVALID_ARG
        assert lib.pcr_frames_select(fr, u32(idx), u64(i_off), 0, None) == _ffi.PCR_ERR_INVALID_ARG
        # frame id >= F
        cl = C.c_void_p(1234)
        assert lib.pcr_frames_frame(fr, 2, C.byref(cl)) == _ffi.PCR_ERR_INVALID_ARG and cl.value is None
        assert lib.pcr_frames_frame(None, 0, C.byref(cl)) == _ffi.PCR_ERR_INVALID_ARG
        # the pcr_cloud filters hand out no handle on failure either
        assert lib.pcr_frames_frame(fr, 0, C.byref(cl)) == _ffi.PCR_OK
        try:
            outside = np.array([300], np.uint32)
            for call in (lambda o: lib.pcr_cloud_select(cl, u32(outside), 1, o),
                         lambda o: lib.pcr_cloud_voxel_downsample(cl, 0.0, o),
                         lambda o: lib.pcr_cloud_statistical_outlier_removal(cl, 10, -1.0, o),
                         lambda o: lib.pcr_cloud_estimate_normals(cl, 0, None, o),
                         lambda o: lib.pcr_cloud_sor_normals(cl, 10, 1.0, 0, None, o)):
                o = C.c_void_p(1234)
                assert call(C.byref(o)) == _ffi.PCR_ERR_INVALID_ARG and o.value is None
        finally:
            lib.pcr_cloud_free(cl)
        # ICP: a pair outside [0, F), point-to-plane without normals
        prm = _ffi.IcpParams(10, 1e-5, float("inf"))
        res = (_ffi.IcpResultC * 1)()
        pr = np.array([[0, 2]], np.uint32)
        assert lib.pcr_frames_icp_point_to_point(fr, u32(pr), 1, C.byref(prm), res) == _ffi.PCR_ERR_INVALID_ARG
        ok = np.array([[1, 0]], np.uint32)
        assert lib.pcr_frames_icp_point_to_plane(fr, u32(ok), 1, C.byref(prm), res) == _ffi.PCR_ERR_INVALID_ARG
        assert lib.pcr_frames_icp_point_to_point(fr, u32(ok), 1, C.byref(prm), res) == _ffi.PCR_OK
        # filters: NULL out, bad parameters; no handle on failure
        for call in (lambda o: lib.pcr_frames_voxel_downsample(fr, 0.0, o),
                     lambda o: lib.pcr_frames_statistical_outlier_removal(fr, 10, -1.0, o),
                     lambda o: lib.pcr_frames_estimate_normals(fr, 0, None, o),
                     lambda o: lib.pcr_frames_sor_normals(fr, 10, 1.0, 0, None, o)):
            o = C.c_void_p(1234)
            assert call(C.byref(o)) == _ffi.PCR_ERR_INVALID_ARG and o.value is None
        assert lib.pcr_frames_radius_outlier_removal(fr, 1.0, 2, None) == _ffi.PCR_ERR_INVALID_ARG
        assert lib.pcr_frames_voxel_downsample(None, 0.1, C.byref(C.c_void_p())) == _ffi.PCR_ERR_INVALID_ARG
        assert lib.pcr_frames_download(fr, x.ctypes.data, y.ctypes.data, z.ctypes.data, x.ctypes.data, y.ctypes.data,
                                       z.ctypes.data) == _ffi.PCR_ERR_INVALID_ARG  # no normals
    finally:
        lib.pcr_frames_free(fr)
    keep = np.zeros(len(pts), np.uint8)
    f = lambda a: a.ctypes.data_as(_ffi.f32p)
    assert lib.pcr_radius_outlier_batch(h, f(x), f(y), f(z), u64(bad), 2, 1.0, 2, keep.ctypes.data_as(_ffi.u8p), None) == _ffi.PCR_ERR_INVALID_ARG
    assert lib.pcr_radius_outlier_batch(h, f(x), f(y), f(z), None, 2, 1.0, 2, keep.ctypes.data_as(_ffi.u8p), None) == _ffi.PCR_ERR_INVALID_ARG
