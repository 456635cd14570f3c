"""Batched RANSAC plane fit and euclidean_cluster (pcr_ransac_plane_samples_batch, pcr_euclidean_cluster_batch): the back
end of the obstacle pipeline over many frames of one buffer, every frame processed as if it were alone.

CPU tests: the Python layer rejects bad arguments (ValueError, IndexError for a triple outside its frame) before it
touches a device.
GPU tests: every cluster frame equal to the oracle and to the single call, through the edge cases of the single call;
frames that share their cells kept apart; the size filter and the threshold edge cases; raw KITTI frames with the ground
left in; a frame's clusters independent of the other frames, of their order, of repetition and of the entry point;
every RANSAC frame bit-exact against the oracle and the single call on both choice paths; the whole obstacle pipeline
over 8 frames equal to the frame-by-frame way; the C error codes.
"""
import ctypes as C
import math

import numpy as np
import pytest

import pointclouds_rs_b200 as P
from pointclouds_rs_b200 import _ffi, scenes

gpu = pytest.mark.gpu


def _pack(frames):
    off = np.zeros(len(frames) + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in frames])
    pts = np.vstack([np.asarray(f, np.float32).reshape(-1, 3) for f in frames]) if frames else np.zeros((0, 3), np.float32)
    return np.ascontiguousarray(pts, np.float32), off


def _cloud(pts):
    return P.PointCloud.from_numpy(np.ascontiguousarray(pts, np.float32))


def _lists(clusters):
    return [list(map(int, c)) for c in clusters]


def _grid_plane(nx, ny, step, zfn):
    i, j = np.meshgrid(np.arange(nx, dtype=np.float32), np.arange(ny, dtype=np.float32), indexing="ij")
    x, y = (i * np.float32(step)).ravel(), (j * np.float32(step)).ravel()
    return np.stack([x, y, zfn(x, y).astype(np.float32)], 1).astype(np.float32)


# ---- argument checks (no device needed) ------------------------------------------------------------------------

@pytest.mark.parametrize("offsets", [[0, 6, 4, 10], [1, 4, 10], [0, 4, 11], [0, 4, 9], [], [0.0, 4.0, 10.0]])
def test_bad_offsets_raise(offsets):
    pts = np.zeros((10, 3), np.float32)
    with pytest.raises(ValueError):
        P.ransac_plane_samples_batch(pts, offsets, 0.1, [np.zeros((0, 3), np.uint32)] * max(len(offsets) - 1, 0))
    with pytest.raises(ValueError):
        P.ransac_plane_batch(pts, offsets, 0.1, 10, seed=1)
    with pytest.raises(ValueError):
        P.cluster_arrays_batch(pts, offsets, 0.5, 1, 10)
    with pytest.raises(ValueError):
        P.euclidean_cluster_batch(pts, offsets, 0.5, 1, 10)


@pytest.mark.parametrize("shape", [(10, 2), (30,), (2, 5, 3), (10, 4)])
def test_bad_point_shape_raises(shape):
    pts = np.zeros(shape, np.float32)
    with pytest.raises(ValueError):
        P.ransac_plane_samples_batch(pts, [0, 4, 10], 0.1, [[[0, 1, 2]], [[0, 1, 2]]])
    with pytest.raises(ValueError):
        P.ransac_plane_batch(pts, [0, 4, 10], 0.1, 10)
    with pytest.raises(ValueError):
        P.euclidean_cluster_batch(pts, [0, 4, 10], 0.5, 1, 10)


@pytest.mark.parametrize("samples", [
    [[[0, 1, 2]]],                                        # one array for two frames
    [[[0, 1, 2]], [[0, 1, 2]], [[0, 1, 2]]],              # three arrays for two frames
    [[[0, 1]], [[0, 1, 2]]],                              # (m, 2)
    [[0, 1, 2], [[0, 1, 2]]],                             # (3,)
    [[[[0, 1, 2]]], [[0, 1, 2]]],                         # (1, 1, 3)
    [np.array([[0.0, 1.0, 2.0]]), [[0, 1, 2]]],           # float triples
    "abc",
    None,
])
def test_bad_sample_lists_raise(samples):
    pts = np.zeros((10, 3), np.float32)
    with pytest.raises(ValueError):
        P.ransac_plane_samples_batch(pts, [0, 4, 10], 0.1, samples)


@pytest.mark.parametrize("bad", [[[0, 1, 4]], [[4, 1, 2]], [[0, -1, 2]]])
def test_triples_outside_their_frame_raise(bad):
    """Frame-local: index 4 exists in the buffer (10 points) but not in the 4-point frame 0."""
    pts = np.zeros((10, 3), np.float32)
    with pytest.raises(IndexError):
        P.ransac_plane_samples_batch(pts, [0, 4, 10], 0.1, [bad, [[0, 1, 5]]])
    with pytest.raises(IndexError):
        P.ransac_plane_samples_batch(pts, [0, 6, 10], 0.1, [[[0, 1, 5]], bad])  # frame 1 holds 4 points


# ---- GPU: clustering --------------------------------------------------------------------------------------------

THR = 1.0


def _cluster_frames():
    """The edge cases of the single call at one threshold (1.0), with random clouds between them."""
    rng = np.random.default_rng(5)
    n = 5000
    line = np.stack([np.arange(n, dtype=np.float32) * np.float32(1e-4), np.zeros(n), np.zeros(n)], 1)  # a few dense cells
    lattice = np.stack(np.meshgrid(*[np.arange(9, dtype=np.float32)] * 3, indexing="ij"), -1).reshape(-1, 3)
    mixed = scenes.uniform_cube(3000, 11, 0, 25)
    mixed[::29, 0] = np.nan
    mixed[7::53, 2] = np.inf
    mixed[11::71, 1] = -np.inf
    return [np.ascontiguousarray(f, np.float32) for f in (
        scenes.uniform_cube(4000, 1, 0, 30),
        np.zeros((0, 3)),                                                        # empty
        np.array([[1.0, 2.0, 3.0]]),                                             # one point
        np.full((6, 3), np.nan),                                                 # nothing finite
        mixed,                                                                   # NaN and inf mixed in
        line,                                                                    # the 5 000-point dense line
        lattice,                                                                 # d == r between lattice neighbours
        lattice * np.float32(1.0 / 0.999),                                       # d just above r: singletons
        np.zeros((0, 3)),
        np.repeat(scenes.uniform_cube(300, 9, 0, 10), 5, axis=0),               # duplicates
        np.vstack([scenes.uniform_cube(2000, 3, 0, 10), [[3e6, -2e6, 1e6]]]),    # a far outlier
        np.array([[0, 0, 0], [3e9, 3e9, 3e9], [3.1e9, 3e9, 3e9], [-4e12, 0, 0]]),  # saturated i32 keys
        np.array([[5.0, 5.0, 5.0]]),
        rng.normal(0, 3, (6000, 3)),
        scenes.kitti_scene(2, (9_000, 400, 80, 200)),
    )]


@pytest.fixture(scope="module")
def cluster_frames():
    return _cluster_frames()


def _check_csr(c_off, offsets, idx, n_frames):
    assert c_off.dtype == np.uint64 and offsets.dtype == np.uint32 and idx.dtype == np.uint32
    assert len(c_off) == n_frames + 1 and c_off[0] == 0 and np.all(np.diff(c_off.astype(np.int64)) >= 0)
    assert len(offsets) == int(c_off[-1]) + 1 and offsets[0] == 0 and int(offsets[-1]) == len(idx)


@gpu
def test_cluster_batch_matches_oracle_and_single(pcr, oracle, cluster_frames):
    pts, off = _pack(cluster_frames)
    mx = len(pts)
    c_off, offsets, idx = pcr.cluster_arrays_batch(pts, off, THR, 1, mx)
    _check_csr(c_off, offsets, idx, len(cluster_frames))
    got = pcr.euclidean_cluster_batch(pts, off, THR, 1, mx)
    assert len(got) == len(cluster_frames)
    for f, fr in enumerate(cluster_frames):
        want = _lists(oracle.euclidean_cluster(fr, THR, 1, mx))
        assert got[f] == want, f"frame {f}"
        assert pcr.euclidean_cluster(_cloud(fr), THR, 1, mx) == want, f"frame {f}"
        s_off, s_idx = pcr.cluster_arrays(_cloud(fr), THR, 1, mx)
        a, b = int(c_off[f]), int(c_off[f + 1])
        assert np.array_equal(offsets[a:b + 1] - offsets[a], s_off), f"frame {f}"
        assert np.array_equal(idx[offsets[a]:offsets[b]], s_idx), f"frame {f}"


@gpu
def test_cluster_frames_sharing_cells_stay_apart(pcr, oracle):
    fr = scenes.uniform_cube(3000, 21, 0, 12)
    pts, off = _pack([fr, fr, fr[:1000]])
    want = _lists(oracle.euclidean_cluster(fr, 0.6, 1, 10_000))
    got = pcr.euclidean_cluster_batch(pts, off, 0.6, 1, 10_000)
    assert got[0] == want and got[1] == want
    assert got[2] == _lists(oracle.euclidean_cluster(fr[:1000], 0.6, 1, 10_000))
    c_off, offsets, _ = pcr.cluster_arrays_batch(pts, off, 0.6, 1, 10_000)
    assert int(c_off[2] - c_off[1]) == int(c_off[1]) == len(want)


@gpu
def test_cluster_size_filter_and_thresholds(pcr, oracle, cluster_frames):
    frames = cluster_frames
    pts, off = _pack(frames)
    for mn, mx in ((1, 1), (2, 50), (10, 20_000), (100, 10**12), (10**6, 10**7), (7, 3)):
        got = pcr.euclidean_cluster_batch(pts, off, THR, mn, mx)
        for f, fr in enumerate(frames):
            assert got[f] == _lists(oracle.euclidean_cluster(fr, THR, mn, mx)), (mn, mx, f)
    for thr, mn in ((0.0, 1), (-1.0, 1), (THR, 0)):
        c_off, offsets, idx = pcr.cluster_arrays_batch(pts, off, thr, mn, 100)
        assert not c_off.any() and offsets.tolist() == [0] and len(idx) == 0
    nan_got = pcr.euclidean_cluster_batch(pts, off, math.nan, 1, len(pts))  # the kernels see it, as in the single call
    for f, fr in enumerate(frames):
        assert nan_got[f] == pcr.euclidean_cluster(_cloud(fr), math.nan, 1, len(pts)), f"frame {f}"
    empty, e_off = _pack([np.zeros((0, 3), np.float32)] * 3)
    c_off, offsets, idx = pcr.cluster_arrays_batch(empty, e_off, THR, 1, 10)
    assert not c_off.any() and offsets.tolist() == [0] and len(idx) == 0


@gpu
def test_cluster_raw_kitti_frames(pcr, oracle):
    """Ground left in: one large component per frame, the union-find's worst case."""
    frames = [scenes.kitti_scene(seed=s) for s in range(8)]
    pts, off = _pack(frames)
    got = pcr.euclidean_cluster_batch(pts, off, 0.5, 30, 25_000)
    for f, fr in enumerate(frames):
        assert got[f] == _lists(oracle.euclidean_cluster(fr, 0.5, 30, 25_000)), f"frame {f}"


def _dev_cluster(pcr, pts, off, thr, mn, mx):
    import torch

    ctx = pcr.default_context()
    n = len(pts)
    d = [torch.from_numpy(np.ascontiguousarray(pts[:, j])).cuda() for j in range(3)]
    o = torch.zeros(n + 1, dtype=torch.int32, device="cuda")
    i = torch.zeros(max(n, 1), dtype=torch.int32, device="cuda")
    lab = torch.zeros(max(n, 1), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    c_off = np.zeros(len(off), np.uint64)
    off = np.ascontiguousarray(off, np.uint64)
    lib = _ffi.load()
    st = lib.pcr_euclidean_cluster_batch_dev(ctx._h, *(t.data_ptr() for t in d), off.ctypes.data_as(_ffi.u64p), len(off) - 1, float(thr),
                                             mn, mx, o.data_ptr(), i.data_ptr(), c_off.ctypes.data_as(_ffi.u64p))
    _ffi.check(st, ctx._h)
    st = lib.pcr_cluster_labels_batch_dev(ctx._h, *(t.data_ptr() for t in d), off.ctypes.data_as(_ffi.u64p), len(off) - 1, float(thr),
                                          lab.data_ptr())
    _ffi.check(st, ctx._h)
    ctx.synchronize()
    k = int(c_off[-1])
    offsets = o[:k + 1].cpu().numpy().view(np.uint32)
    return c_off, offsets, i[:int(offsets[-1])].cpu().numpy().view(np.uint32), lab[:n].cpu().numpy().view(np.uint32)


def _single_labels(pcr, fr, thr):
    import torch

    ctx = pcr.default_context()
    d = [torch.from_numpy(np.ascontiguousarray(fr[:, j])).cuda() for j in range(3)]
    lab = torch.zeros(max(len(fr), 1), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    st = _ffi.load().pcr_cluster_labels_dev(ctx._h, *(t.data_ptr() for t in d), len(fr), float(thr), lab.data_ptr())
    _ffi.check(st, ctx._h)
    ctx.synchronize()
    return lab[:len(fr)].cpu().numpy().view(np.uint32)


@gpu
def test_cluster_frames_independent_and_reproducible(pcr, cluster_frames):
    frames = cluster_frames
    pts, off = _pack(frames)
    mn, mx = 2, 3000
    full = pcr.euclidean_cluster_batch(pts, off, THR, mn, mx)
    perm = np.random.default_rng(3).permutation(len(frames))
    p_pts, p_off = _pack([frames[i] for i in perm])
    assert pcr.euclidean_cluster_batch(p_pts, p_off, THR, mn, mx) == [full[i] for i in perm]
    rep = [0, 4, 0, 13, 4, 4]
    r_pts, r_off = _pack([frames[i] for i in rep])
    assert pcr.euclidean_cluster_batch(r_pts, r_off, THR, mn, mx) == [full[i] for i in rep]
    for f, fr in enumerate(frames):
        assert pcr.euclidean_cluster_batch(fr, [0, len(fr)], THR, mn, mx) == [full[f]], f"frame {f}"
    host = pcr.cluster_arrays_batch(pts, off, THR, mn, mx)
    c_off, offsets, idx, labels = _dev_cluster(pcr, pts, off, THR, mn, mx)
    assert np.array_equal(c_off, host[0]) and np.array_equal(offsets, host[1]) and np.array_equal(idx, host[2])
    for f, fr in enumerate(frames):
        if len(fr):
            assert np.array_equal(labels[int(off[f]):int(off[f + 1])], _single_labels(pcr, fr, THR)), f"frame {f}"
    for _ in range(10):
        again = pcr.cluster_arrays_batch(pts, off, THR, mn, mx)
        assert all(np.array_equal(a, b) for a, b in zip(again, host))


# ---- GPU: RANSAC ------------------------------------------------------------------------------------------------

def _ransac_frames():
    """(points, triples) per frame: both choice paths, the early exit, the degenerate frames, KITTI frames."""
    rng = np.random.default_rng(1)
    plane = np.concatenate([rng.uniform(-5, 5, (6000, 2)), rng.normal(0, 0.02, (6000, 1))], 1)
    noise = rng.uniform(-5, 5, (6000, 3))
    line = np.stack([np.arange(50), np.zeros(50), np.zeros(50)], 1)
    bad = np.vstack([plane[:3000], [[np.nan, 0, 0], [np.inf, 1, 1]]])
    s = P.draw_plane_samples
    frames = [
        (np.vstack([plane, noise]), s(12000, 700, 4)),                        # parallel rule, two model chunks
        (np.zeros((0, 3)), np.zeros((0, 3))),                                 # empty
        (np.array([[1.0, 2.0, 3.0]]), np.zeros((0, 3))),                      # one point
        (np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0]]), [[0, 1, 1]]),          # two points: triples never read
        (np.vstack([plane[:4000], noise[:5000]]), s(9000, 64, 3)),            # sequential rule
        (_grid_plane(20, 20, 0.1, lambda x, y: 0 * x), s(400, 100)),          # plane-dominated: the early exit fires
        (line, s(50, 30)),                                                    # only collinear triples: default model
        (np.vstack([plane[:2000], noise[:500]]), np.zeros((0, 3))),           # no triples: inliers of z = 0
        (bad, s(3002, 40, 5)),                                                # non-finite points never count
        (scenes.kitti_scene(3), s(122_000, 500, 7)),
        (scenes.kitti_scene(4, scenes.KITTI_COUNTS["frame80k"]), s(80_000, 500, 8)),
        (np.vstack([plane, noise[:4500]]), s(10500, 15, 9)),                  # n >= 10000 but m < 16: sequential
    ]
    return [(np.ascontiguousarray(p, np.float32), np.asarray(t, np.uint32).reshape(-1, 3)) for p, t in frames]


@pytest.fixture(scope="module")
def ransac_frames():
    return _ransac_frames()


def _check_ransac(pcr, oracle, frames, thr, models, inl, inl_off):
    assert models.shape == (len(frames), 4) and models.dtype == np.float32 and inl.dtype == np.uint32
    assert inl_off.dtype == np.uint64 and len(inl_off) == len(frames) + 1 and inl_off[0] == 0 and int(inl_off[-1]) == len(inl)
    for f, (fr, smp) in enumerate(frames):
        m, want = oracle.ransac_plane_samples(fr, thr, smp)
        assert np.array_equal(models[f].view(np.uint32), m.view(np.uint32)), f"frame {f}"
        assert np.array_equal(inl[int(inl_off[f]):int(inl_off[f + 1])], want), f"frame {f}"
        single = pcr.ransac_plane_samples(_cloud(fr), thr, smp)
        assert np.array_equal(np.array(single.normal + [single.d], np.float32).view(np.uint32), m.view(np.uint32)), f"frame {f}"
        assert single.inliers == want.tolist(), f"frame {f}"


@gpu
@pytest.mark.parametrize("thr", [0.05, 0.15])
def test_ransac_batch_matches_oracle_and_single(pcr, oracle, ransac_frames, thr):
    pts, off = _pack([p for p, _ in ransac_frames])
    models, inl, inl_off = pcr.ransac_plane_samples_batch(pts, off, thr, [t for _, t in ransac_frames])
    _check_ransac(pcr, oracle, ransac_frames, thr, models, inl, inl_off)
    assert models[1].tolist() == models[2].tolist() == models[3].tolist() == models[6].tolist() == [0.0, 0.0, 1.0, 0.0]
    assert inl_off[2] == inl_off[4] and int(inl_off[7] - inl_off[6]) == 50 and int(inl_off[8] - inl_off[7]) > 1000


@gpu
def test_ransac_frames_independent(pcr, ransac_frames):
    import torch

    pts, off = _pack([p for p, _ in ransac_frames])
    smp = [t for _, t in ransac_frames]
    models, inl, inl_off = pcr.ransac_plane_samples_batch(pts, off, 0.15, smp)
    per = [inl[int(inl_off[f]):int(inl_off[f + 1])] for f in range(len(smp))]
    perm = np.random.default_rng(6).permutation(len(smp))
    p_pts, p_off = _pack([ransac_frames[i][0] for i in perm])
    p_models, p_inl, p_inl_off = pcr.ransac_plane_samples_batch(p_pts, p_off, 0.15, [smp[i] for i in perm])
    for j, f in enumerate(perm):
        assert np.array_equal(p_models[j].view(np.uint32), models[f].view(np.uint32))
        assert np.array_equal(p_inl[int(p_inl_off[j]):int(p_inl_off[j + 1])], per[f])
    for f, (fr, t) in enumerate(ransac_frames):
        m1, i1, o1 = pcr.ransac_plane_samples_batch(fr, [0, len(fr)], 0.15, [t])
        assert np.array_equal(m1[0].view(np.uint32), models[f].view(np.uint32)) and np.array_equal(i1, per[f])
    # the _dev form
    ctx = pcr.default_context()
    d = [torch.from_numpy(np.ascontiguousarray(pts[:, j])).cuda() for j in range(3)]
    d_inl = torch.zeros(len(pts), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    s_all = np.ascontiguousarray(np.vstack(smp), np.uint32)
    s_off = np.zeros(len(smp) + 1, np.uint64)
    s_off[1:] = np.cumsum([len(t) for t in smp])
    d_models = np.zeros((len(smp), 4), np.float32)
    d_off = np.zeros(len(smp) + 1, np.uint64)
    st = _ffi.load().pcr_ransac_plane_samples_batch_dev(ctx._h, *(t.data_ptr() for t in d), off.ctypes.data_as(_ffi.u64p), len(smp), 0.15,
                                                        s_all.ctypes.data_as(_ffi.u32p), s_off.ctypes.data_as(_ffi.u64p),
                                                        d_models.ctypes.data_as(_ffi.f32p), d_inl.data_ptr(), d_off.ctypes.data_as(_ffi.u64p))
    _ffi.check(st, ctx._h)
    assert np.array_equal(d_models.view(np.uint32), models.view(np.uint32)) and np.array_equal(d_off, inl_off)
    assert np.array_equal(d_inl[:len(inl)].cpu().numpy().view(np.uint32), inl)
    # seeded draws: frame f's triples are draw_plane_samples(n_f, iterations, [seed, f])
    sub = [p for p, _ in ransac_frames[:6]]
    b_pts, b_off = _pack(sub)
    drawn = [P.draw_plane_samples(len(p), 200, [11, f]) for f, p in enumerate(sub)]
    got = pcr.ransac_plane_batch(b_pts, b_off, 0.1, 200, seed=11)
    want = pcr.ransac_plane_samples_batch(b_pts, b_off, 0.1, drawn)
    assert all(np.array_equal(a, b) for a, b in zip(got, want))


# ---- GPU: the obstacle pipeline ---------------------------------------------------------------------------------

@gpu
def test_obstacle_chain(pcr):
    """voxel batch (0.15) -> SOR batch (20, 2.0) -> compaction -> RANSAC batch (0.15, 500 triples) -> select_inverse ->
    cluster batch (0.8, 10, 20000) over 8 frames: the same clusters as the single calls frame by frame."""
    frames = [scenes.kitti_scene(seed=40 + s, counts=scenes.KITTI_COUNTS["frame80k"]) for s in range(8)]
    pts, off = _pack(frames)
    vox, v_off = pcr.voxel_downsample_batch(pts, off, 0.15)
    keep, _, kept = pcr.sor_normals_batch(vox, v_off, 20, 2.0, 0)
    kept_pts = vox[keep.astype(bool)]
    k_off = np.zeros(len(frames) + 1, np.uint64)
    k_off[1:] = np.cumsum(kept)
    triples = [P.draw_plane_samples(int(k_off[f + 1] - k_off[f]), 500, [99, f]) for f in range(len(frames))]
    models, inl, inl_off = pcr.ransac_plane_samples_batch(kept_pts, k_off, 0.15, triples)
    ground = np.zeros(len(kept_pts), bool)
    for f in range(len(frames)):
        ground[int(k_off[f]) + inl[int(inl_off[f]):int(inl_off[f + 1])].astype(np.int64)] = True
    rest = kept_pts[~ground]
    r_off = np.zeros(len(frames) + 1, np.uint64)
    r_off[1:] = np.cumsum([int(k_off[f + 1] - k_off[f]) - int(inl_off[f + 1] - inl_off[f]) for f in range(len(frames))])
    batched = pcr.euclidean_cluster_batch(rest, r_off, 0.8, 10, 20_000)
    for f, fr in enumerate(frames):
        v = pcr.voxel_downsample(_cloud(fr), 0.15)
        s = pcr.statistical_outlier_removal(v, 20, 2.0)
        r = pcr.ransac_plane_samples(s, 0.15, triples[f])
        assert np.array_equal(np.array(r.normal + [r.d], np.float32).view(np.uint32), models[f].view(np.uint32)), f"frame {f}"
        obstacles = s.select_inverse(r.inliers)
        assert batched[f] == pcr.euclidean_cluster(obstacles, 0.8, 10, 20_000), f"frame {f}"
    assert sum(len(c) for c in batched) > 0


# ---- GPU: C error codes -----------------------------------------------------------------------------------------

@gpu
def test_errors(pcr):
    pts, off = _pack([scenes.hemisphere(300, 1), scenes.hemisphere(300, 2)])
    lib, h = _ffi.load(), pcr.default_context()._h
    x, y, z = (np.ascontiguousarray(pts[:, j]) for j in range(3))
    f = lambda a: a.ctypes.data_as(_ffi.f32p)
    u32 = lambda a: a.ctypes.data_as(_ffi.u32p)
    u64 = lambda a: a.ctypes.data_as(_ffi.u64p)
    smp = np.array([[0, 1, 2], [3, 4, 5], [0, 1, 2]], np.uint32)
    s_off = np.array([0, 2, 3], np.uint64)
    models = np.zeros((2, 4), np.float32)
    inl = np.zeros(len(pts), np.uint32)
    inl_off = np.zeros(3, np.uint64)
    c_offsets = np.zeros(len(pts) + 1, np.uint32)
    c_idx = np.zeros(len(pts), np.uint32)
    c_off = np.zeros(3, np.uint64)
    null32, null64, nullf = C.cast(None, _ffi.u32p), C.cast(None, _ffi.u64p), C.cast(None, _ffi.f32p)

    def ransac(xp=None, offp=None, nf=2, sp=None, sop=None, mp=None, ip=None, iop=None):
        return lib.pcr_ransac_plane_samples_batch(h, f(x) if xp is None else xp, f(y), f(z), u64(off) if offp is None else offp, nf, 0.1,
                                                  u32(smp) if sp is None else sp, u64(s_off) if sop is None else sop,
                                                  f(models) if mp is None else mp, u32(inl) if ip is None else ip,
                                                  u64(inl_off) if iop is None else iop)

    def cluster(xp=None, offp=None, nf=2, op=None, ip=None, cop=None):
        return lib.pcr_euclidean_cluster_batch(h, f(x) if xp is None else xp, f(y), f(z), u64(off) if offp is None else offp, nf, 0.5, 1, 100,
                                               u32(c_offsets) if op is None else op, u32(c_idx) if ip is None else ip,
                                               u64(c_off) if cop is None else cop)

    assert ransac() == _ffi.PCR_OK and inl_off[2] > 0
    assert cluster() == _ffi.PCR_OK and c_off[2] > 0
    # null pointers
    assert ransac(xp=nullf) == _ffi.PCR_ERR_INVALID_ARG
    assert ransac(offp=null64) == _ffi.PCR_ERR_INVALID_ARG
    assert ransac(sp=null32) == _ffi.PCR_ERR_INVALID_ARG                    # triples announced, none given
    assert ransac(sop=null64) == _ffi.PCR_ERR_INVALID_ARG                   # triples given, no offsets
    assert ransac(mp=nullf) == _ffi.PCR_ERR_INVALID_ARG
    assert ransac(ip=null32) == _ffi.PCR_ERR_INVALID_ARG
    assert ransac(iop=null64) == _ffi.PCR_ERR_INVALID_ARG
    assert ransac(sp=null32, sop=null64) == _ffi.PCR_OK                      # no triples at all: the default models
    assert models.tolist() == [[0.0, 0.0, 1.0, 0.0]] * 2
    assert cluster(xp=nullf) == _ffi.PCR_ERR_INVALID_ARG
    assert cluster(offp=null64) == _ffi.PCR_ERR_INVALID_ARG
    assert cluster(op=null32) == _ffi.PCR_ERR_INVALID_ARG
    assert cluster(ip=null32) == _ffi.PCR_ERR_INVALID_ARG
    assert cluster(cop=null64) == _ffi.PCR_ERR_INVALID_ARG
    # bad frame offsets, bad sample offsets
    for bad in ([0, 400, 300], [1, 300, 600]):
        b = np.array(bad, np.uint64)
        assert ransac(offp=u64(b)) == _ffi.PCR_ERR_INVALID_ARG
        assert cluster(offp=u64(b)) == _ffi.PCR_ERR_INVALID_ARG
    for bad in ([1, 2, 3], [0, 3, 2]):
        assert ransac(sop=u64(np.array(bad, np.uint64))) == _ffi.PCR_ERR_INVALID_ARG
    # a triple index valid in the buffer but not in its frame
    far = np.array([[0, 1, 2], [3, 4, 300], [0, 1, 2]], np.uint32)
    assert ransac(sp=u32(far)) == _ffi.PCR_ERR_INVALID_ARG
    assert "frame 0" in _ffi.last_error(h)
    # more than 65535 frames
    many = np.zeros(65537, np.uint64)
    many[-1] = len(pts)
    big_models = np.zeros((65536, 4), np.float32)
    big_off = np.zeros(65537, np.uint64)
    assert ransac(offp=u64(many), nf=65536, sp=null32, sop=null64, mp=f(big_models), iop=u64(big_off)) == _ffi.PCR_ERR_UNSUPPORTED
    assert cluster(offp=u64(many), nf=65536, cop=u64(big_off)) == _ffi.PCR_ERR_UNSUPPORTED
    # 65535 frames are accepted (all empty but the last, which holds every point)
    assert cluster(offp=u64(many[1:]), nf=65535, cop=u64(big_off)) == _ffi.PCR_OK
    assert not big_off[:65535].any() and int(big_off[65535]) == len(pcr.euclidean_cluster(_cloud(pts), 0.5, 1, 100))
    # the labels form: threshold <= 0 and null pointers
    d = lambda a: C.c_void_p(a.ctypes.data)
    assert lib.pcr_cluster_labels_batch_dev(h, None, None, None, u64(off), 2, 0.5, None) == _ffi.PCR_ERR_INVALID_ARG
    assert lib.pcr_cluster_labels_batch_dev(h, d(x), d(y), d(z), u64(off), 2, 0.0, d(c_idx)) == _ffi.PCR_ERR_INVALID_ARG
