"""Batched voxel_downsample and estimate_normals (pcr_voxel_downsample_batch, pcr_estimate_normals_batch): many frames
of one buffer in one call, every frame processed as if it were alone.

CPU tests: the Python layer rejects bad arguments with ValueError before it touches a device.
GPU tests: every voxel frame bit-exact against the CPU oracle, through both sort paths (packed key, and the per-axis
passes plus a frame pass); a frame's output independent of the other frames, of their order, of repetition and of the
entry point; the frame-stream key box untouched; every normals frame bit-identical to the single call and within the
oracle's bar; the voxel -> SOR/normals and voxel -> normals -> ICP chains equal to the per-frame way; the C error codes.
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


def _frame(a, off, f):
    return a[int(off[f]):int(off[f + 1])]


def _cloud(pts):
    return P.PointCloud.from_numpy(np.ascontiguousarray(pts, np.float32))


def _angles(a, b):
    a = a.astype(np.float64)
    b = b.astype(np.float64)
    return np.arctan2(np.linalg.norm(np.cross(a, b), axis=1), np.abs(np.sum(a * b, axis=1)))


# ---- argument checks (no device needed) ------------------------------------------------------------------------

@pytest.mark.parametrize("offsets", [[0, 6, 4, 10], [1, 4, 10], [0, 4, 11], [0, 4, 9], []])
def test_bad_offsets_raise(offsets):
    pts = np.zeros((10, 3), np.float32)
    with pytest.raises(ValueError):
        P.voxel_downsample_batch(pts, offsets, 0.1)
    with pytest.raises(ValueError):
        P.estimate_normals_batch(pts, offsets, 10)


@pytest.mark.parametrize("voxel", [0.0, -1.0, math.nan, math.inf])
def test_bad_voxel_size_raises(voxel):
    with pytest.raises(ValueError):
        P.voxel_downsample_batch(np.zeros((10, 3), np.float32), [0, 4, 10], voxel)


@pytest.mark.parametrize("shape", [(10, 2), (30,), (2, 5, 3), (10, 4)])
def test_bad_point_shape_raises(shape):
    pts = np.zeros(shape, np.float32)
    with pytest.raises(ValueError):
        P.voxel_downsample_batch(pts, [0, 4, 10], 0.1)
    with pytest.raises(ValueError):
        P.estimate_normals_batch(pts, [0, 4, 10], 10)


# ---- GPU: voxel -------------------------------------------------------------------------------------------------

def _voxel_frames():
    """KITTI frames of different seeds and sizes, the edge cases of the single call, and two frames whose key boxes need
    more than 63 bits (a far outlier, saturated keys): the whole batch then takes the per-axis passes."""
    rng = np.random.default_rng(8)
    base = rng.uniform(-5, 5, (4000, 3)).astype(np.float32)
    bad = scenes.kitti_scene(3, (9_000, 400, 80, 200))
    bad[::37, 0] = np.nan
    bad[5::91, 2] = np.inf
    tall = np.column_stack([rng.uniform(0.0, 0.01, 6000), rng.uniform(0.0, 0.01, 6000), rng.uniform(0.0, 60.0, 6000)])
    packed = [
        scenes.kitti_scene(1, (9_000, 400, 80, 200)),
        np.zeros((0, 3), np.float32),                                     # empty
        scenes.kitti_scene(2, scenes.KITTI_COUNTS["frame80k"]),
        np.array([[1.0, 2.0, 3.0]], np.float32),                          # one point
        np.full((5, 3), np.nan, np.float32),                              # nothing finite
        bad,                                                              # NaN and inf points
        np.repeat(base[:500], 9, axis=0),                                 # duplicated points
        tall.astype(np.float32),                                          # a column of thousands of points
        scenes.kitti_scene(4, (20_000, 1_000, 150, 500)),
        np.zeros((0, 3), np.float32),
    ]
    wide = [
        np.vstack([base, [[3e6, -2e6, 1e6]], [[-4e7, 5e7, 9e6]]]),         # far outliers: key box > 63 bits
        np.vstack([base[:100], [[3e9, 3e9, 3e9]], [[3.5e9, 3e9, 3e9]], [[-1e12, 0, 0]]]),  # saturated i32 keys merge
    ]
    return [np.ascontiguousarray(f, np.float32) for f in packed], [np.ascontiguousarray(f, np.float32) for f in wide]


@pytest.fixture(scope="module")
def voxel_frames():
    return _voxel_frames()


def _check_frames_equal(got, got_off, want_frames):
    assert len(got_off) == len(want_frames) + 1 and got_off[0] == 0
    assert int(got_off[-1]) == len(got)
    for f, want in enumerate(want_frames):
        g = _frame(got, got_off, f)
        assert g.shape == want.shape, (f, g.shape, want.shape)
        assert np.array_equal(g.view(np.uint32), want.view(np.uint32)), f"frame {f}"


@gpu
@pytest.mark.parametrize("voxel", [0.05, 0.5])
@pytest.mark.parametrize("which", ["packed_key", "axis_passes"])
def test_voxel_batch_matches_oracle(pcr, oracle, voxel_frames, voxel, which):
    packed, wide = voxel_frames
    frames = packed if which == "packed_key" else packed[:4] + wide[:1] + packed[4:] + wide[1:]
    pts, off = _pack(frames)
    got, got_off = pcr.voxel_downsample_batch(pts, off, voxel)
    assert got.dtype == np.float32 and got_off.dtype == np.uint64
    _check_frames_equal(got, got_off, [oracle.voxel_downsample(f, voxel) for f in frames])


def _voxel_dev(pcr, pts, off, voxel, ctx):
    import torch

    n = len(pts)
    d = [torch.from_numpy(np.ascontiguousarray(pts[:, j])).cuda() for j in range(3)]
    o = [torch.zeros(max(n, 1), dtype=torch.float32, device="cuda") for _ in range(3)]
    torch.cuda.synchronize()
    out_off = np.zeros(len(off), np.uint64)
    off = np.ascontiguousarray(off, np.uint64)
    st = _ffi.load().pcr_voxel_downsample_batch_dev(ctx._h, *(t.data_ptr() for t in d), off.ctypes.data_as(_ffi.u64p), len(off) - 1,
                                                    float(voxel), *(t.data_ptr() for t in o), out_off.ctypes.data_as(_ffi.u64p))
    _ffi.check(st, ctx._h)
    m = int(out_off[-1])
    return np.stack([t[:m].cpu().numpy() for t in o], axis=1), out_off


@gpu
@pytest.mark.parametrize("voxel", [0.05, 0.5])
def test_voxel_frames_independent_and_reproducible(pcr, voxel_frames, voxel):
    packed, wide = voxel_frames
    frames = packed + wide
    pts, off = _pack(frames)
    full, full_off = pcr.voxel_downsample_batch(pts, off, voxel)
    want = [_frame(full, full_off, f) for f in range(len(frames))]
    again = pcr.voxel_downsample_batch(pts, off, voxel)
    _check_frames_equal(*again, want)
    perm = np.random.default_rng(2).permutation(len(frames))
    p_pts, p_off = _pack([frames[i] for i in perm])
    _check_frames_equal(*pcr.voxel_downsample_batch(p_pts, p_off, voxel), [want[i] for i in perm])
    for f, fr in enumerate(frames):
        _check_frames_equal(*pcr.voxel_downsample_batch(fr, [0, len(fr)], voxel), [want[f]])
        if len(fr):
            single = pcr.voxel_downsample(_cloud(fr), voxel).to_numpy()
            assert np.array_equal(single.view(np.uint32), want[f].view(np.uint32)), f"frame {f}"
    _check_frames_equal(*_voxel_dev(pcr, pts, off, voxel, pcr.default_context()), want)
    # the packed-key subset alone (its frames' key boxes fit 63 bits): the same frames, the same bits
    sub_pts, sub_off = _pack(packed)
    _check_frames_equal(*pcr.voxel_downsample_batch(sub_pts, sub_off, voxel), want[:len(packed)])


@gpu
def test_voxel_batch_leaves_the_frame_stream_box_alone(pcr, oracle):
    ctx = pcr.Context(device=0)
    ctx.set_frame_stream(True)
    a = scenes.kitti_scene(41)  # (a full frame: its 5 cm column table is small enough for the guessed box to be used)
    for _ in range(3):  # measured, then guessed from the kept box
        assert np.array_equal(pcr.voxel_downsample(_cloud(a), 0.05, ctx).to_numpy(), oracle.voxel_downsample(a, 0.05))
    before = ctx.hint_stats()
    assert before["voxel_box_guess_held"] == 2
    far = (a + np.float32(300.0)).astype(np.float32)
    pts, off = _pack([far, a, np.full((3, 3), np.nan, np.float32)])
    for v in (0.05, 0.2):
        got, got_off = pcr.voxel_downsample_batch(pts, off, v, ctx=ctx)
        _check_frames_equal(got, got_off, [oracle.voxel_downsample(f, v) for f in (far, a, np.full((3, 3), np.nan, np.float32))])
    assert ctx.hint_stats() == before
    assert np.array_equal(pcr.voxel_downsample(_cloud(a), 0.05, ctx).to_numpy(), oracle.voxel_downsample(a, 0.05))
    after = ctx.hint_stats()
    assert after["voxel_box_guess_held"] == before["voxel_box_guess_held"] + 1  # the box kept before the batch still served
    ctx.close()


# ---- GPU: normals -----------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def normals_frames():
    bad = scenes.kitti_scene(12, (6_000, 300, 60, 150))
    bad[::41] = np.nan
    bad[7::97, 1] = np.inf
    return [
        scenes.kitti_scene(10, (9_000, 400, 80, 200)),
        np.zeros((0, 3), np.float32),
        np.array([[0.0, 0.0, 0.0]], np.float32),
        bad,
        scenes.kitti_scene(11, (14_000, 700, 100, 300)),
        np.repeat(scenes.uniform_cube(200, 5, 0, 3), 4, axis=0),
        np.full((4, 3), np.nan, np.float32),
    ]


@gpu
@pytest.mark.parametrize("k", [20, 40])
def test_normals_batch_matches_single_calls_and_oracle(pcr, oracle, normals_frames, k):
    pts, off = _pack(normals_frames)
    nrm = pcr.estimate_normals_batch(pts, off, k)
    assert nrm.shape == (len(pts), 3) and nrm.dtype == np.float32
    for f, fr in enumerate(normals_frames):
        if len(fr) == 0:
            continue
        got = _frame(nrm, off, f)
        single = pcr.normals_array(_cloud(fr), k)
        assert np.array_equal(got.view(np.uint32), single.view(np.uint32)), f"frame {f}"
        ang = _angles(got, oracle.normals(fr, k, threads=T))
        assert not np.isfinite(ang).any() or np.nanmax(ang) < 1e-4, f"frame {f}: {np.nanmax(ang)} rad"
    # independent of the other frames and of their order, reproducible, and the same through the _dev form
    perm = np.random.default_rng(4).permutation(len(normals_frames))
    p_pts, p_off = _pack([normals_frames[i] for i in perm])
    p_nrm = pcr.estimate_normals_batch(p_pts, p_off, k)
    for j, f in enumerate(perm):
        assert np.array_equal(_frame(p_nrm, p_off, j).view(np.uint32), _frame(nrm, off, f).view(np.uint32)), f"frame {f}"
    assert np.array_equal(pcr.estimate_normals_batch(pts, off, k).view(np.uint32), nrm.view(np.uint32))
    import torch

    ctx = pcr.default_context()
    d = [torch.from_numpy(np.ascontiguousarray(pts[:, j])).cuda() for j in range(3)]
    o = [torch.zeros(len(pts), dtype=torch.float32, device="cuda") for _ in range(3)]
    torch.cuda.synchronize()
    vp = np.zeros(3, np.float32)
    st = _ffi.load().pcr_estimate_normals_batch_dev(ctx._h, *(t.data_ptr() for t in d), off.ctypes.data_as(_ffi.u64p), len(off) - 1, k,
                                                    vp.ctypes.data_as(_ffi.f32p), *(t.data_ptr() for t in o))
    _ffi.check(st, ctx._h)
    ctx.synchronize()
    dev = np.stack([t.cpu().numpy() for t in o], axis=1)
    assert np.array_equal(dev.view(np.uint32), nrm.view(np.uint32))


@gpu
def test_normals_batch_k_zero_and_empty(pcr, normals_frames):
    pts, off = _pack(normals_frames)
    assert pcr.estimate_normals_batch(pts, off, 0).shape == (0, 3)
    empty, e_off = _pack([np.zeros((0, 3), np.float32)] * 3)
    assert pcr.estimate_normals_batch(empty, e_off, 10).shape == (0, 3)
    lib, h = _ffi.load(), pcr.default_context()._h
    x, y, z = (np.ascontiguousarray(pts[:, j]) for j in range(3))
    nx, ny, nz = (np.full(len(pts), 7.0, np.float32) for _ in range(3))
    f = lambda a: a.ctypes.data_as(_ffi.f32p)
    vp = np.zeros(3, np.float32)
    st = lib.pcr_estimate_normals_batch(h, f(x), f(y), f(z), off.ctypes.data_as(_ffi.u64p), len(off) - 1, 0, f(vp), f(nx), f(ny), f(nz))
    assert st == _ffi.PCR_OK and (nx == 7.0).all() and (ny == 7.0).all() and (nz == 7.0).all()  # nothing written


# ---- GPU: chains ------------------------------------------------------------------------------------------------

@gpu
def test_voxel_batch_feeds_sor_normals_batch(pcr):
    frames = [scenes.kitti_scene(s, (12_000, 600, 100, 300)) for s in (30, 31, 32, 33)]
    pts, off = _pack(frames)
    vox, v_off = pcr.voxel_downsample_batch(pts, off, 0.05)
    keep, nrm, kept = pcr.sor_normals_batch(vox, v_off, 10, 1.0, 20)
    for f, fr in enumerate(frames):
        v = pcr.voxel_downsample(_cloud(fr), 0.05).to_numpy()
        k1, n1, c1 = pcr.sor_normals_batch(v, [0, len(v)], 10, 1.0, 20)
        assert np.array_equal(_frame(keep, v_off, f), k1), f"frame {f}"
        assert np.array_equal(_frame(nrm, v_off, f).view(np.uint32), n1.view(np.uint32)), f"frame {f}"
        assert int(kept[f]) == int(c1[0])


def _icp_bits(r):
    return (np.float32(r.rotation).tobytes(), np.float32(r.translation).tobytes(), np.float32(r.rmse).tobytes(),
            np.float32(r.fitness).tobytes(), r.num_iterations, r.converged)


@gpu
def test_odometry_front_end_chain(pcr):
    """voxel batch -> normals batch -> point-to-plane ICP batch over consecutive frames: the same result bits as the ICP
    batch fed with the single calls' outputs."""
    seq = scenes.kitti_sequence(6, seed=3, counts=(17_600, 880, 145, 495))
    pts, off = _pack(seq)
    pairs = np.array([(i + 1, i) for i in range(len(seq) - 1)], np.uint32)
    kw = dict(max_iterations=30, tolerance=0.0)
    vox, v_off = pcr.voxel_downsample_batch(pts, off, 0.2)
    nrm = pcr.estimate_normals_batch(vox, v_off, 15)
    chained = pcr.icp_point_to_plane_batch(vox, v_off, pairs, nrm, **kw)
    singles = [pcr.voxel_downsample(_cloud(f), 0.2).to_numpy() for f in seq]
    s_pts, s_off = _pack(singles)
    assert np.array_equal(s_off, v_off) and np.array_equal(s_pts.view(np.uint32), vox.view(np.uint32))
    s_nrm = np.vstack([pcr.normals_array(_cloud(v), 15) for v in singles])
    assert np.array_equal(s_nrm.view(np.uint32), nrm.view(np.uint32))
    looped = pcr.icp_point_to_plane_batch(s_pts, s_off, pairs, s_nrm, **kw)
    assert [_icp_bits(r) for r in chained] == [_icp_bits(r) for r in looped]
    assert all(r.num_iterations == 30 for r in chained)


# ---- GPU: C error codes -----------------------------------------------------------------------------------------

@gpu
def test_errors(pcr):
    pts, off = _pack([scenes.hemisphere(300, 1), scenes.hemisphere(300, 2)])
    lib, h = _ffi.load(), pcr.default_context()._h
    x, y, z = (np.ascontiguousarray(pts[:, j]) for j in range(3))
    o = [np.zeros(len(pts), np.float32) for _ in range(3)]
    f = lambda a: a.ctypes.data_as(_ffi.f32p)
    u64 = lambda a: a.ctypes.data_as(_ffi.u64p)
    out_off = np.zeros(3, np.uint64)
    vp = np.zeros(3, np.float32)

    def vox(xp, offp, nf, v=0.1, outp=None):
        return lib.pcr_voxel_downsample_batch(h, xp, f(y), f(z), offp, nf, v, f(o[0]), f(o[1]), f(o[2]),
                                              u64(out_off) if outp is None else outp)

    def nrm(xp, offp, nf, k=10, vpp=None):
        return lib.pcr_estimate_normals_batch(h, xp, f(y), f(z), offp, nf, k, f(vp) if vpp is None else vpp, f(o[0]), f(o[1]), f(o[2]))

    assert vox(f(x), u64(off), 2) == _ffi.PCR_OK and out_off[0] == 0 and out_off[2] > 0
    assert nrm(f(x), u64(off), 2) == _ffi.PCR_OK
    # null pointers
    assert vox(None, u64(off), 2) == _ffi.PCR_ERR_INVALID_ARG
    assert vox(f(x), None, 2) == _ffi.PCR_ERR_INVALID_ARG
    assert vox(f(x), u64(off), 2, outp=C.cast(None, _ffi.u64p)) == _ffi.PCR_ERR_INVALID_ARG
    assert nrm(None, u64(off), 2) == _ffi.PCR_ERR_INVALID_ARG
    assert nrm(f(x), None, 2) == _ffi.PCR_ERR_INVALID_ARG
    assert nrm(f(x), u64(off), 2, vpp=C.cast(None, _ffi.f32p)) == _ffi.PCR_ERR_INVALID_ARG
    # bad offsets
    for bad in ([0, 400, 300], [1, 300, 600]):
        b = np.array(bad, np.uint64)
        assert vox(f(x), u64(b), 2) == _ffi.PCR_ERR_INVALID_ARG
        assert nrm(f(x), u64(b), 2) == _ffi.PCR_ERR_INVALID_ARG
    # bad voxel size, k above PCR_MAX_K
    for v in (0.0, -1.0, math.nan, math.inf):
        assert vox(f(x), u64(off), 2, v=v) == _ffi.PCR_ERR_INVALID_ARG
    assert nrm(f(x), u64(off), 2, k=1025) == _ffi.PCR_ERR_UNSUPPORTED
    # more than 65535 frames
    many = np.zeros(65537, np.uint64)
    many[-1] = len(pts)
    big_out = np.zeros(65537, np.uint64)
    assert vox(f(x), u64(many), 65536, outp=u64(big_out)) == _ffi.PCR_ERR_UNSUPPORTED
    assert nrm(f(x), u64(many), 65536) == _ffi.PCR_ERR_UNSUPPORTED
    # 65535 frames are accepted (all empty but the last, which holds every point)
    assert vox(f(x), u64(many[1:]), 65535, outp=u64(big_out)) == _ffi.PCR_OK
    assert not big_out[:65535].any() and int(big_out[65535]) == len(pcr.voxel_downsample(_cloud(pts), 0.1))
    # SOR + normals batch, all three forms: bad frame offsets are rejected before any device work and named in the
    # message, also for one frame; no frames is nothing to do
    import torch

    d = [torch.from_numpy(a).cuda() for a in (x, y, z)]
    d_out = [torch.zeros(len(pts), dtype=dt, device="cuda") for dt in (torch.uint8, torch.float32, torch.float32, torch.float32)]
    torch.cuda.synchronize()
    keep, kept = np.zeros(len(pts), np.uint8), np.zeros(2, np.uint64)
    rows, nrm_rows = np.ascontiguousarray(pts, np.float32), np.zeros((len(pts), 3), np.float32)
    u8 = lambda a: a.ctypes.data_as(_ffi.u8p)
    forms = (lambda offp, nf: lib.pcr_sor_normals_batch(h, f(x), f(y), f(z), offp, nf, 10, 1.0, 20, f(vp), u8(keep), f(o[0]), f(o[1]), f(o[2]),
                                                        u64(kept)),
             lambda offp, nf: lib.pcr_sor_normals_batch_dev(h, *(t.data_ptr() for t in d), offp, nf, 10, 1.0, 20, f(vp),
                                                            *(t.data_ptr() for t in d_out)),
             lambda offp, nf: lib.pcr_sor_normals_batch_rows(h, f(rows), offp, nf, 10, 1.0, 20, f(vp), u8(keep), f(nrm_rows), u64(kept)))
    for call in forms:
        for bad in ([0, 400, 300], [1, 300, 600], [1, 300]):
            b = np.array(bad, np.uint64)
            assert call(u64(b), len(bad) - 1) == _ffi.PCR_ERR_INVALID_ARG
            assert "frame_offsets" in _ffi.last_error(h)
        assert call(u64(off), 0) == _ffi.PCR_OK
