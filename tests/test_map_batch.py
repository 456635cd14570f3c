"""Batched apply_transform, pose chaining and frame merge (pcr_apply_transform_batch, pcr_frames_apply_transform,
pcr_transform_compose, pcr_frames_merge): the map of an odometry chain assembled on the device.

CPU tests: the Python layer rejects bad transforms, offsets and chain inputs (ValueError) before it touches a device;
compose / pcr_transform_compose are bit for bit oracle.compose on seeded random transforms; chain_poses is a loop of
oracle.compose.
GPU tests: the raw and _dev batch calls against the oracle and the single call on a mixed batch with one transform per
frame; frame independence; DeviceFrames.apply_transform against DeviceCloud.apply_transform per frame; merge; the
odometry map over 8 frames against the per-frame way and the oracle, and its poses against the generator's; the C error
codes.
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


def _mixed():
    """KITTI frames, an empty, a one-point, an all-NaN and a NaN / inf-mixed frame, and two identical frames."""
    rng = np.random.default_rng(21)
    nan_mixed = scenes.hemisphere(500, 3)
    nan_mixed[rng.choice(500, 60, replace=False), rng.integers(0, 3, 60)] = np.nan
    nan_mixed[::97, 0] = np.inf
    nan_mixed[5::89, 2] = -np.inf
    return [
        scenes.kitti_scene(seed=11, counts=(7_000, 350, 60, 150)),
        np.zeros((0, 3), np.float32),
        np.array([[1.0, 2.0, 3.0]], np.float32),
        np.full((40, 3), np.nan, np.float32),
        nan_mixed,
        scenes.hemisphere(800, 9),
        scenes.hemisphere(800, 9),
        scenes.kitti_scene(seed=12, counts=(5_000, 250, 40, 120)),
    ]


def _rotation(rng):
    q, r = np.linalg.qr(rng.normal(size=(3, 3)))
    q = q * np.sign(np.diag(r))
    if np.linalg.det(q) < 0:
        q[:, 0] = -q[:, 0]
    return q.astype(np.float32)


def _random_transforms(n, seed):
    """(n, 12) f32: random rotations and translations, with the identity, negative zeros and a non-orthogonal matrix."""
    rng = np.random.default_rng(seed)
    out = np.zeros((n, 12), np.float32)
    for i in range(n):
        out[i, :9] = _rotation(rng).reshape(9)
        out[i, 9:] = rng.normal(0.0, 20.0, 3).astype(np.float32)
    out[0] = [1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0]
    if n > 1:
        out[1] = [1, -0.0, 0, 0, 1, -0.0, -0.0, 0, 1, -0.0, -0.0, -0.0]
    if n > 2:
        out[2] = rng.uniform(-3, 3, 12).astype(np.float32)
    return out


def _rt(t12):
    return t12[:9].reshape(3, 3), t12[9:]


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _same_as_oracle(got, ref):
    """Bit for bit, except that a NaN matches any NaN: the device writes the canonical NaN where the host propagates the
    input's payload."""
    nan = np.isnan(ref)
    return got.shape == ref.shape and np.array_equal(np.isnan(got), nan) and np.array_equal(_bits(got)[~nan], _bits(ref)[~nan])


# ---- argument checks and compose (no device needed) -------------------------------------------------------------

@pytest.mark.parametrize("transforms", [np.zeros((3, 9)), np.zeros((3, 3, 3)), np.zeros((2, 12)), np.zeros((4, 12)), np.zeros(36),
                                        np.zeros((3, 4, 3)), np.array([["a"] * 12] * 3), [[0.0] * 12] * 2, None])
def test_bad_transforms_raise(transforms):
    pts = np.zeros((10, 3), np.float32)
    with pytest.raises(ValueError):
        P.apply_transform_batch(pts, [0, 4, 4, 10], transforms)
    with pytest.raises(ValueError):
        P._frame_transforms(transforms, 3)


@pytest.mark.parametrize("offsets", [[0, 6, 4, 10], [1, 4, 10], [0, 4, 11], [0, 4, 9], [], [0.0, 4.0, 10.0]])
def test_bad_offsets_raise(offsets):
    with pytest.raises(ValueError):
        P.apply_transform_batch(np.zeros((10, 3), np.float32), offsets, np.zeros((max(len(offsets) - 1, 0), 12), np.float32))


def test_transform_layouts():
    t34 = np.arange(24, dtype=np.float32).reshape(2, 3, 4)
    got = P._frame_transforms(t34, 2)
    assert got.dtype == np.float32 and got.flags["C_CONTIGUOUS"]
    for f in range(2):
        assert got[f, :9].tolist() == t34[f, :, :3].reshape(9).tolist() and got[f, 9:].tolist() == t34[f, :, 3].tolist()
    t12 = np.arange(24, dtype=np.float64).reshape(2, 12)
    assert P._frame_transforms(t12, 2).tolist() == t12.tolist()
    assert P._frame_transforms(np.zeros((0, 12)), 0).shape == (0, 12)


@pytest.mark.parametrize("relative", [np.zeros((3, 9)), np.zeros(12), np.zeros((2, 4, 3)), [[0.0] * 12, [0.0] * 11], [[0.0] * 9],
                                      [np.zeros((3, 4)), np.zeros((4, 3))], [np.zeros((2, 6))]])
def test_bad_chain_input_raises(relative):
    with pytest.raises(ValueError):
        P.chain_poses(relative)


def test_compose_matches_oracle_bit_for_bit():
    ts = _random_transforms(300, seed=8)
    lib = _ffi.load()
    f32 = lambda a: a.ctypes.data_as(_ffi.f32p)
    rng = np.random.default_rng(9)
    for _ in range(400):
        a, b = ts[rng.integers(len(ts))], ts[rng.integers(len(ts))]
        oR, ot = O.compose(_rt(a), _rt(b))
        R, t = P.compose(_rt(a), _rt(b))
        assert R.shape == (3, 3) and t.shape == (3,) and R.dtype == t.dtype == np.float32
        assert _bits(R).tobytes() == _bits(oR).tobytes() and _bits(t).tobytes() == _bits(ot).tobytes()
        out = np.empty(12, np.float32)
        assert lib.pcr_transform_compose(f32(a), f32(b), f32(out)) == _ffi.PCR_OK
        assert out.tobytes() == np.concatenate([oR.reshape(9), ot]).astype(np.float32).tobytes()
        alias = a.copy()  # out may be one of the inputs
        assert lib.pcr_transform_compose(f32(alias), f32(b), f32(alias)) == _ffi.PCR_OK and alias.tobytes() == out.tobytes()
    # negative zero survives where the reference keeps it: identity with -0 entries composed with itself
    nz = ts[1]
    R, t = P.compose(_rt(nz), _rt(nz))
    oR, ot = O.compose(_rt(nz), _rt(nz))
    assert _bits(R).tobytes() == _bits(oR).tobytes() and _bits(t).tobytes() == _bits(ot).tobytes()
    assert lib.pcr_transform_compose(None, f32(nz), f32(out)) == _ffi.PCR_ERR_INVALID_ARG
    assert lib.pcr_transform_compose(f32(nz), f32(nz), None) == _ffi.PCR_ERR_INVALID_ARG


def test_chain_poses_is_a_loop_of_oracle_compose():
    rel = _random_transforms(40, seed=10)
    poses = P.chain_poses(rel)
    assert poses.shape == (41, 12) and poses.dtype == np.float32
    assert poses[0].tolist() == [1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0]
    R, t = np.eye(3, dtype=np.float32), np.zeros(3, np.float32)
    for i in range(len(rel)):
        R, t = O.compose(_rt(rel[i]), (R, t))
        assert poses[i + 1].tobytes() == np.concatenate([R.reshape(9), t]).astype(np.float32).tobytes(), i
    # IcpResult-like input (rotation as nested lists) and the list form give the same poses
    res = []
    for r in rel:
        ir = P.IcpResult.__new__(P.IcpResult)
        ir.rotation, ir.translation = r[:9].reshape(3, 3).tolist(), r[9:].tolist()
        res.append(ir)
    assert P.chain_poses(res).tobytes() == poses.tobytes()
    assert P.chain_poses(rel.tolist()).tobytes() == poses.tobytes()
    # [R | t] matrices, as an (n, 3, 4) array or a list of (3, 4) entries, are read as apply_transform_batch reads them
    rt34 = np.concatenate([rel[:, :9].reshape(-1, 3, 3), rel[:, 9:, None]], axis=2)
    assert P.chain_poses(rt34).tobytes() == poses.tobytes()
    assert P.chain_poses(list(rt34)).tobytes() == poses.tobytes()
    assert P.chain_poses([]).tobytes() == poses[:1].tobytes()


# ---- GPU: the batch against the oracle and the single call -------------------------------------------------------

def _dev_batch(pcr, pts, off, tr):
    """pcr_apply_transform_batch_dev on the device arrays of an uploaded batch, into those of a second one."""
    lib, ctx = _ffi.load(), pcr.default_context()
    src, dst = P.DeviceFrames.from_numpy(pts, off), P.DeviceFrames.from_numpy(np.zeros_like(pts), off)
    sp, dp = [C.c_void_p() for _ in range(6)], [C.c_void_p() for _ in range(6)]
    _ffi.check(lib.pcr_frames_device_pointers(src._h, *(C.byref(p) for p in sp)), ctx._h)
    _ffi.check(lib.pcr_frames_device_pointers(dst._h, *(C.byref(p) for p in dp)), ctx._h)
    tr_host = np.ascontiguousarray(tr, np.float32).copy()
    off_host = np.ascontiguousarray(off, np.uint64).copy()
    st = lib.pcr_apply_transform_batch_dev(ctx._h, sp[0], sp[1], sp[2], off_host.ctypes.data_as(_ffi.u64p), len(off) - 1,
                                           tr_host.ctypes.data_as(_ffi.f32p), dp[0], dp[1], dp[2])
    _ffi.check(st, ctx._h)
    tr_host[:] = np.nan  # the host arrays are free again on return
    off_host[:] = 0
    ctx.synchronize()
    return dst.to_numpy()[0]


@gpu
def test_batch_equals_oracle_and_single_call(pcr):
    frames = _mixed()
    pts, off = _pack(frames)
    tr = _random_transforms(len(frames), seed=3)
    tr[5] = tr[3]  # the first of the two identical frames gets another frame's transform, the second its own
    raw = pcr.apply_transform_batch(pts, off, tr)
    dev = _dev_batch(pcr, pts, off, tr)
    assert raw.dtype == np.float32 and raw.shape == pts.shape
    assert raw.tobytes() == dev.tobytes()
    for f, fr in enumerate(frames):
        b, e = int(off[f]), int(off[f + 1])
        R, t = _rt(tr[f])
        assert _same_as_oracle(raw[b:e], O.apply_transform(fr, R, t)), f"frame {f}: oracle"
        if len(fr):
            assert raw[b:e].tobytes() == pcr.apply_transform(P.PointCloud.from_numpy(fr), R, t).to_numpy().tobytes(), f"frame {f}: single"
    assert raw[int(off[5]):int(off[6])].tobytes() != raw[int(off[6]):int(off[7])].tobytes()
    # (F, 3, 4) [R | t] gives the same bits
    t34 = np.concatenate([tr[:, :9].reshape(-1, 3, 3), tr[:, 9:, None]], axis=2)
    assert pcr.apply_transform_batch(pts, off, t34).tobytes() == raw.tobytes()


@gpu
def test_frame_independence(pcr):
    frames = _mixed()
    tr = _random_transforms(len(frames), seed=4)
    perm = np.random.default_rng(6).permutation(len(frames))

    def run(order):
        pts, off = _pack([frames[i] for i in order])
        out = pcr.apply_transform_batch(pts, off, tr[order])
        return [out[int(off[j]):int(off[j + 1])].tobytes() for j in range(len(order))]

    base = run(np.arange(len(frames)))
    permuted = run(perm)
    assert [permuted[j] for j in np.argsort(perm)] == base


@gpu
@pytest.mark.parametrize("with_normals", [False, True])
def test_device_frames_apply_transform(pcr, with_normals):
    frames = _mixed()
    batch = P.DeviceFrames.from_numpy(*_pack(frames))
    if with_normals:
        batch = batch.estimate_normals(8)
    tr = _random_transforms(len(frames), seed=5)
    moved = batch.apply_transform(tr)
    assert not moved.has_normals() and moved.normals_to_numpy() is None
    assert np.array_equal(moved.offsets, batch.offsets) and moved.n_frames == batch.n_frames
    pts, off = moved.to_numpy()
    for f in range(len(frames)):
        single = batch.frame(f).apply_transform(*_rt(tr[f]))
        assert pts[int(off[f]):int(off[f + 1])].tobytes() == single.to_numpy().tobytes(), f"frame {f}"
    assert batch.to_numpy()[0].tobytes() == _pack(frames)[0].tobytes()  # the input is left unchanged
    with pytest.raises(ValueError):
        batch.apply_transform(tr[:-1])
    with pytest.raises(ValueError):
        batch.apply_transform(tr[:, :9])


@gpu
def test_merge(pcr):
    frames = [np.zeros((0, 3), np.float32), scenes.hemisphere(300, 1), np.zeros((0, 3), np.float32), scenes.hemisphere(200, 2),
              np.zeros((0, 3), np.float32)]
    batch = P.DeviceFrames.from_numpy(*_pack(frames))
    merged = batch.merge()
    assert not merged.has_normals() and merged.to_numpy().tobytes() == batch.to_numpy()[0].tobytes()
    with_n = batch.estimate_normals(10)
    merged = with_n.merge()
    assert merged.has_normals() and len(merged) == 500
    assert merged.to_numpy().tobytes() == with_n.to_numpy()[0].tobytes()
    assert merged.normals_to_numpy().tobytes() == with_n.normals_to_numpy().tobytes()
    empty = P.DeviceFrames.from_numpy(np.zeros((0, 3), np.float32), [0, 0, 0]).merge()
    assert len(empty) == 0 and empty.to_numpy().shape == (0, 3)


@gpu
def test_odometry_map(pcr):
    """voxel 0.2 -> normals 15 -> point-to-plane ICP over (i+1, i) -> chain_poses -> apply_transform -> merge -> voxel 0.1."""
    n, yaw, step = 8, 0.01, np.array([0.4, 0.05, 0.0])
    seq = scenes.kitti_sequence(n, seed=3, counts=(17_600, 880, 145, 495), step=tuple(step), yaw=yaw)
    fr = P.DeviceFrames.from_numpy(*_pack(seq)).voxel_downsample(0.2).estimate_normals(15)
    res = fr.icp_point_to_plane(np.c_[np.arange(1, n), np.arange(n - 1)], max_iterations=30, tolerance=0.0)
    poses = P.chain_poses(res)
    world = fr.apply_transform(poses).merge().voxel_downsample(0.1).to_numpy()
    assert len(world) > 1000

    vox, v_off = fr.to_numpy()
    # the per-frame way: DeviceCloud.apply_transform, download, host concatenation, single voxel call
    slow = np.vstack([fr.frame(f).apply_transform(*_rt(poses[f])).to_numpy() for f in range(n)])
    assert world.tobytes() == pcr.voxel_downsample(P.PointCloud.from_numpy(slow), 0.1).to_numpy().tobytes()
    # the oracle
    moved = np.vstack([O.apply_transform(vox[int(v_off[f]):int(v_off[f + 1])], *_rt(poses[f])) for f in range(n)])
    assert world.tobytes() == O.voxel_downsample(moved, 0.1).tobytes()

    # the chained poses against the generator's: pose i = (rot_z(yaw * i), step * i)
    rot_err, trans_err = 0.0, 0.0
    for i in range(n):
        R, t = _rt(poses[i].astype(np.float64))
        d = R @ scenes.rot_z(yaw * i).astype(np.float64).T
        rot_err = max(rot_err, float(np.arccos(np.clip((np.trace(d) - 1.0) / 2.0, -1.0, 1.0))))
        trans_err = max(trans_err, float(np.linalg.norm(t - step * i)))
    # measured on a B200: at most 3.18e-3 rad and 6.29e-2 m over the 8 poses (the drift of 7 chained registrations of
    # 1 cm-jittered, voxelised frames); the bounds leave about 3x margin
    assert rot_err < 1e-2, f"rotation drift {rot_err:.3e} rad"
    assert trans_err < 0.2, f"translation drift {trans_err:.3e} m"


# ---- GPU: C error codes -----------------------------------------------------------------------------------------

@gpu
def test_errors(pcr):
    pts, off = _pack([scenes.hemisphere(300, 1), scenes.hemisphere(200, 2)])
    lib, h = _ffi.load(), pcr.default_context()._h
    x, y, z = (np.ascontiguousarray(pts[:, j]) for j in range(3))
    o = [np.zeros(len(pts), np.float32) for _ in range(3)]
    f = lambda a: a.ctypes.data_as(_ffi.f32p)
    u64 = lambda a: a.ctypes.data_as(_ffi.u64p)
    tr = _random_transforms(2, seed=1)
    call = lambda ctx, offs, nf, t, xs=(x, y, z), os_=o: lib.pcr_apply_transform_batch(ctx, *(f(a) if a is not None else None for a in xs),
                                                                                      offs, nf, t, *(f(a) for a in os_))
    assert call(h, u64(off), 2, f(tr)) == _ffi.PCR_OK
    assert call(None, u64(off), 2, f(tr)) == _ffi.PCR_ERR_INVALID_ARG
    assert call(h, u64(off), 2, None) == _ffi.PCR_ERR_INVALID_ARG
    assert call(h, u64(off), 2, f(tr), xs=(x, None, z)) == _ffi.PCR_ERR_INVALID_ARG
    assert call(h, None, 2, f(tr)) == _ffi.PCR_ERR_INVALID_ARG
    for bad in (np.array([0, 400, 300], np.uint64), np.array([1, 300, 500], np.uint64)):
        assert call(h, u64(bad), 2, f(tr)) == _ffi.PCR_ERR_INVALID_ARG
        assert "frame_offsets" in _ffi.last_error(h)
        assert lib.pcr_apply_transform_batch_dev(h, None, None, None, u64(bad), 2, f(tr), None, None, None) == _ffi.PCR_ERR_INVALID_ARG
        assert "frame_offsets" in _ffi.last_error(h)
    many = np.zeros(65537, np.uint64)  # 65536 empty frames
    many_tr = np.zeros((65536, 12), np.float32)
    assert call(h, u64(many), 65536, f(many_tr)) == _ffi.PCR_ERR_UNSUPPORTED
    zero = np.zeros(1, np.uint64)
    assert call(h, u64(zero), 0, None) == _ffi.PCR_OK
    assert lib.pcr_apply_transform_batch_dev(h, None, None, None, u64(zero), 0, None, None, None, None) == _ffi.PCR_OK

    fr = C.c_void_p()
    assert lib.pcr_frames_upload(h, x.ctypes.data, y.ctypes.data, z.ctypes.data, u64(off), 2, C.byref(fr)) == _ffi.PCR_OK
    try:
        out = C.c_void_p(1234)
        assert lib.pcr_frames_apply_transform(fr, None, C.byref(out)) == _ffi.PCR_ERR_INVALID_ARG and out.value is None
        out = C.c_void_p(1234)
        assert lib.pcr_frames_apply_transform(None, f(tr), C.byref(out)) == _ffi.PCR_ERR_INVALID_ARG and out.value is None
        assert lib.pcr_frames_apply_transform(fr, f(tr), None) == _ffi.PCR_ERR_INVALID_ARG
        cl = C.c_void_p(1234)
        assert lib.pcr_frames_merge(None, C.byref(cl)) == _ffi.PCR_ERR_INVALID_ARG and cl.value is None
        assert lib.pcr_frames_merge(fr, None) == _ffi.PCR_ERR_INVALID_ARG
        assert lib.pcr_frames_apply_transform(fr, f(tr), C.byref(out)) == _ffi.PCR_OK and out.value
        lib.pcr_frames_free(out)
        assert lib.pcr_frames_merge(fr, C.byref(cl)) == _ffi.PCR_OK and cl.value
        lib.pcr_cloud_free(cl)
    finally:
        lib.pcr_frames_free(fr)
