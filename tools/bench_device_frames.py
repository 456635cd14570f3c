"""Device-resident frame batches (DeviceFrames) against the other ways to chain the batch calls (DESIGN 3.9, 6).

Workloads (BASELINE configs[4] frames: 100 x 80 K, kitti_scene seeds 0..99):
  obstacle   upload -> voxel 0.15 -> SOR 20 / 2.0 -> RANSAC 0.15 with 500 triples per frame and the outliers -> cluster
             (0.8, 10, 20000) -> the clusters on the host.  Arms: `frames` (DeviceFrames), `raw` (the _dev batch calls
             on torch buffers with torch compactions in between, as tools/bench_obstacle_batch.py removes the ground) and
             `loop` (one DeviceCloud per frame through the same chain).  The triples are drawn once, outside the timing,
             for the frame sizes the chain produces.
  odometry   kitti_sequence(100): upload -> voxel 0.2 -> normals 15 -> point-to-plane ICP over the 99 pairs (i+1, i), 30
             iterations.  Arms: `frames` and `raw` (the three _dev batch calls of tools/bench_frontend_batch.py).
  ror        radius_outlier_removal (2.0, 5) of 16 aerial tiles (aerial_scene seeds 0..15, 0.1 scale, 241 K points each):
             `frames` (upload, filter, download) against `loop` (a DeviceCloud per tile through the same steps).
  one        a batch of one 80 K frame for each filter (voxel 0.15, SOR 20 / 2.0, radius 0.5 / 5, normals 15, SOR ->
             normals 20 / 2.0 / 15), on resident data: DeviceFrames against DeviceCloud.
Every timed call ends in a host result (host clock, synchronous).  The arms alternate after warm-up; median, min and max
over --reps repetitions.  The arms' outputs are compared bit for bit on every row.  One JSON line; --out FILE also
writes it.
"""
import argparse
import ctypes as C
import json
import os
import sys

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import pointclouds_rs_b200 as pcr  # noqa: E402
from pointclouds_rs_b200 import _ffi, scenes  # noqa: E402
from bench_obstacle_batch import gpu_info, stats, timed, cluster_csr, cluster_from_device, same_clusters  # noqa: E402

VOXEL, K_SOR, STD_MUL, PLANE_THR, TRIPLES, CLUSTER = 0.15, 20, 2.0, 0.15, 500, (0.8, 10, 20_000)
u32p = lambda a: a.ctypes.data_as(_ffi.u32p)  # noqa: E731
u64p = lambda a: a.ctypes.data_as(_ffi.u64p)  # noqa: E731
f32p = lambda a: a.ctypes.data_as(_ffi.f32p)  # noqa: E731
VP = np.zeros(3, np.float32)


def pack(frames):
    off = np.zeros(len(frames) + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in frames])
    return np.ascontiguousarray(np.vstack(frames), np.float32), off


def row(name, ts, identical, extra=None):
    r = {"row": name, "identical": bool(identical)}
    r.update({f"{k}_ms": stats(v) for k, v in ts.items()})
    if "frames" in ts:
        for k in ts:
            if k != "frames":
                r[f"{k}_over_frames"] = round(float(np.median(ts[k]) / np.median(ts["frames"])), 3)
    r.update(extra or {})
    print(json.dumps(r), file=sys.stderr)
    return r


def icp_bits(rs):
    return [(np.float32(r.rotation).tobytes(), np.float32(r.translation).tobytes(), r.num_iterations) for r in rs]


# ---- obstacle pipeline -----------------------------------------------------------------------------------------------

def obstacle_frames(ctx, pts, off, samples):
    s = pcr.DeviceFrames.from_numpy(pts, off, ctx).voxel_downsample(VOXEL).statistical_outlier_removal(K_SOR, STD_MUL)
    planes, rest = s.ransac_plane_samples(PLANE_THR, samples, outliers=True)
    c_off, offsets, idx = rest.cluster_arrays(*CLUSTER)
    return [np.float32(p.normal + [p.d]) for p in planes], cluster_csr(c_off, offsets, idx)


def frame_ids(counts_np, total):
    counts = torch.from_numpy(counts_np.astype(np.int64)).cuda()
    return torch.repeat_interleave(torch.arange(len(counts_np), device="cuda"), counts, output_size=total)


def obstacle_raw(ctx, pts, off, samples):
    lib, F = _ffi.load(), len(off) - 1
    rows = torch.from_numpy(pts).cuda()
    x, y, z = (rows[:, j].contiguous() for j in range(3))
    n = len(pts)
    v = [torch.empty(n, dtype=torch.float32, device="cuda") for _ in range(3)]
    v_off = np.zeros(F + 1, np.uint64)
    _ffi.check(lib.pcr_voxel_downsample_batch_dev(ctx._h, x.data_ptr(), y.data_ptr(), z.data_ptr(), u64p(off), F, VOXEL,
                                                  *(t.data_ptr() for t in v), u64p(v_off)), ctx._h)
    m = int(v_off[-1])
    v = [t[:m] for t in v]
    keep = torch.empty(max(m, 1), dtype=torch.uint8, device="cuda")
    _ffi.check(lib.pcr_sor_normals_batch_dev(ctx._h, *(t.data_ptr() for t in v), u64p(v_off), F, K_SOR, STD_MUL, 0, f32p(VP),
                                             keep.data_ptr(), None, None, None), ctx._h)
    kb = keep[:m].bool()
    s = [t[kb] for t in v]
    kept = torch.zeros(F, dtype=torch.int64, device="cuda").index_add_(0, frame_ids(np.diff(v_off), m), kb.long()).cpu().numpy()
    k_off = np.zeros(F + 1, np.uint64)
    k_off[1:] = np.cumsum(kept)
    smp = np.ascontiguousarray(np.vstack(samples), np.uint32)
    s_off = np.zeros(F + 1, np.uint64)
    s_off[1:] = np.cumsum([len(t) for t in samples])
    models, io = np.zeros((F, 4), np.float32), np.zeros(F + 1, np.uint64)
    d_inl = torch.empty(max(int(k_off[-1]), 1), dtype=torch.int32, device="cuda")
    _ffi.check(lib.pcr_ransac_plane_samples_batch_dev(ctx._h, *(t.data_ptr() for t in s), u64p(k_off), F, PLANE_THR, u32p(smp), u64p(s_off),
                                                      f32p(models), d_inl.data_ptr(), u64p(io)), ctx._h)
    k = int(io[-1])
    starts = torch.from_numpy(k_off[:-1].astype(np.int64)).cuda()
    ground = torch.ones(int(k_off[-1]), dtype=torch.bool, device="cuda")
    ground[d_inl[:k].long() + starts[frame_ids(np.diff(io), k)]] = False
    rest = [t[ground] for t in s]
    r_off = (k_off.astype(np.int64) - io.astype(np.int64)).astype(np.uint64)
    nr = int(r_off[-1])
    d_offsets = torch.empty(nr + 1, dtype=torch.int32, device="cuda")
    d_idx = torch.empty(max(nr, 1), dtype=torch.int32, device="cuda")
    co = np.zeros(F + 1, np.uint64)
    _ffi.check(lib.pcr_euclidean_cluster_batch_dev(ctx._h, *(t.data_ptr() for t in rest), u64p(r_off), F, CLUSTER[0], CLUSTER[1], CLUSTER[2],
                                                   d_offsets.data_ptr(), d_idx.data_ptr(), u64p(co)), ctx._h)
    return list(models), cluster_from_device(co, d_offsets, d_idx)


def obstacle_loop(ctx, pts, off, samples):
    models, out = [], []
    for f in range(len(off) - 1):
        c = pcr.DeviceCloud.from_numpy(pts[int(off[f]):int(off[f + 1])], ctx).voxel_downsample(VOXEL).statistical_outlier_removal(K_SOR, STD_MUL)
        p = c.ransac_plane_samples(PLANE_THR, samples[f])
        models.append(np.float32(p.normal + [p.d]))
        rest = c.select(np.setdiff1d(np.arange(len(c)), p.inliers))  # (DeviceCloud's select_inverse)
        o, i = np.zeros(len(rest) + 1, np.uint32), np.zeros(max(len(rest), 1), np.uint32)
        nc = C.c_size_t()
        _ffi.check(_ffi.load().pcr_cloud_euclidean_cluster(rest._h, CLUSTER[0], CLUSTER[1], CLUSTER[2], u32p(o), u32p(i), C.byref(nc)), ctx._h)
        kk = int(nc.value)
        out.append((o[:kk + 1].copy(), i[:int(o[kk])].copy()))
    return models, out


def obstacle(ctx, a, frames):
    pts, off = pack(frames)
    sizes = np.diff(pcr.DeviceFrames.from_numpy(pts, off, ctx).voxel_downsample(VOXEL).statistical_outlier_removal(K_SOR, STD_MUL).offsets)
    samples = [pcr.draw_plane_samples(int(sizes[f]), TRIPLES, [2024, f]) for f in range(len(frames))]
    ts, o = timed({"frames": lambda: obstacle_frames(ctx, pts, off, samples), "raw": lambda: obstacle_raw(ctx, pts, off, samples),
                   "loop": lambda: obstacle_loop(ctx, pts, off, samples)}, a.reps, a.warmup)
    same = lambda p, q: all(x.tobytes() == y.tobytes() for x, y in zip(p[0], q[0])) and same_clusters(p[1], q[1])  # noqa: E731
    return row("obstacle_pipeline", ts, same(o["frames"], o["raw"]) and same(o["frames"], o["loop"]),
               {"frames": len(frames), "points": len(pts), "clusters": sum(len(c[0]) - 1 for c in o["frames"][1])})


# ---- odometry front end ----------------------------------------------------------------------------------------------

def odometry(ctx, a):
    seq = scenes.kitti_sequence(a.frames)
    pts, off = pack(seq)
    F = len(seq)
    pairs = np.array([(i + 1, i) for i in range(F - 1)], np.uint32)
    prm = _ffi.IcpParams(30, 0.0, float("inf"))
    lib = _ffi.load()

    def frames_arm():
        return icp_bits(pcr.DeviceFrames.from_numpy(pts, off, ctx).voxel_downsample(0.2).estimate_normals(15)
                        .icp_point_to_plane(pairs, max_iterations=30, tolerance=0.0))

    def raw_arm():
        rows = torch.from_numpy(pts).cuda()
        xyz = [rows[:, j].contiguous() for j in range(3)]
        v = [torch.empty(len(pts), dtype=torch.float32, device="cuda") for _ in range(3)]
        v_off = np.zeros(F + 1, np.uint64)
        _ffi.check(lib.pcr_voxel_downsample_batch_dev(ctx._h, *(t.data_ptr() for t in xyz), u64p(off), F, 0.2, *(t.data_ptr() for t in v),
                                                      u64p(v_off)), ctx._h)
        nrm = [torch.empty(len(pts), dtype=torch.float32, device="cuda") for _ in range(3)]
        _ffi.check(lib.pcr_estimate_normals_batch_dev(ctx._h, *(t.data_ptr() for t in v), u64p(v_off), F, 15, f32p(VP),
                                                      *(t.data_ptr() for t in nrm)), ctx._h)
        res = (_ffi.IcpResultC * len(pairs))()
        _ffi.check(lib.pcr_icp_point_to_plane_batch_dev(ctx._h, *(t.data_ptr() for t in v), u64p(v_off), F, *(t.data_ptr() for t in nrm),
                                                        int(v_off[-1]), u32p(pairs), len(pairs), C.byref(prm), res), ctx._h)
        return icp_bits([pcr.IcpResult(r) for r in res])

    ts, o = timed({"frames": frames_arm, "raw": raw_arm}, a.reps, a.warmup)
    return row("odometry_front_end", ts, o["frames"] == o["raw"], {"frames": F, "points": len(pts), "pairs": len(pairs)})


# ---- radius outlier removal over aerial tiles ------------------------------------------------------------------------

def ror(ctx, a):
    tiles = [scenes.aerial_scene(seed=s) for s in range(a.tiles)]
    pts, off = pack(tiles)

    def frames_arm():
        return pcr.DeviceFrames.from_numpy(pts, off, ctx).radius_outlier_removal(2.0, 5).to_numpy()[0]

    def loop_arm():
        return np.vstack([pcr.DeviceCloud.from_numpy(t, ctx).radius_outlier_removal(2.0, 5).to_numpy() for t in tiles])

    ts, o = timed({"frames": frames_arm, "loop": loop_arm}, a.reps, a.warmup)
    return row("ror_aerial_tiles", ts, o["frames"].tobytes() == o["loop"].tobytes(), {"frames": len(tiles), "points": len(pts),
                                                                                       "kept": len(o["frames"])})


# ---- a batch of one ----------------------------------------------------------------------------------------------------

def one(ctx, a):
    fr = scenes.kitti_scene(seed=0, counts=scenes.KITTI_COUNTS["frame80k"])
    batch = pcr.DeviceFrames.from_numpy(fr, [0, len(fr)], ctx)
    cloud = pcr.DeviceCloud.from_numpy(fr, ctx)
    out = []
    for name, fn in (("voxel", lambda x: x.voxel_downsample(VOXEL)), ("sor", lambda x: x.statistical_outlier_removal(K_SOR, STD_MUL)),
                     ("ror", lambda x: x.radius_outlier_removal(0.5, 5)), ("normals", lambda x: x.estimate_normals(15)),
                     ("sor_normals", lambda x: x.sor_normals(K_SOR, STD_MUL, 15))):
        def arm(x, fn=fn):
            r = fn(x)
            p = r.to_numpy()
            p = p[0] if isinstance(p, tuple) else p
            nrm = r.normals_to_numpy()
            return p.tobytes() + (b"" if nrm is None else nrm.tobytes())

        ts, o = timed({"frames": lambda: arm(batch), "cloud": lambda: arm(cloud)}, a.reps, a.warmup)
        out.append(row(f"one_frame_{name}", ts, o["frames"] == o["cloud"], {"points": len(fr)}))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--tiles", type=int, default=16)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", default="obstacle,odometry,ror,one")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_device_frames: no CUDA device (the measurement needs a B200)")
    ctx = pcr.default_context()
    info = gpu_info()
    only = a.only.split(",")
    rows = []
    if "obstacle" in only:
        rows.append(obstacle(ctx, a, [scenes.kitti_scene(seed=f, counts=scenes.KITTI_COUNTS["frame80k"]) for f in range(a.frames)]))
        torch.cuda.empty_cache()
    if "odometry" in only:
        rows.append(odometry(ctx, a))
        torch.cuda.empty_cache()
    if "ror" in only:
        rows.append(ror(ctx, a))
    if "one" in only:
        rows += one(ctx, a)
    line = {"tool": "bench_device_frames", "gpu": info, "reps": a.reps, "warmup": a.warmup, "rows": rows,
            "all_identical": all(r["identical"] for r in rows)}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
