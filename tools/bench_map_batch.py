"""Batched apply_transform and the device-side map assembly against per-frame calls (DESIGN 3.11).

Workloads:
  transform  BASELINE configs[4] frames (100 x 80 K, kitti_scene seeds 0..99): one pcr_apply_transform_batch_dev call
             against 100 pcr_cloud_apply_transform calls on resident per-frame clouds, a different transform per frame.
             Two copies of the input alternate between repetitions (2 x 96 MB in, 96 MB out: more than the 126 MB L2),
             and the batch row reports bytes/s at 24 B per point (12 read, 12 written) and its share of 7.7 TB/s.
  map        scenes.kitti_sequence of 100 122 K-point frames through voxel 0.2 -> normals k = 15 -> point-to-plane ICP
             over the 99 consecutive pairs (30 iterations, tolerance 0), computed once; then the map assembly is timed:
             chain_poses -> DeviceFrames.apply_transform -> merge -> voxel_downsample(0.1), against the per-frame way
             (frame(f) -> DeviceCloud.apply_transform -> download, host concatenation, upload, voxel_downsample(0.1)).
             The whole chain (voxel, normals, ICP and the assembly, from the resident upload) is timed the same way;
             its two arms differ only in the assembly.
  one_frame  one 122 K-point frame: pcr_frames_apply_transform on a batch of one against pcr_cloud_apply_transform.
Every timed call is synchronous (host clock around the call and a synchronise).  The two arms alternate in one
process after warm-up; the median and min / max over --reps repetitions are reported, and the two arms' outputs
are compared bit for bit.  One JSON line; --out FILE also writes it there.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import pointclouds_rs_b200 as pcr  # noqa: E402
from pointclouds_rs_b200 import _ffi, scenes  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU
BYTES_PER_POINT = 24      # x, y, z read and written once


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_clock_max_mhz": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_clock_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:  # (the row still names the card)
        info["query_error"] = str(e)
    return info


def stats(ts):
    return {"median": round(float(np.median(ts)), 3), "min": round(float(min(ts)), 3), "max": round(float(max(ts)), 3)}


def timed(arms, reps, warmup, release=None):
    """arms: {name: fn(rep) -> outputs}.  Alternating repetitions after warm-up -> ({name: times}, {name: last outputs}).
    release(name, outputs), if given, frees the outputs of every repetition but the last, outside the timed window."""
    outs = {}
    for w in range(warmup):
        for k, fn in arms.items():
            o = fn(w)
            if release:
                release(k, o)
    ts = {k: [] for k in arms}
    for r in range(reps):
        for k, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o = fn(r)
            ts[k].append((time.perf_counter() - t0) * 1e3)
            if release and r < reps - 1:
                release(k, o)
            else:
                outs[k] = o
    return ts, outs


def compare_row(name, ts, identical, extra=None):
    b, l = np.median(ts["batch"]), np.median(ts["loop"])
    row = {"row": name, "batch_ms": stats(ts["batch"]), "loop_ms": stats(ts["loop"]), "speedup_median": round(float(l / b), 3),
           "outputs_identical": identical}
    row.update(extra or {})
    print(json.dumps(row), file=sys.stderr)
    return row


def transforms(n, seed):
    """(n, 12) f32: rotations about a random axis by up to 0.5 rad and translations up to 5 m."""
    rng = np.random.default_rng(seed)
    out = np.zeros((n, 12), np.float32)
    for i in range(n):
        ax = rng.normal(size=3)
        ax /= np.linalg.norm(ax)
        a = rng.uniform(-0.5, 0.5)
        k = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
        out[i, :9] = (np.eye(3) + np.sin(a) * k + (1 - np.cos(a)) * k @ k).reshape(9)
        out[i, 9:] = rng.uniform(-5, 5, 3)
    return out


def dev_ptrs(ts, first=0):
    return [t.data_ptr() + 4 * first for t in ts]


def transform(ctx, a):
    lib, F = _ffi.load(), a.frames
    frames = [scenes.kitti_scene(seed=f, counts=scenes.KITTI_COUNTS["frame80k"]) for f in range(F)]
    off = np.zeros(F + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in frames])
    pts = np.ascontiguousarray(np.vstack(frames), np.float32)
    n = len(pts)
    tr = transforms(F, 1)
    inputs = [[torch.from_numpy(np.ascontiguousarray(pts[:, j])).cuda() for j in range(3)] for _ in range(2)]
    out = [torch.empty(n, dtype=torch.float32, device="cuda") for _ in range(3)]
    clouds = []  # two resident copies of every frame
    for copy in range(2):
        hs = []
        for f in range(F):
            h = C.c_void_p()
            b, e = int(off[f]), int(off[f + 1])
            cols = [np.ascontiguousarray(pts[b:e, j]) for j in range(3)]  # (alive until the upload has returned)
            _ffi.check(lib.pcr_cloud_upload(ctx._h, *(c.ctypes.data for c in cols), e - b, C.byref(h)), ctx._h)
            hs.append(h)
        clouds.append(hs)
    torch.cuda.synchronize()
    rt = [(np.ascontiguousarray(tr[f, :9]), np.ascontiguousarray(tr[f, 9:])) for f in range(F)]

    def batch(rep):
        st = lib.pcr_apply_transform_batch_dev(ctx._h, *dev_ptrs(inputs[rep % 2]), off.ctypes.data_as(_ffi.u64p), F,
                                               tr.ctypes.data_as(_ffi.f32p), *dev_ptrs(out))
        _ffi.check(st, ctx._h)
        ctx.synchronize()
        return None

    def loop(rep):
        res = []
        for f, h in enumerate(clouds[rep % 2]):
            o = C.c_void_p()
            _ffi.check(lib.pcr_cloud_apply_transform(h, rt[f][0].ctypes.data_as(_ffi.f32p), rt[f][1].ctypes.data_as(_ffi.f32p), C.byref(o)),
                       ctx._h)
            res.append(o)
        ctx.synchronize()
        return res

    def release(arm, o):
        for h in o or []:
            lib.pcr_cloud_free(h)

    ts, o = timed({"batch": batch, "loop": loop}, a.reps, a.warmup, release)
    got = np.stack([t.cpu().numpy() for t in out], axis=1)
    ref = np.zeros_like(got)
    for f, h in enumerate(o["loop"]):
        b, e = int(off[f]), int(off[f + 1])
        cols = [np.empty(e - b, np.float32) for _ in range(3)]
        _ffi.check(lib.pcr_cloud_download(h, *(c.ctypes.data_as(_ffi.f32p) for c in cols)), ctx._h)
        ref[b:e] = np.stack(cols, axis=1)
    release("loop", o["loop"])
    for hs in clouds:
        release("loop", hs)
    med_s = float(np.median(ts["batch"])) * 1e-3
    bw = BYTES_PER_POINT * n / med_s
    return [compare_row("transform_100x80k", ts, got.tobytes() == ref.tobytes(),
                        {"frames": F, "points": n, "batch_bytes_per_s": round(bw, 1), "batch_share_of_7.7TBps": round(bw / HBM_BYTES_PER_S, 4),
                         "input": "two copies alternated (192 MB in, 96 MB out)"})]


def map_rows(ctx, a):
    F = a.map_frames
    seq = scenes.kitti_sequence(F, seed=7, counts=scenes.KITTI_COUNTS["frame122k"])
    off = np.zeros(F + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in seq])
    pts = np.ascontiguousarray(np.vstack(seq), np.float32)
    up = pcr.DeviceFrames.from_numpy(pts, off, ctx=ctx)
    pairs = np.c_[np.arange(1, F), np.arange(F - 1)]

    def front():
        fr = up.voxel_downsample(0.2).estimate_normals(15)
        return fr, fr.icp_point_to_plane(pairs, max_iterations=a.iters, tolerance=0.0)

    def assemble_batch(fr, res):
        world = fr.apply_transform(pcr.chain_poses(res)).merge().voxel_downsample(0.1)
        ctx.synchronize()
        return world

    def assemble_loop(fr, res):
        poses = pcr.chain_poses(res)
        parts = [fr.frame(f).apply_transform(poses[f, :9].reshape(3, 3), poses[f, 9:]).to_numpy() for f in range(F)]
        world = pcr.DeviceCloud.from_numpy(np.ascontiguousarray(np.vstack(parts)), ctx=ctx).voxel_downsample(0.1)
        ctx.synchronize()
        return world

    fr, res = front()
    ctx.synchronize()
    ts, o = timed({"batch": lambda r: assemble_batch(fr, res), "loop": lambda r: assemble_loop(fr, res)}, a.reps, a.warmup)
    m = len(o["batch"])
    rows = [compare_row("map_assembly", ts, o["batch"].to_numpy().tobytes() == o["loop"].to_numpy().tobytes(),
                        {"frames": F, "points": int(off[-1]), "voxels_0.2": len(fr), "map_points_0.1": m})]
    ts, o = timed({"batch": lambda r: assemble_batch(*front()), "loop": lambda r: assemble_loop(*front())}, a.reps, a.warmup)
    rows.append(compare_row("map_whole_chain", ts, o["batch"].to_numpy().tobytes() == o["loop"].to_numpy().tobytes(),
                            {"frames": F, "pairs": F - 1, "iterations": a.iters, "map_points_0.1": len(o["batch"])}))
    return rows


def one_frame(ctx, a):
    lib = _ffi.load()
    p = scenes.kitti_scene(seed=0)
    fr = pcr.DeviceFrames.from_numpy(p, [0, len(p)], ctx=ctx)
    cl = pcr.DeviceCloud.from_numpy(p, ctx=ctx)
    tr = transforms(1, 2)
    r, t = np.ascontiguousarray(tr[0, :9]), np.ascontiguousarray(tr[0, 9:])

    def batch(rep):
        o = C.c_void_p()
        _ffi.check(lib.pcr_frames_apply_transform(fr._h, tr.ctypes.data_as(_ffi.f32p), C.byref(o)), ctx._h)
        ctx.synchronize()
        return pcr.DeviceFrames(o, ctx)

    def loop(rep):
        o = C.c_void_p()
        _ffi.check(lib.pcr_cloud_apply_transform(cl._h, r.ctypes.data_as(_ffi.f32p), t.ctypes.data_as(_ffi.f32p), C.byref(o)), ctx._h)
        ctx.synchronize()
        return pcr.DeviceCloud(o, ctx)

    ts, o = timed({"batch": batch, "loop": loop}, a.reps * 20, a.warmup * 5, lambda k, h: h.free())
    return [compare_row("one_frame_122k", ts, o["batch"].to_numpy()[0].tobytes() == o["loop"].to_numpy().tobytes(), {"points": len(p)})]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--map-frames", type=int, default=100)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", default="transform,map,one_frame")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_map_batch: no CUDA device (the measurement needs a B200)")
    ctx = pcr.default_context()
    info = gpu_info()
    rows = []
    for name, fn in (("transform", transform), ("map", map_rows), ("one_frame", one_frame)):
        if name in a.only.split(","):
            rows += fn(ctx, a)
            torch.cuda.empty_cache()
    line = {"tool": "bench_map_batch", "gpu": info, "reps": a.reps, "warmup": a.warmup, "rows": rows,
            "all_outputs_identical": all(r["outputs_identical"] for r in rows)}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
