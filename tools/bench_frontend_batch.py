"""Batched voxel_downsample / estimate_normals against loops of single calls on the same device buffers (DESIGN 3.6).

Workloads:
  configs4   BASELINE configs[4] frames (100 x 80 K, kitti_scene seeds 0..99): the voxel batch at 0.05, and the voxel
             batch -> pcr_sor_normals_batch_dev (k_sor 10, std 1.0, k_normals 20, the configs[1] chain) against a
             loop of pcr_voxel_downsample_dev calls (-> the same sor_normals_batch_dev call on the loop's output).
  odometry   scenes.kitti_sequence of 100 122 K-point frames: voxel batch at 0.2 -> normals batch k = 15 ->
             point-to-plane ICP batch over the 99 consecutive pairs (30 iterations, tolerance 0), against loops of
             the single _dev calls for each stage.  Each stage and the whole chain are timed.
  one_frame  one 122 K-point frame as a batch of one against the single calls (voxel 0.05, normals k = 15).
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

K_SOR, STD_MUL, K_NORMALS = 10, 1.0, 20


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


def dev(n):
    return [torch.zeros(max(n, 1), dtype=torch.float32, device="cuda") for _ in range(3)]


def ptrs(ts, first=0):
    return [t.data_ptr() + 4 * first for t in ts]


def host(ts, n):
    return np.stack([t[:n].cpu().numpy() for t in ts], axis=1)


class Frames:
    """Frames back to back on the device (x | y | z), offsets on the host."""

    def __init__(self, frames):
        self.off = np.zeros(len(frames) + 1, np.uint64)
        self.off[1:] = np.cumsum([len(f) for f in frames])
        pts = np.ascontiguousarray(np.vstack(frames), np.float32)
        self.n = len(pts)
        self.xyz = [torch.from_numpy(np.ascontiguousarray(pts[:, j])).cuda() for j in range(3)]
        torch.cuda.synchronize()


def voxel_batch(ctx, fr, voxel, out):
    o = np.zeros(len(fr.off), np.uint64)
    st = _ffi.load().pcr_voxel_downsample_batch_dev(ctx._h, *ptrs(fr.xyz), fr.off.ctypes.data_as(_ffi.u64p), len(fr.off) - 1, float(voxel),
                                                    *ptrs(out), o.ctypes.data_as(_ffi.u64p))
    _ffi.check(st, ctx._h)
    return o


def voxel_loop(ctx, fr, voxel, out):
    lib, o, m = _ffi.load(), np.zeros(len(fr.off), np.uint64), C.c_size_t()
    for f in range(len(fr.off) - 1):
        b, n = int(fr.off[f]), int(fr.off[f + 1] - fr.off[f])
        st = lib.pcr_voxel_downsample_dev(ctx._h, *ptrs(fr.xyz, b), n, float(voxel), *ptrs(out, int(o[f])), C.byref(m))
        _ffi.check(st, ctx._h)
        o[f + 1] = o[f] + m.value
    return o


def normals_batch(ctx, xyz, off, k, nrm):
    vp = np.zeros(3, np.float32)
    st = _ffi.load().pcr_estimate_normals_batch_dev(ctx._h, *ptrs(xyz), off.ctypes.data_as(_ffi.u64p), len(off) - 1, k,
                                                    vp.ctypes.data_as(_ffi.f32p), *ptrs(nrm))
    _ffi.check(st, ctx._h)
    ctx.synchronize()


def normals_loop(ctx, xyz, off, k, nrm):
    lib, vp = _ffi.load(), np.zeros(3, np.float32)
    for f in range(len(off) - 1):
        b, n = int(off[f]), int(off[f + 1] - off[f])
        st = lib.pcr_estimate_normals_dev(ctx._h, *ptrs(xyz, b), n, k, vp.ctypes.data_as(_ffi.f32p), *ptrs(nrm, b))
        _ffi.check(st, ctx._h)
    ctx.synchronize()


def sor_normals(ctx, xyz, off, keep, nrm):
    vp = np.zeros(3, np.float32)
    pcr.sor_normals_batch_raw(ctx, *ptrs(xyz), int(off[-1]), off, K_SOR, STD_MUL, K_NORMALS, vp, keep.data_ptr(), *ptrs(nrm), device=True)
    ctx.synchronize()


def icp_batch(ctx, xyz, off, nrm, pairs, prm):
    res = (_ffi.IcpResultC * len(pairs))()
    st = _ffi.load().pcr_icp_point_to_plane_batch_dev(ctx._h, *ptrs(xyz), off.ctypes.data_as(_ffi.u64p), len(off) - 1, *ptrs(nrm), int(off[-1]),
                                                      pairs.ctypes.data_as(_ffi.u32p), len(pairs), C.byref(prm), res)
    _ffi.check(st, ctx._h)
    return list(res)


def icp_loop(ctx, xyz, off, nrm, pairs, prm):
    lib, out = _ffi.load(), []
    for s, t in pairs:
        bs, ns, bt, nt = int(off[s]), int(off[s + 1] - off[s]), int(off[t]), int(off[t + 1] - off[t])
        r = _ffi.IcpResultC()
        st = lib.pcr_icp_point_to_plane_dev(ctx._h, *ptrs(xyz, bs), ns, *ptrs(xyz, bt), nt, *ptrs(nrm, bt), nt, C.byref(prm), C.byref(r))
        _ffi.check(st, ctx._h)
        out.append(r)
    return out


def icp_bits(rs):
    return [(np.float32(list(r.rotation)).tobytes(), np.float32(list(r.translation)).tobytes(), np.float32(r.rmse).tobytes(),
             np.float32(r.fitness).tobytes(), int(r.num_iterations), int(r.converged)) for r in rs]


def icp_diff(ra, rb):
    """Largest transform difference of two result lists (0.0 when identical)."""
    dr = max((float(np.abs(np.array(a.rotation) - np.array(b.rotation)).max()) for a, b in zip(ra, rb)), default=0.0)
    dt = max((float(np.abs(np.array(a.translation) - np.array(b.translation)).max()) for a, b in zip(ra, rb)), default=0.0)
    return {"max_abs_diff_rotation": dr, "max_abs_diff_translation": dt}


def same(a, b):
    return bool(a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32)))


def timed(arms, reps, warmup):
    """arms: {name: fn() -> outputs}.  Alternating repetitions after warm-up -> ({name: times}, {name: last outputs})."""
    for _ in range(warmup):
        for fn in arms.values():
            fn()
    ts, outs = {k: [] for k in arms}, {}
    for _ in range(reps):
        for k, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            outs[k] = fn()
            ts[k].append((time.perf_counter() - t0) * 1e3)
    return ts, outs


def compare_row(name, ts, identical, extra=None):
    b, l = np.median(ts["batch"]), np.median(ts["loop"])
    row = {"row": name, "batch_ms": stats(ts["batch"]), "loop_ms": stats(ts["loop"]), "speedup_median": round(float(l / b), 3),
           "outputs_identical": identical}
    row.update(extra or {})
    print(json.dumps(row), file=sys.stderr)
    return row


def configs4(ctx, a):
    fr = Frames([scenes.kitti_scene(seed=f, counts=scenes.KITTI_COUNTS["frame80k"]) for f in range(a.frames)])
    vb, vl = dev(fr.n), dev(fr.n)
    keep_b, keep_l = (torch.zeros(max(fr.n, 1), dtype=torch.uint8, device="cuda") for _ in range(2))
    nb, nl = dev(fr.n), dev(fr.n)
    rows = []
    ts, o = timed({"batch": lambda: voxel_batch(ctx, fr, 0.05, vb), "loop": lambda: voxel_loop(ctx, fr, 0.05, vl)}, a.reps, a.warmup)
    m = int(o["batch"][-1])
    ident = bool(np.array_equal(o["batch"], o["loop"]) and same(host(vb, m), host(vl, m)))
    rows.append(compare_row("configs4_voxel_0.05", ts, ident, {"frames": a.frames, "points": fr.n, "voxels": m}))

    def chain(arm):
        v, keep, nrm = (vb, keep_b, nb) if arm == "batch" else (vl, keep_l, nl)
        off = voxel_batch(ctx, fr, 0.05, v) if arm == "batch" else voxel_loop(ctx, fr, 0.05, v)
        sor_normals(ctx, v, off, keep, nrm)
        return off

    ts, o = timed({"batch": lambda: chain("batch"), "loop": lambda: chain("loop")}, a.reps, a.warmup)
    m = int(o["batch"][-1])
    ident = bool(np.array_equal(o["batch"], o["loop"]) and torch.equal(keep_b[:m], keep_l[:m]) and same(host(nb, m), host(nl, m)))
    rows.append(compare_row("configs4_voxel_0.05_then_sor_normals_batch", ts, ident, {"frames": a.frames, "voxels": m}))
    return rows


def odometry(ctx, a):
    base = scenes.KITTI_COUNTS["frame122k"]
    fr = Frames(scenes.kitti_sequence(a.frames, seed=7, counts=base))
    pairs = np.ascontiguousarray([(i + 1, i) for i in range(a.frames - 1)], np.uint32)
    prm = _ffi.IcpParams(a.iters, 0.0, float("inf"))
    bufs = {arm: (dev(fr.n), dev(fr.n)) for arm in ("batch", "loop")}
    offs = {}

    def stage(arm, what):
        v, nrm = bufs[arm]
        if what == "voxel":
            offs[arm] = voxel_batch(ctx, fr, 0.2, v) if arm == "batch" else voxel_loop(ctx, fr, 0.2, v)
            return offs[arm]
        if what == "normals":
            (normals_batch if arm == "batch" else normals_loop)(ctx, v, offs[arm], 15, nrm)
            return None
        return (icp_batch if arm == "batch" else icp_loop)(ctx, v, offs[arm], nrm, pairs, prm)

    rows, outs = [], {}
    for what in ("voxel", "normals", "icp"):
        ts, o = timed({arm: (lambda arm=arm: stage(arm, what)) for arm in ("batch", "loop")}, a.reps, a.warmup)
        outs[what] = o
        m = int(offs["batch"][-1])
        if what == "voxel":
            ident = bool(np.array_equal(o["batch"], o["loop"]) and same(host(bufs["batch"][0], m), host(bufs["loop"][0], m)))
        elif what == "normals":
            ident = same(host(bufs["batch"][1], m), host(bufs["loop"][1], m))
        else:
            ident = icp_bits(o["batch"]) == icp_bits(o["loop"])
        extra = {"frames": a.frames, "points": fr.n, "voxels": m}
        if what == "icp":
            extra.update(icp_diff(o["batch"], o["loop"]), pairs=len(pairs), iterations=a.iters)
        rows.append(compare_row(f"odometry_{what}", ts, ident, extra))

    def chain(arm):
        stage(arm, "voxel")
        stage(arm, "normals")
        return stage(arm, "icp")

    ts, o = timed({"batch": lambda: chain("batch"), "loop": lambda: chain("loop")}, a.reps, a.warmup)
    rows.append(compare_row("odometry_chain", ts, icp_bits(o["batch"]) == icp_bits(o["loop"]),
                            dict(icp_diff(o["batch"], o["loop"]), frames=a.frames, pairs=len(pairs), iterations=a.iters)))
    return rows


def one_frame(ctx, a):
    fr = Frames([scenes.kitti_scene(seed=0)])
    vb, vl, nb, nl = dev(fr.n), dev(fr.n), dev(fr.n), dev(fr.n)
    rows = []
    ts, o = timed({"batch": lambda: voxel_batch(ctx, fr, 0.05, vb), "loop": lambda: voxel_loop(ctx, fr, 0.05, vl)}, a.reps, a.warmup)
    m = int(o["batch"][-1])
    rows.append(compare_row("one_frame_voxel_0.05", ts, bool(np.array_equal(o["batch"], o["loop"]) and same(host(vb, m), host(vl, m))),
                            {"points": fr.n}))
    ts, _ = timed({"batch": lambda: normals_batch(ctx, fr.xyz, fr.off, 15, nb), "loop": lambda: normals_loop(ctx, fr.xyz, fr.off, 15, nl)},
                  a.reps, a.warmup)
    rows.append(compare_row("one_frame_normals_k15", ts, same(host(nb, fr.n), host(nl, fr.n)), {"points": fr.n}))
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", default="configs4,odometry,one_frame")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_frontend_batch: no CUDA device (the measurement needs a B200)")
    ctx = pcr.default_context()
    info = gpu_info()
    rows = []
    for name, fn in (("configs4", configs4), ("odometry", odometry), ("one_frame", one_frame)):
        if name in a.only.split(","):
            rows += fn(ctx, a)
            torch.cuda.empty_cache()
    line = {"tool": "bench_frontend_batch", "gpu": info, "reps": a.reps, "warmup": a.warmup, "rows": rows,
            "all_outputs_identical": all(r["outputs_identical"] for r in rows)}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
