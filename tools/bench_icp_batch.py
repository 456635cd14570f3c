"""Batched ICP against a loop of single-pair calls on the same device buffers (DESIGN section 3.4).

Workload: a seeded sequence of KITTI-shaped frames (scenes.kitti_sequence: frame i+1 is frame i under a small rigid
motion, another point subset, 1 cm jitter), frame-to-frame registration of the consecutive pairs (i+1 onto i), target
normals from the product's estimate_normals (k = 15), tolerance 0 so that every pair runs exactly --iters iterations.
Each row times, alternately in the same process, ONE pcr_icp_point_to_*_batch_dev call and a loop of
pcr_icp_point_to_*_dev calls over the same pairs (both synchronous: host clock around the call), after warm-up, and
reports the median with the spread (min / max) over --reps repetitions.  Rows: point-to-plane and point-to-point on the
sequence, and one 1 M-point pair (aerial scene, BASELINE configs[3] shape) as a batch of one against the single call.
One JSON line; --out FILE also writes it there.  --stages adds the per-stage device times (pcr_ctx_set_timing) of one
extra call of each kind, taken after the timed repetitions.
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


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_clock_max_mhz": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_clock_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:  # (the row still names the card)
        info["query_error"] = str(e)
    return info


class Workload:
    """Frames back to back on the device (torch tensors: x | y | z | nx | ny | nz), frame offsets and pairs on the host."""

    def __init__(self, frames, pairs, k_normals=15):
        off = np.zeros(len(frames) + 1, np.uint64)
        off[1:] = np.cumsum([len(f) for f in frames])
        pts = np.ascontiguousarray(np.vstack(frames), np.float32)
        nrm = np.vstack([pcr.normals_array(pcr.PointCloud.from_numpy(f), k_normals) for f in frames]).astype(np.float32)
        self.off, self.n, self.pairs = off, len(pts), np.ascontiguousarray(pairs, np.uint32)
        self.dev = [torch.from_numpy(np.ascontiguousarray(a[:, j])).cuda() for a in (pts, nrm) for j in range(3)]
        torch.cuda.synchronize()
        self.ptr = [t.data_ptr() for t in self.dev]
        self.src_points = int(sum(off[s + 1] - off[s] for s, _ in self.pairs))

    def batch(self, ctx, plane, prm):
        res = (_ffi.IcpResultC * len(self.pairs))()
        lib, x, y, z, nx, ny, nz = _ffi.load(), *self.ptr
        op, pp = self.off.ctypes.data_as(_ffi.u64p), self.pairs.ctypes.data_as(_ffi.u32p)
        if plane:
            st = lib.pcr_icp_point_to_plane_batch_dev(ctx._h, x, y, z, op, len(self.off) - 1, nx, ny, nz, self.n, pp, len(self.pairs),
                                                      C.byref(prm), res)
        else:
            st = lib.pcr_icp_point_to_point_batch_dev(ctx._h, x, y, z, op, len(self.off) - 1, pp, len(self.pairs), C.byref(prm), res)
        _ffi.check(st, ctx._h)
        return list(res)

    def loop(self, ctx, plane, prm):
        lib, out = _ffi.load(), []
        for s, t in self.pairs:
            bs, ns, bt, nt = int(self.off[s]), int(self.off[s + 1] - self.off[s]), int(self.off[t]), int(self.off[t + 1] - self.off[t])
            sx, sy, sz = (p + 4 * bs for p in self.ptr[:3])
            tx, ty, tz, nx, ny, nz = (p + 4 * bt for p in self.ptr)
            r = _ffi.IcpResultC()
            if plane:
                st = lib.pcr_icp_point_to_plane_dev(ctx._h, sx, sy, sz, ns, tx, ty, tz, nt, nx, ny, nz, nt, C.byref(prm), C.byref(r))
            else:
                st = lib.pcr_icp_point_to_point_dev(ctx._h, sx, sy, sz, ns, tx, ty, tz, nt, C.byref(prm), C.byref(r))
            _ffi.check(st, ctx._h)
            out.append(r)
        return out


def stats(ts):
    return {"median": round(float(np.median(ts)), 3), "min": round(float(min(ts)), 3), "max": round(float(max(ts)), 3)}


def row(ctx, w, plane, iters, reps, warmup, want_stages):
    prm = _ffi.IcpParams(iters, 0.0, float("inf"))
    for _ in range(warmup):
        w.batch(ctx, plane, prm)
        w.loop(ctx, plane, prm)
    tb, tl = [], []
    for _ in range(reps):  # alternating, same process
        t0 = time.perf_counter()
        rb = w.batch(ctx, plane, prm)
        tb.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        rl = w.loop(ctx, plane, prm)
        tl.append((time.perf_counter() - t0) * 1e3)
    dr = max(float(np.abs(np.array(a.rotation) - np.array(b.rotation)).max()) for a, b in zip(rb, rl))
    dt = max(float(np.abs(np.array(a.translation) - np.array(b.translation)).max()) for a, b in zip(rb, rl))
    its = [int(r.num_iterations) for r in rb]
    assert its == [int(r.num_iterations) for r in rl], "iteration counts of the two ways differ"
    work = sum(int(w.off[s + 1] - w.off[s]) * it for (s, _), it in zip(w.pairs, its))  # source points x iterations
    P = len(w.pairs)
    out = {
        "kind": "point_to_plane" if plane else "point_to_point", "pairs": P, "frames": len(w.off) - 1,
        "points_per_frame": int(w.n // (len(w.off) - 1)), "iterations": iters,
        "batch_ms_per_call": stats(tb), "loop_ms_per_call": stats(tl),
        "batch_ms_per_pair": round(float(np.median(tb)) / P, 4), "loop_ms_per_pair": round(float(np.median(tl)) / P, 4),
        "batch_src_point_iters_per_s": round(work / (float(np.median(tb)) * 1e-3)),
        "loop_src_point_iters_per_s": round(work / (float(np.median(tl)) * 1e-3)),
        "speedup_median": round(float(np.median(tl)) / float(np.median(tb)), 3),
        "max_abs_diff_rotation": dr, "max_abs_diff_translation": dt,
    }
    if want_stages:
        st = {}
        for name, fn in (("batch", w.batch), ("loop", w.loop)):
            ctx.set_timing(True)
            ctx.get_timing()
            fn(ctx, plane, prm)
            tm = ctx.get_timing()
            ctx.set_timing(False)
            st[name] = {k: round(v[0], 3) for k, v in tm.items() if v[1]}
        out["stages_ms"] = st
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--points", type=int, default=122_000, help="points per frame (KITTI frame122k proportions)")
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--large", type=float, default=0.415, help="aerial scene scale of the single large pair (0 = skip)")
    ap.add_argument("--stages", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_icp_batch: no CUDA device (the measurement needs a B200)")
    ctx = pcr.default_context()
    base = scenes.KITTI_COUNTS["frame122k"]
    counts = tuple(max(1, round(c * a.points / scenes.kitti_points(base))) for c in base)
    seq = Workload(scenes.kitti_sequence(a.frames, seed=7, counts=counts), [(i + 1, i) for i in range(a.frames - 1)])
    rows = [row(ctx, seq, True, a.iters, a.reps, a.warmup, a.stages), row(ctx, seq, False, a.iters, a.reps, a.warmup, a.stages)]
    del seq
    if a.large > 0:
        tgt = scenes.aerial_scene(42, a.large)
        src = (tgt.astype(np.float64) @ scenes.rot_z(0.05).T.astype(np.float64) + [0.3, -0.2, 0.1]).astype(np.float32)
        big = Workload([src, tgt], [(0, 1)])
        rows.append(row(ctx, big, True, a.iters, a.reps, a.warmup, a.stages))
    line = {"tool": "bench_icp_batch", "gpu": gpu_info(), "sequence_points": scenes.kitti_points(counts), "rows": rows}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
