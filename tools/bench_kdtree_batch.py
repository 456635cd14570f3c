"""Batch index (pcr_index_build_batch / pcr_knn_batch ...) against a loop of single calls on the same frames (DESIGN 3.10, 6).

Workloads:
  sequence   kitti_sequence(100) after voxel 0.2 (the batch voxel call, outside the timing): frames 1..99 queried against
             an index of frames 0..98 (scan t against scan t-1), k = 1 and k = 10.
  config4    BASELINE configs[4] frames (100 x 80 K, kitti_scene seeds 0..99), queries = the frame's points with seeded
             Gaussian jitter (sigma 2 cm): KNN at k = 16 and k = 64, radius count r = 0.5 and CSR radius search r = 0.3.
  one_frame  one raw 122 K-point frame and its jittered copy as a batch of one, KNN k = 10.
KNN rows: the batch arm is pcr_index_build_batch_dev + pcr_knn_batch_dev on device buffers, the loop arm
pcr_index_build_dev + pcr_knn_dev per frame on slices of the SAME buffers ("build+query"); a second row times the queries
alone against indexes built once before ("query").  Radius rows use the host forms of both arms (pcr_radius_count_batch /
pcr_radius_search_batch against pcr_radius_count / pcr_radius_search per frame; there is no single-frame device form),
with the indexes prebuilt.  Every arm ends with a synchronise of the context; the two arms alternate in one process after
warm-up, and the median and min / max over --reps repetitions are reported.  Every row compares the two arms' outputs bit
for bit (indices, distance bits, counts, CSR).  One JSON line; --out FILE also writes it.
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

u32p = lambda a: a.ctypes.data_as(_ffi.u32p)  # noqa: E731
u64p = lambda a: a.ctypes.data_as(_ffi.u64p)  # noqa: E731
f32p = lambda a: a.ctypes.data_as(_ffi.f32p)  # noqa: E731


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


def timed(ctx, arms, reps, warmup):
    """arms: {name: fn() -> outputs}.  Alternating repetitions after warm-up -> ({name: times}, {name: last outputs})."""
    for _ in range(warmup):
        for fn in arms.values():
            fn()
            ctx.synchronize()
    ts, outs = {k: [] for k in arms}, {}
    for _ in range(reps):
        for k, fn in arms.items():
            torch.cuda.synchronize()
            ctx.synchronize()
            t0 = time.perf_counter()
            outs[k] = fn()
            ctx.synchronize()
            ts[k].append((time.perf_counter() - t0) * 1e3)
    return ts, outs


def compare_row(name, ts, identical, extra=None):
    b, l = np.median(ts["batch"]), np.median(ts["loop"])
    row = {"row": name, "batch_ms": stats(ts["batch"]), "loop_ms": stats(ts["loop"]), "speedup_median": round(float(l / b), 3),
           "identical": bool(identical)}
    row.update(extra or {})
    print(json.dumps(row), file=sys.stderr)
    return row


class Side:
    """Frames back to back: host rows and SoA, device x | y | z, offsets on the host."""

    def __init__(self, pts, off):
        self.pts = np.ascontiguousarray(pts, np.float32)
        self.off = np.ascontiguousarray(off, np.uint64)
        self.F, self.n = len(off) - 1, len(pts)
        self.soa = [np.ascontiguousarray(self.pts[:, j]) for j in range(3)]
        self.xyz = [torch.from_numpy(a).cuda() for a in self.soa]
        torch.cuda.synchronize()

    def ptrs(self, f=None):
        b = 0 if f is None else int(self.off[f]) * 4
        return [C.c_void_p(t.data_ptr() + b) for t in self.xyz]

    def size(self, f):
        return int(self.off[f + 1] - self.off[f])


def pack(frames):
    off = np.zeros(len(frames) + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in frames])
    return np.vstack(frames).astype(np.float32), off


# ---- index builds --------------------------------------------------------------------------------------------------

def build_batch(ctx, ix, k_hint):
    h = C.c_void_p()
    _ffi.check(_ffi.load().pcr_index_build_batch_dev(ctx._h, *ix.ptrs(), u64p(ix.off), ix.F, k_hint, C.byref(h)), ctx._h)
    return h


def build_loop(ctx, ix, k_hint):
    lib, hs = _ffi.load(), []
    for f in range(ix.F):
        h = C.c_void_p()
        _ffi.check(lib.pcr_index_build_dev(ctx._h, *ix.ptrs(f), ix.size(f), k_hint, C.byref(h)), ctx._h)
        hs.append(h)
    return hs


def free_all(hs):
    for h in hs:
        _ffi.load().pcr_index_free(h)


# ---- KNN -----------------------------------------------------------------------------------------------------------

class KnnOut:
    def __init__(self, nq, k):
        self.k = k
        self.idx = torch.zeros(max(nq * k, 1), dtype=torch.int32, device="cuda")
        self.dist = torch.zeros(max(nq * k, 1), dtype=torch.float32, device="cuda")
        self.cnt = torch.zeros(max(nq, 1), dtype=torch.int32, device="cuda")

    def ptrs(self, q0=0):
        return (C.c_void_p(self.idx.data_ptr() + q0 * self.k * 4), C.c_void_p(self.dist.data_ptr() + q0 * self.k * 4),
                C.c_void_p(self.cnt.data_ptr() + q0 * 4))

    def host(self):
        return (self.idx.cpu().numpy().view(np.uint32).copy(), self.dist.cpu().numpy().view(np.uint32).copy(),
                self.cnt.cpu().numpy().view(np.uint32).copy())


def knn_batch(ctx, h, qs, k, out):
    _ffi.check(_ffi.load().pcr_knn_batch_dev(h, *qs.ptrs(), u64p(qs.off), qs.F, k, *out.ptrs()), ctx._h)


def knn_loop(ctx, hs, qs, k, out):
    lib = _ffi.load()
    for f, h in enumerate(hs):
        _ffi.check(lib.pcr_knn_dev(h, *qs.ptrs(f), qs.size(f), k, *out.ptrs(int(qs.off[f]))), ctx._h)


def knn_rows(ctx, a, label, ix, qs, k):
    ob, ol = KnnOut(qs.n, k), KnnOut(qs.n, k)
    extra = {"frames": ix.F, "points": ix.n, "queries": qs.n, "k": k}

    def batch_full():
        h = build_batch(ctx, ix, k)
        knn_batch(ctx, h, qs, k, ob)
        ctx.synchronize()
        free_all([h])

    def loop_full():
        hs = build_loop(ctx, ix, k)
        knn_loop(ctx, hs, qs, k, ol)
        ctx.synchronize()
        free_all(hs)

    rows = []
    ts, _ = timed(ctx, {"batch": batch_full, "loop": loop_full}, a.reps, a.warmup)
    hb, hl = ob.host(), ol.host()
    rows.append(compare_row(f"{label}_knn{k}_build_query", ts, all(np.array_equal(x, y) for x, y in zip(hb, hl)), extra))
    h = build_batch(ctx, ix, k)
    hs = build_loop(ctx, ix, k)
    ctx.synchronize()
    ob.idx.zero_(), ol.idx.zero_()
    ts, _ = timed(ctx, {"batch": lambda: knn_batch(ctx, h, qs, k, ob), "loop": lambda: knn_loop(ctx, hs, qs, k, ol)}, a.reps, a.warmup)
    hb, hl = ob.host(), ol.host()
    rows.append(compare_row(f"{label}_knn{k}_query", ts, all(np.array_equal(x, y) for x, y in zip(hb, hl)), extra))
    free_all([h] + hs)
    return rows


# ---- radius (host forms) -------------------------------------------------------------------------------------------

def radius_rows(ctx, a, label, ix, qs, r_count, r_search):
    lib = _ffi.load()
    h = build_batch(ctx, ix, 0)
    hs = build_loop(ctx, ix, 0)
    ctx.synchronize()
    extra = {"frames": ix.F, "points": ix.n, "queries": qs.n}
    cb, cl = np.zeros(qs.n, np.uint32), np.zeros(qs.n, np.uint32)

    def count_batch():
        _ffi.check(lib.pcr_radius_count_batch(h, *(f32p(x) for x in qs.soa), u64p(qs.off), qs.F, r_count, u32p(cb)), ctx._h)

    def count_loop():
        for f, hf in enumerate(hs):
            b = int(qs.off[f])
            _ffi.check(lib.pcr_radius_count(hf, *(f32p(x[b:]) for x in qs.soa), qs.size(f), r_count, u32p(cl[b:])), ctx._h)

    rows = []
    ts, _ = timed(ctx, {"batch": count_batch, "loop": count_loop}, a.reps, a.warmup)
    rows.append(compare_row(f"{label}_radius_count_r{r_count}", ts, np.array_equal(cb, cl), dict(extra, neighbours=int(cb.sum()))))

    def search_batch():
        off, total = np.zeros(qs.n + 1, np.uint64), C.c_size_t()
        st = lib.pcr_radius_search_batch(h, *(f32p(x) for x in qs.soa), u64p(qs.off), qs.F, r_search, u64p(off), None, 0, C.byref(total))
        if st != _ffi.PCR_ERR_CAPACITY and st != _ffi.PCR_OK:
            _ffi.check(st, ctx._h)
        idx = np.zeros(max(total.value, 1), np.uint32)
        _ffi.check(lib.pcr_radius_search_batch(h, *(f32p(x) for x in qs.soa), u64p(qs.off), qs.F, r_search, u64p(off), u32p(idx), total.value,
                                               C.byref(total)), ctx._h)
        return off, idx[:total.value]

    def search_loop():
        outs = []
        for f, hf in enumerate(hs):
            b, m = int(qs.off[f]), qs.size(f)
            off, total = np.zeros(m + 1, np.uint64), C.c_size_t()
            st = lib.pcr_radius_search(hf, *(f32p(x[b:]) for x in qs.soa), m, r_search, u64p(off), None, 0, C.byref(total))
            if st != _ffi.PCR_ERR_CAPACITY and st != _ffi.PCR_OK:
                _ffi.check(st, ctx._h)
            idx = np.zeros(max(total.value, 1), np.uint32)
            _ffi.check(lib.pcr_radius_search(hf, *(f32p(x[b:]) for x in qs.soa), m, r_search, u64p(off), u32p(idx), total.value, C.byref(total)),
                       ctx._h)
            outs.append((off, idx[:total.value]))
        return outs

    ts, o = timed(ctx, {"batch": search_batch, "loop": search_loop}, a.reps, a.warmup)
    off_b, idx_b = o["batch"]
    ident = True
    for f, (off_l, idx_l) in enumerate(o["loop"]):
        b, e = int(qs.off[f]), int(qs.off[f + 1])
        ident &= np.array_equal(off_b[b:e + 1] - off_b[b], off_l) and np.array_equal(idx_b[int(off_b[b]):int(off_b[e])], idx_l)
    rows.append(compare_row(f"{label}_radius_search_r{r_search}", ts, ident, dict(extra, neighbours=int(off_b[-1]))))
    free_all([h] + hs)
    return rows


def jittered(frames, seed):
    rng = np.random.default_rng(seed)
    return [(f + rng.normal(0.0, 0.02, f.shape)).astype(np.float32) for f in frames]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", default="sequence,config4,one_frame")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_kdtree_batch: no CUDA device (the measurement needs a B200)")
    ctx = pcr.default_context()
    info = gpu_info()
    rows = []
    only = a.only.split(",")
    if "sequence" in only:
        pts, off = pack(scenes.kitti_sequence(a.frames))
        vox, v_off = pcr.voxel_downsample_batch(pts, off, 0.2, ctx=ctx)
        frames = [vox[int(v_off[f]):int(v_off[f + 1])] for f in range(a.frames)]
        ix, qs = Side(*pack(frames[:-1])), Side(*pack(frames[1:]))
        for k in (1, 10):
            rows += knn_rows(ctx, a, "sequence", ix, qs, k)
        del ix, qs
        torch.cuda.empty_cache()
    if "config4" in only:
        frames = [scenes.kitti_scene(seed=f, counts=scenes.KITTI_COUNTS["frame80k"]) for f in range(a.frames)]
        ix, qs = Side(*pack(frames)), Side(*pack(jittered(frames, 2024)))
        for k in (16, 64):
            rows += knn_rows(ctx, a, "config4", ix, qs, k)
        torch.cuda.empty_cache()
        rows += radius_rows(ctx, a, "config4", ix, qs, 0.5, 0.3)
        del ix, qs
        torch.cuda.empty_cache()
    if "one_frame" in only:
        one = scenes.kitti_scene(seed=0)
        ix, qs = Side(*pack([one])), Side(*pack(jittered([one], 7)))
        rows += knn_rows(ctx, a, "one_frame", ix, qs, 10)
    line = {"tool": "bench_kdtree_batch", "gpu": info, "reps": a.reps, "warmup": a.warmup, "rows": rows,
            "all_identical": all(r["identical"] for r in rows)}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
