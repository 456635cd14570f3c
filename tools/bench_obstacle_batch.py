"""Batched RANSAC plane fit and euclidean_cluster against loops of single calls (DESIGN 3.5, 3.8, 6).

Workloads:
  obstacle   BASELINE configs[4] frames (100 x 80 K, kitti_scene seeds 0..99) put through voxel 0.15 -> SOR 20 / 2.0 with
             the existing batches once, outside the timing; 500 triples per frame drawn once with fixed seeds.  Timed:
             the RANSAC batch _dev (0.15) against a loop of pcr_cloud_ransac_plane_samples on resident per-frame clouds;
             the cluster batch _dev (0.8, 10, 20000) on the non-ground points against a loop of
             pcr_cloud_euclidean_cluster; the two steps together (the batch arm removes the ground with torch on the
             device, the loop arm with the library's device select of each resident cloud); and the host-pointer forms
             from numpy, the batch against a loop of pcr_ransac_plane_samples / pcr_euclidean_cluster.
  raw        the cluster batch on the 100 raw frames, ground left in, at (0.5, 30, 25000): the union-find's worst case.
  one_frame  one raw 122 K-point frame as a batch of one against the single calls, with the rows of `obstacle` (RANSAC
             500 triples at 0.15; clustering of its non-ground points at (0.8, 10, 20000)).
Every timed call is synchronous (host clock around the call and a synchronise).  The two arms alternate in one
process after warm-up; the median and min / max over --reps repetitions are reported, and the two arms' outputs
(model bits, inlier lists, cluster CSR per frame) are compared bit for bit.  One JSON line; --out FILE also writes it.
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

VOXEL, K_SOR, STD_MUL = 0.15, 20, 2.0
PLANE_THR, TRIPLES = 0.15, 500
CLUSTER = (0.8, 10, 20_000)
RAW_CLUSTER = (0.5, 30, 25_000)

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
           "identical": bool(identical)}
    row.update(extra or {})
    print(json.dumps(row), file=sys.stderr)
    return row


class Frames:
    """Frames back to back: host rows, device x | y | z, offsets on the host, and one resident pcr cloud per frame."""

    def __init__(self, ctx, pts, off):
        self.pts = np.ascontiguousarray(pts, np.float32)
        self.off = np.ascontiguousarray(off, np.uint64)
        self.F, self.n = len(off) - 1, len(pts)
        self.soa = [np.ascontiguousarray(self.pts[:, j]) for j in range(3)]
        self.xyz = [torch.from_numpy(a).cuda() for a in self.soa]
        torch.cuda.synchronize()
        self.clouds = [pcr.DeviceCloud.from_numpy(self.pts[int(off[f]):int(off[f + 1])], ctx) for f in range(self.F)]

    def sizes(self):
        return [int(self.off[f + 1] - self.off[f]) for f in range(self.F)]

    def ptrs(self):
        return [t.data_ptr() for t in self.xyz]


def stack_triples(samples):
    s_off = np.zeros(len(samples) + 1, np.uint64)
    s_off[1:] = np.cumsum([len(s) for s in samples])
    return np.ascontiguousarray(np.vstack(samples), np.uint32), s_off


# ---- RANSAC arms ---------------------------------------------------------------------------------------------------

def ransac_batch_dev(ctx, fr, smp, s_off, d_inl):
    models, io = np.zeros((fr.F, 4), np.float32), np.zeros(fr.F + 1, np.uint64)
    st = _ffi.load().pcr_ransac_plane_samples_batch_dev(ctx._h, *fr.ptrs(), u64p(fr.off), fr.F, PLANE_THR, u32p(smp), u64p(s_off), f32p(models),
                                                        d_inl.data_ptr(), u64p(io))
    _ffi.check(st, ctx._h)
    return models, io


def ransac_batch_host(ctx, fr, smp, s_off, h_inl):
    models, io = np.zeros((fr.F, 4), np.float32), np.zeros(fr.F + 1, np.uint64)
    st = _ffi.load().pcr_ransac_plane_samples_batch(ctx._h, *(f32p(a) for a in fr.soa), u64p(fr.off), fr.F, PLANE_THR, u32p(smp), u64p(s_off),
                                                    f32p(models), u32p(h_inl), u64p(io))
    _ffi.check(st, ctx._h)
    return models, [h_inl[int(io[f]):int(io[f + 1])].copy() for f in range(fr.F)]


def ransac_loop(ctx, fr, samples, device=True):
    lib, models, inls = _ffi.load(), np.zeros((fr.F, 4), np.float32), []
    for f, n in enumerate(fr.sizes()):
        smp, k, inl = np.ascontiguousarray(samples[f], np.uint32), C.c_size_t(), np.zeros(max(n, 1), np.uint32)
        if device:
            st = lib.pcr_cloud_ransac_plane_samples(fr.clouds[f]._h, PLANE_THR, u32p(smp), len(smp), f32p(models[f]), u32p(inl), C.byref(k))
        else:
            b = int(fr.off[f])
            st = lib.pcr_ransac_plane_samples(ctx._h, *(f32p(a[b:]) for a in fr.soa), n, PLANE_THR, u32p(smp), len(smp), f32p(models[f]),
                                              u32p(inl), C.byref(k))
        _ffi.check(st, ctx._h)
        inls.append(inl[:k.value].copy())
    return models, inls


def same_ransac(a_models, a_inls, b_models, b_inls):
    return bool(np.array_equal(a_models.view(np.uint32), b_models.view(np.uint32)) and len(a_inls) == len(b_inls)
                and all(np.array_equal(x, y) for x, y in zip(a_inls, b_inls)))


# ---- clustering arms -----------------------------------------------------------------------------------------------

def cluster_batch_dev(ctx, ptrs, off, args, d_offsets, d_idx):
    co = np.zeros(len(off), np.uint64)
    st = _ffi.load().pcr_euclidean_cluster_batch_dev(ctx._h, *ptrs, u64p(off), len(off) - 1, float(args[0]), args[1], args[2],
                                                     d_offsets.data_ptr(), d_idx.data_ptr(), u64p(co))
    _ffi.check(st, ctx._h)
    return co


def cluster_csr(co, offsets, idx):
    """per frame: (offsets rebased to 0, indices)"""
    out = []
    for f in range(len(co) - 1):
        a, b = int(co[f]), int(co[f + 1])
        o = offsets[a:b + 1] - offsets[a]
        out.append((o, idx[int(offsets[a]):int(offsets[b])]))
    return out


def cluster_from_device(co, d_offsets, d_idx):
    k = int(co[-1])
    offsets = d_offsets[:k + 1].cpu().numpy().view(np.uint32)
    return cluster_csr(co, offsets, d_idx[:int(offsets[-1])].cpu().numpy().view(np.uint32))


def cluster_batch_host(ctx, fr, args, h_offsets, h_idx):
    co = np.zeros(fr.F + 1, np.uint64)
    st = _ffi.load().pcr_euclidean_cluster_batch(ctx._h, *(f32p(a) for a in fr.soa), u64p(fr.off), fr.F, float(args[0]), args[1], args[2],
                                                 u32p(h_offsets), u32p(h_idx), u64p(co))
    _ffi.check(st, ctx._h)
    return cluster_csr(co, h_offsets, h_idx)


def cluster_one(ctx, cloud_h, n, args, x=None):
    """one frame through pcr_cloud_euclidean_cluster (resident cloud) or pcr_euclidean_cluster (x = host SoA)"""
    lib, nc = _ffi.load(), C.c_size_t()
    o, i = np.zeros(n + 1, np.uint32), np.zeros(max(n, 1), np.uint32)
    if x is None:
        st = lib.pcr_cloud_euclidean_cluster(cloud_h, float(args[0]), args[1], args[2], u32p(o), u32p(i), C.byref(nc))
    else:
        st = lib.pcr_euclidean_cluster(ctx._h, *(f32p(a) for a in x), n, float(args[0]), args[1], args[2], u32p(o), u32p(i), C.byref(nc))
    _ffi.check(st, ctx._h)
    k = int(nc.value)
    return o[:k + 1].copy(), i[:int(o[k])].copy()


def cluster_loop(ctx, fr, args, device=True):
    out = []
    for f, n in enumerate(fr.sizes()):
        if device:
            out.append(cluster_one(ctx, fr.clouds[f]._h, n, args))
        else:
            b = int(fr.off[f])
            out.append(cluster_one(ctx, None, n, args, [a[b:b + n] for a in fr.soa]))
    return out


def same_clusters(a, b):
    return len(a) == len(b) and all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) for x, y in zip(a, b))


# ---- workloads -----------------------------------------------------------------------------------------------------

def preprocess(ctx, frames):
    """voxel batch -> SOR batch once (outside the timing) -> the kept points of every frame, back to back"""
    pts, off = np.vstack(frames).astype(np.float32), np.zeros(len(frames) + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in frames])
    vox, v_off = pcr.voxel_downsample_batch(pts, off, VOXEL, ctx=ctx)
    keep, _, kept = pcr.sor_normals_batch(vox, v_off, K_SOR, STD_MUL, 0, ctx=ctx)
    k_off = np.zeros(len(frames) + 1, np.uint64)
    k_off[1:] = np.cumsum(kept)
    return vox[keep.astype(bool)], k_off


def ground_removed(fr, io, inls_dev):
    """select_inverse of every frame's inliers, with torch on the device -> (x, y, z tensors, offsets)"""
    k = int(io[-1])
    counts = torch.from_numpy(np.diff(io).astype(np.int64)).cuda()
    starts = torch.from_numpy(fr.off[:-1].astype(np.int64)).cuda()
    fid = torch.repeat_interleave(torch.arange(fr.F, device="cuda"), counts, output_size=k)
    keep = torch.ones(fr.n, dtype=torch.bool, device="cuda")
    keep[inls_dev[:k].long() + starts[fid]] = False
    r_off = (fr.off.astype(np.int64) - io.astype(np.int64)).astype(np.uint64)
    return [t[keep] for t in fr.xyz], r_off


def obstacle_rows(ctx, a, pts, off, label, samples):
    fr = Frames(ctx, pts, off)
    smp, s_off = stack_triples(samples)
    d_inl = torch.zeros(max(fr.n, 1), dtype=torch.int32, device="cuda")
    rows = []
    extra = {"frames": fr.F, "points": fr.n, "triples_per_frame": TRIPLES}

    ts, o = timed({"batch": lambda: ransac_batch_dev(ctx, fr, smp, s_off, d_inl), "loop": lambda: ransac_loop(ctx, fr, samples)},
                  a.reps, a.warmup)
    models, io = o["batch"]
    inls = [d_inl[int(io[f]):int(io[f + 1])].cpu().numpy().view(np.uint32) for f in range(fr.F)]
    rows.append(compare_row(f"{label}_ransac_dev", ts, same_ransac(models, inls, *o["loop"]), dict(extra, inliers=int(io[-1]))))

    # the non-ground points of every frame, on the device and as resident clouds
    rest, r_off = ground_removed(fr, io, d_inl)
    rest_np = np.stack([t.cpu().numpy() for t in rest], 1)
    ng = Frames(ctx, rest_np, r_off)
    d_offsets = torch.zeros(ng.n + 1, dtype=torch.int32, device="cuda")
    d_idx = torch.zeros(max(ng.n, 1), dtype=torch.int32, device="cuda")
    ts, o = timed({"batch": lambda: cluster_batch_dev(ctx, ng.ptrs(), ng.off, CLUSTER, d_offsets, d_idx),
                   "loop": lambda: cluster_loop(ctx, ng, CLUSTER)}, a.reps, a.warmup)
    got = cluster_from_device(o["batch"], d_offsets, d_idx)
    rows.append(compare_row(f"{label}_cluster_dev", ts, same_clusters(got, o["loop"]),
                            dict(frames=ng.F, points=ng.n, clusters=int(o["batch"][-1]))))

    c_offsets = torch.zeros(fr.n + 1, dtype=torch.int32, device="cuda")
    c_idx = torch.zeros(max(fr.n, 1), dtype=torch.int32, device="cuda")

    def chain_batch():
        m, io_b = ransac_batch_dev(ctx, fr, smp, s_off, d_inl)
        xyz, off = ground_removed(fr, io_b, d_inl)
        co = cluster_batch_dev(ctx, [t.data_ptr() for t in xyz], off, CLUSTER, c_offsets, c_idx)
        return m, co

    def chain_loop():
        lib, models_l, out = _ffi.load(), np.zeros((fr.F, 4), np.float32), []
        for f, n in enumerate(fr.sizes()):
            smp_f, k, inl = np.ascontiguousarray(samples[f], np.uint32), C.c_size_t(), np.zeros(max(n, 1), np.uint32)
            _ffi.check(lib.pcr_cloud_ransac_plane_samples(fr.clouds[f]._h, PLANE_THR, u32p(smp_f), len(smp_f), f32p(models_l[f]), u32p(inl),
                                                          C.byref(k)), ctx._h)
            keep = np.ones(n, bool)
            keep[inl[:k.value]] = False
            rest_idx = np.flatnonzero(keep).astype(np.uint32)
            h = C.c_void_p()
            _ffi.check(lib.pcr_cloud_select(fr.clouds[f]._h, u32p(rest_idx), len(rest_idx), C.byref(h)), ctx._h)
            out.append(cluster_one(ctx, h, len(rest_idx), CLUSTER))
            lib.pcr_cloud_free(h)
        return models_l, out

    ts, o = timed({"batch": chain_batch, "loop": chain_loop}, a.reps, a.warmup)
    ident = bool(np.array_equal(o["batch"][0].view(np.uint32), o["loop"][0].view(np.uint32))
                 and same_clusters(cluster_from_device(o["batch"][1], c_offsets, c_idx), o["loop"][1]))
    rows.append(compare_row(f"{label}_ransac_then_cluster_dev", ts, ident, dict(extra, clusters=int(o["batch"][1][-1]))))

    h_inl = np.zeros(max(fr.n, 1), np.uint32)
    ts, o = timed({"batch": lambda: ransac_batch_host(ctx, fr, smp, s_off, h_inl), "loop": lambda: ransac_loop(ctx, fr, samples, False)},
                  a.reps, a.warmup)
    rows.append(compare_row(f"{label}_ransac_host", ts, same_ransac(*o["batch"], *o["loop"]), extra))
    h_offsets, h_idx = np.zeros(ng.n + 1, np.uint32), np.zeros(max(ng.n, 1), np.uint32)
    ts, o = timed({"batch": lambda: cluster_batch_host(ctx, ng, CLUSTER, h_offsets, h_idx), "loop": lambda: cluster_loop(ctx, ng, CLUSTER, False)},
                  a.reps, a.warmup)
    rows.append(compare_row(f"{label}_cluster_host", ts, same_clusters(o["batch"], o["loop"]), dict(frames=ng.F, points=ng.n)))
    for c in fr.clouds + ng.clouds:
        c.free()
    return rows


def raw_rows(ctx, a, frames):
    pts = np.vstack(frames).astype(np.float32)
    off = np.zeros(len(frames) + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in frames])
    fr = Frames(ctx, pts, off)
    d_offsets = torch.zeros(fr.n + 1, dtype=torch.int32, device="cuda")
    d_idx = torch.zeros(max(fr.n, 1), dtype=torch.int32, device="cuda")
    ts, o = timed({"batch": lambda: cluster_batch_dev(ctx, fr.ptrs(), fr.off, RAW_CLUSTER, d_offsets, d_idx),
                   "loop": lambda: cluster_loop(ctx, fr, RAW_CLUSTER)}, a.reps, a.warmup)
    row = compare_row("raw_cluster_dev", ts, same_clusters(cluster_from_device(o["batch"], d_offsets, d_idx), o["loop"]),
                      dict(frames=fr.F, points=fr.n, clusters=int(o["batch"][-1]), params=list(RAW_CLUSTER)))
    for c in fr.clouds:
        c.free()
    return [row]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", default="obstacle,raw,one_frame")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_obstacle_batch: no CUDA device (the measurement needs a B200)")
    ctx = pcr.default_context()
    info = gpu_info()
    rows = []
    only = a.only.split(",")
    frames = [scenes.kitti_scene(seed=f, counts=scenes.KITTI_COUNTS["frame80k"]) for f in range(a.frames)]
    if "obstacle" in only:
        kept, k_off = preprocess(ctx, frames)
        samples = [pcr.draw_plane_samples(int(k_off[f + 1] - k_off[f]), TRIPLES, [2024, f]) for f in range(len(frames))]
        rows += obstacle_rows(ctx, a, kept, k_off, "obstacle", samples)
        torch.cuda.empty_cache()
    if "raw" in only:
        rows += raw_rows(ctx, a, frames)
        torch.cuda.empty_cache()
    if "one_frame" in only:
        one = scenes.kitti_scene(seed=0)  # the raw 122 K-point frame
        rows += obstacle_rows(ctx, a, one, np.array([0, len(one)], np.uint64), "one_frame", [pcr.draw_plane_samples(len(one), TRIPLES, [2024, 0])])
    line = {"tool": "bench_obstacle_batch", "gpu": info, "reps": a.reps, "warmup": a.warmup, "rows": rows,
            "all_identical": all(r["identical"] for r in rows)}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
