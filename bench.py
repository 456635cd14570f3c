#!/usr/bin/env python3
"""bench.py -- the headline benchmark of the B200 KNN engine (driver contract: ONE JSON line).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): SOR + normals points/sec, k = 10 / 20; ICP ms/iter at 1 M points.

Headline workload at every N (weak scaling, one process per GPU, no data-path collective): BASELINE configs[1] --
KITTI-shaped synthetic frames of 122 000 points (numpy PCG64; every rank cycles through EIGHT different frames, so the
frame-stream hints of the library -- reused cell size, guessed voxel key box, coarser level built ahead -- can miss
and the line says how often they did); per step

    voxel_downsample(0.05) -> statistical_outlier_removal(k = 10, std_mul = 1.0) -> estimate_normals(k = 20)
    on the kept points

A step is one pass of that pipeline over one frame; points/s counts the RAW input points.
  value : points/s, the raw frames resident in HBM (pcr_cloud_voxel_downsample + pcr_cloud_sor_normals on a
          device-resident pcr_cloud), CUDA events on the stream the kernels run on, max over ranks; L2 is flushed
          between steps and the GPU is idle when the start event is recorded (launch latency is inside the number).
  e2e   : the same through the C ABI from PINNED host buffers: pcr_cloud_upload_block of x | y | z, the two calls,
          pcr_cloud_download_block of the kept points and their normals, all inside the timed region (wall clock).
  roofline     : the dominant kernel (grid KNN level 0, SOR mean distance + neighbour lists), algorithmic bytes / its
                 device time measured live with cudaEvents inside the library (pcr_ctx_get_timing), plus the FP32 /
                 issue view SURVEY 8d asks for (candidates per query counted by the kernel itself).
  cpu_baseline : the CPU oracle (C port of the reference path, gcc -O2) timed on this box's host cores on a bounded
                 sample, rank 0, N = 1 only.
Secondary blocks on the same line, at EVERY N (strong scaling: the total work is fixed, dealt over the ranks):
  batch8m     : BASELINE configs[4] -- 100 frames x 80 000 points, frames dealt round-robin, one pcr_sor_normals_batch
                call per rank; device-resident and host-API (pinned buffers, copies inside) points/s.
  icp_sharded : BASELINE configs[3] -- point-to-plane ICP, 1 M points, 30 iterations, the SOURCE sharded over the ranks,
                the 30-double normal equations all-reduced over NCCL inside the library every iteration; ms/iter and
                the checks of tests/multi_gpu_check.py (identical on all ranks, equal to the unsharded run).
  config3     : BASELINE configs[2] -- aerial 241 K points: normals k = 20, radius outlier removal and a radius-search
                CSR with the QUERIES sharded over the ranks (index replicated, results merged over NCCL), checked
                bit for bit against the one-GPU call.
--impl reference times the CPU port as the reference arm (the Rust reference cannot be built in this image: no
cargo/rustc; see DESIGN.md); at N ranks rank 0 processes N frames per step, so both arms do the same work.
--dump-outputs DIR writes what rank 0's last timed step of the headline returned, float32, after the timing:
  device_points.npy / device_normals.npy (kept points and their normals, (n_kept, 3), device-resident arm) and
  e2e_points.npy / e2e_normals.npy (the same from the host block of the end-to-end arm).  The frames are seeded, so
  two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: importing the package and the oracle writes nothing there

K_SOR, STD_MUL, K_NORMALS = 10, 1.0, 20
VOXEL = 0.05
METRIC = "sor_normals_points_per_sec"
UNIT = "points/s"
L2_FLUSH_BYTES = 256 << 20
FRAMES_PER_RANK = 8  # distinct frames every rank cycles through in both timed loops


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def frame_seed(rank: int, j: int) -> int:
    return 42 + FRAMES_PER_RANK * rank + j


def make_frames(rank: int, count: int = FRAMES_PER_RANK):
    from pointclouds_rs_b200 import scenes

    return [np.ascontiguousarray(scenes.kitti_scene(seed=frame_seed(rank, j)), np.float32) for j in range(count)]


def workload_config(n_raw: int, n_in: int, world: int):
    return {
        "workload": "BASELINE configs[1]: KITTI-shaped synthetic frame 122K pts: voxel 0.05 -> SOR k=10 -> normals",
        "points_per_step_per_gpu": n_raw,
        "points_after_voxel": n_in,
        "k_sor": K_SOR,
        "std_mul": STD_MUL,
        "k_normals": K_NORMALS,
        "frames_per_step_per_gpu": 1,
        "distinct_frames_per_gpu": FRAMES_PER_RANK,
        "sharding": f"frames: one independent frame per GPU per step x {world} GPU(s), no data-path collective",
        "l2": "256 MiB buffer overwritten between timed steps, GPU idle at the start event; the frame itself is L2-sized",
        "seed": f"numpy PCG64, 42 + {FRAMES_PER_RANK} * rank + (step mod {FRAMES_PER_RANK})",
        "frame_stream": "pcr_ctx_set_frame_stream(1): cell size / voxel key box / coarser level are carried from frame to frame; "
                        "hits and misses over the run are reported in frame_stream_hints",
    }


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8)),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40)),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20)),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)),
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2.0)
        return {
            "sm_mhz": float(np.median(self.samples)) if self.samples else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(self.samples),
        }


# ---------------------------------------------------------------------------------------------------
# CPU arm: the C port of the reference path (oracle/, gcc -O2 -ffp-contract=off)
# ---------------------------------------------------------------------------------------------------
def cpu_reference_run(frames, threads_normals: int):
    """One step = the pipeline over every frame of `frames`, threaded the way the reference is: voxel_downsample and
    SOR are serial loops (voxel_downsample.rs:24, statistical_outlier.rs:19), normals run on all cores (rayon
    par_iter, estimate.rs:42-44)."""
    from oracle import oracle as O  # the checker, used here only as the timed CPU baseline

    t0 = time.perf_counter()
    for raw in frames:
        pts = O.voxel_downsample(raw, VOXEL)
        keep, _, _ = O.sor(pts, K_SOR, STD_MUL, threads=1)
        O.normals(pts[keep.astype(bool)], K_NORMALS, threads=threads_normals)
    return time.perf_counter() - t0


def cpu_reference_all_threads(raw: np.ndarray, threads: int):
    from oracle import oracle as O

    t0 = time.perf_counter()
    pts = O.voxel_downsample(raw, VOXEL)
    keep, _, _ = O.sor(pts, K_SOR, STD_MUL, threads=threads)
    O.normals(pts[keep.astype(bool)], K_NORMALS, threads=threads)
    return time.perf_counter() - t0


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0  # the CPU arm runs on rank 0 only
    from oracle import oracle as O
    from pointclouds_rs_b200 import scenes

    O.lib()
    world = max(1, args.gpus)
    # the same work as the GPU arm at N ranks: N frames per step (the first frame of every rank)
    frames = [np.ascontiguousarray(scenes.kitti_scene(seed=frame_seed(r, 0)), np.float32) for r in range(world)]
    n_in = len(scenes.voxel_downsample_np(frames[0], VOXEL))
    cores = os.cpu_count() or 1
    warm = max(0, min(args.warmup, 1))
    for _ in range(warm):
        cpu_reference_run(frames[:1], cores)
    steps = args.steps  # (a step is ~0.25 s of CPU work per frame)
    times = [cpu_reference_run(frames, cores) for _ in range(steps)]
    t = float(np.mean(times))
    n_total = sum(len(f) for f in frames)
    value = n_total / t
    t_all = cpu_reference_all_threads(frames[0], cores)
    sample = (f"{steps} step(s) of the full workload ({world} frame(s) of {len(frames[0])} points per step, as the GPU arm at {world} rank(s)); "
              f"voxel and SOR on 1 thread (the reference's loops are serial), normals on {cores} threads (reference: rayon); "
              f"C port of the reference path (oracle/, gcc -O2 -ffp-contract=off), not the Rust build")
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(len(frames[0]), n_in, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "all_threads_value": len(frames[0]) / t_all},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-icp", action="store_true", help="skip the ICP block")
    ap.add_argument("--no-extras", action="store_true", help="headline only: skip batch8m / icp_sharded / config3 / frames_in_flight")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the kept points and normals of rank 0's last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")

    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    distributed = world > 1
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    D = dist if distributed else None

    import pointclouds_rs_b200 as pcr
    from pointclouds_rs_b200 import dist as pdist
    from pointclouds_rs_b200 import scenes

    stream = torch.cuda.current_stream()
    ctx = pcr.Context(device=local_rank, stream=stream.cuda_stream)
    ctx.set_frame_stream(True)  # the steps are consecutive frames of one sensor (config.frame_stream)

    frames = make_frames(rank)
    n_raw = len(frames[0])
    n_in = len(scenes.voxel_downsample_np(frames[0], VOXEL))  # (for sizes and the roofline only)
    F = len(frames)

    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    # the raw frames resident in HBM (device arm) and in pinned host memory (end-to-end arm)
    h_raw = [torch.from_numpy(np.ascontiguousarray(f.T)).pin_memory() for f in frames]  # (3, n_raw): x | y | z
    h_out = torch.empty((6, n_raw), dtype=torch.float32).pin_memory()                   # kept x, y, z, nx, ny, nz
    d_raw = [pcr.DeviceCloud.upload_raw(ctx, h[0].data_ptr(), h[1].data_ptr(), h[2].data_ptr(), n_raw) for h in h_raw]
    last = {}

    def pipeline(cloud):
        v = cloud.voxel_downsample(VOXEL)
        o = v.sor_normals(K_SOR, STD_MUL, K_NORMALS)
        v.free()
        return o

    def step_device(j):
        o = pipeline(d_raw[j])
        if "dev" in last:
            last["dev"].free()
        last["dev"] = o

    def step_e2e(j):
        # x | y | z rows of one pinned block that nobody writes: the copy is queued, the voxel step runs right behind it
        d = pcr.DeviceCloud.upload_block(ctx, h_raw[j].data_ptr(), n_raw, n_raw, wait=False)
        o = pipeline(d)
        d.free()
        o.download_block(h_out.data_ptr(), n_raw, with_normals=True)  # x | y | z | nx | ny | nz rows
        last["e2e_len"] = len(o)
        o.free()

    def barrier():
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also grows every scratch buffer to its final size) -------------------------------
    for i in range(max(args.warmup, 3)):
        step_device(i % F)
        step_e2e(i % F)
    torch.cuda.synchronize()
    hints0 = ctx.hint_stats()

    # ---- timed region 1: device-resident ------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    ctx.set_timing(True)
    ctx.get_timing()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    launches0 = ctx.launch_count
    barrier()
    sampler.start()
    for i in range(args.steps):
        flush.fill_(i & 0xFF)  # evict L2 ...
        stream.synchronize()   # ... and let the GPU go idle: the step's launch latency is inside the events
        starts[i].record(stream)
        step_device(i % F)
        stops[i].record(stream)
    barrier()
    launches = ctx.launch_count - launches0
    stage = ctx.get_timing()
    knn_counters = ctx.knn_counters()
    ctx.set_timing(False)
    dev_ms = sum(s.elapsed_time(e) for s, e in zip(starts, stops))

    # ---- timed region 2: end to end through the host-pointer C ABI --------------------------------
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step_e2e(i % F)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    clocks = sampler.stop()
    hints1 = ctx.hint_stats()

    if args.dump_outputs and rank == 0:  # before the parity check below reruns frame 0
        m = last["e2e_len"]
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in (("device_points", last["dev"].to_numpy()), ("device_normals", last["dev"].normals_to_numpy()),
                        ("e2e_points", h_out[0:3, :m].numpy().T), ("e2e_normals", h_out[3:6, :m].numpy().T)):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.ascontiguousarray(a, np.float32))

    dev_ms_max = pdist.max_over_ranks(D, dev_ms, "cuda")
    e2e_s_max = pdist.max_over_ranks(D, e2e_s, "cuda")
    n_total = pdist.sum_over_ranks(D, float(n_raw), "cuda")

    # parity spot check of the timed configuration: device arm and e2e arm on the same frame give the same bits
    step_device(0)
    step_e2e(0)
    torch.cuda.synchronize()
    n_kept = len(last["dev"])
    dev_pts, dev_nrm = last["dev"].to_numpy(), last["dev"].normals_to_numpy()
    m = last["e2e_len"]
    same = (m == len(dev_pts) and np.array_equal(dev_pts.T, h_out[0:3, :m].numpy()) and np.array_equal(dev_nrm.T, h_out[3:6, :m].numpy()))

    value = n_total * args.steps / (dev_ms_max * 1e-3)
    e2e_value = n_total * args.steps / e2e_s_max

    # ---- roofline of the dominant kernel -----------------------------------------------------------
    peak, peak_src = load_peaks()
    knn_n_ms, knn_n_cnt = stage["knn_normals"]
    knn_s_ms, knn_s_cnt = stage["knn"]
    # The dominant kernel of the fused pipeline is the level-0 KNN of the SOR pass: it searches
    # K = max(k_sor, k_normals) + 1 neighbours once, writes the SOR mean distance and keeps the neighbour
    # lists the normals are later computed from.  Algorithmic bytes per query (DESIGN.md section 6): read the
    # cell-sorted float4 (16), write the mean distance (4), the K list entries (4 K) and the list length (1).
    K_LIST = max(K_SOR, K_NORMALS) + 1
    # The kernel counts the queries it finishes or hands on itself (the dense / sparse / thin classes run in other launches,
    # concurrently): the bytes are those of ITS queries.
    q_per_launch = (knn_counters["queries"] / max(knn_s_cnt, 1)) if knn_counters["queries"] else n_in
    bytes_knn = q_per_launch * (16 + 4 + 4 * K_LIST + 1)
    dur_knn = knn_s_ms / max(knn_s_cnt, 1) * 1e-3
    achieved = bytes_knn / dur_knn / 1e9 if dur_knn > 0 else 0.0
    props = torch.cuda.get_device_properties(local_rank)
    prof = {}
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            prof = json.load(f)
    except Exception:
        pass
    sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
    issue_slots = props.multi_processor_count * 4 * sm_hz * dur_knn  # one warp instruction per SM sub-partition per cycle
    q_cnt, cand_cnt = knn_counters["queries"], knn_counters["candidates"]
    thread_instr = prof.get("dominant_kernel_thread_instructions_per_launch")
    warp_instr = prof.get("dominant_kernel_warp_instructions_per_launch")
    cand_per_launch = cand_cnt / max(knn_s_cnt, 1)
    fp32 = {
        "candidates_per_query": cand_cnt / q_cnt if q_cnt else None,
        "candidate_evaluations_per_launch": cand_per_launch,
        "counted": "by the kernel itself (distance evaluations of both passes: threshold histogram + collection), live",
        "fp32_instr_per_candidate": 9,
        "fp32_lane_instr_per_s": cand_per_launch * 9 / dur_knn if dur_knn > 0 else None,
        "fp32_peak_lane_instr_per_s": props.multi_processor_count * 128 * sm_hz,
        "frac_of_fp32_peak": (cand_per_launch * 9 / dur_knn) / (props.multi_processor_count * 128 * sm_hz) if dur_knn > 0 else None,
        "thread_instr_per_candidate": (thread_instr / cand_per_launch) if (thread_instr and cand_per_launch) else None,
        "frac_of_issue_peak": (warp_instr / issue_slots) if (warp_instr and issue_slots) else None,
        "instruction_counts_from": prof.get("source"),
    }
    roofline = {
        "bound": "hbm",
        "kernel": f"knn_tile_kernel<3> (grid KNN K={K_LIST}: SOR mean distance + neighbour lists kept for the normals; level 0 as cell tiles: 32 "
                  "neighbouring queries per warp, their cubes' cell runs staged in shared memory by cp.async.bulk, threshold histogram + "
                  "register sorting network on 23-bit keys)",
        "queries_per_launch": q_per_launch,
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
        "traffic": prof.get("dominant_kernel_dram_bytes_per_launch"),
        "algorithmic_bytes_per_launch": bytes_knn, "avg_launch_ms": dur_knn * 1e3,
        "note": "a 119 K-point frame is L2-resident: the kernel is bound by instruction issue and per-warp latency, not by HBM (DESIGN.md); "
                "avg_launch_ms is the event time on the launching stream, during which the dense- and sparse-class launches share the GPU "
                "(alone, under ncu, the kernel takes 0.089-0.092 ms: profiles/)",
        "fp32": fp32,
        # (the library's catch-all tag "other" holds only the voxel step in this pipeline)
        "stage_ms_per_step": {("voxel" if k == "other" else k): v[0] / args.steps for k, v in stage.items() if v[1]},
        "normals_from_lists_kernel": {"avg_launch_ms": knn_n_ms / max(knn_n_cnt, 1), "algorithmic_bytes_per_launch": n_kept * (16 + 4 * K_LIST + 1 + 12)},
        "device": {"name": torch.cuda.get_device_name(local_rank), "sm_count": props.multi_processor_count, "l2_bytes": props.L2_cache_size},
    }
    hints = {k: hints1[k] - hints0[k] for k in hints1}
    hints["frames"] = 2 * args.steps

    # ---- secondary blocks (every N) -------------------------------------------------------------------
    extra = {}
    if not args.no_extras:
        for name, fn in (("batch8m", lambda: batch8m_measurement(pcr, pdist, D, local_rank, rank, world)),
                         ("icp_sharded", (lambda: None) if args.no_icp else (lambda: icp_measurement(pcr, pdist, D, local_rank, rank, world))),
                         ("config3", lambda: config3_measurement(pcr, pdist, D, local_rank, rank, world))):
            try:
                r = fn()
                if r is not None:
                    extra[name] = r
            except Exception as ex:  # the headline must not die on a secondary measurement
                extra[name] = {"error": f"{type(ex).__name__}: {ex}"}
                if distributed:  # (a rank that failed alone would leave the others in a collective)
                    raise
        if world == 1:
            try:
                extra["frames_in_flight"] = frames_in_flight_measurement(pcr, local_rank, h_raw[0], n_raw, h_out, last["e2e_len"])
            except Exception as ex:
                extra["frames_in_flight"] = {"error": str(ex)}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        times = [cpu_reference_run(frames[:1], cores) for _ in range(3)]
        t_all = cpu_reference_all_threads(frames[0], cores)
        cpu_baseline = {
            "value": n_raw / float(np.mean(times)), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": (f"3 steps of one frame ({n_raw} points): voxel and SOR on 1 thread (the reference's loops are serial), "
                       f"normals on {cores} threads (reference: rayon); C port of the reference (oracle/, gcc -O2 -ffp-contract=off), not the Rust build"),
            "all_threads_value": n_raw / t_all,
        }

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(n_raw, n_in, world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 3 * 4 * n_raw, "d2h_bytes_per_step": 6 * 4 * n_kept,
                    "ms_per_step": e2e_s_max / args.steps * 1e3,
                    "timer": "wall clock around pcr_cloud_upload_block_nowait -> voxel -> sor_normals -> pcr_cloud_download_block, pinned host buffers"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "kept_points": n_kept,
            "device_and_e2e_results_identical": bool(same),
            "frame_stream_hints": hints,
        }
        line.update(extra)
        print(json.dumps(line))
    if distributed:
        dist.barrier()
        dist.destroy_process_group()
    return 0


# ---------------------------------------------------------------------------------------------------
def _sync_all(torch, D):
    torch.cuda.synchronize()
    if D is not None:
        D.barrier()
        torch.cuda.synchronize()


def batch8m_measurement(pcr, pdist, D, device, rank, world, n_frames=100, reps=5):
    """BASELINE configs[4]: 100 frames x 80 000 points, SOR k=10 + normals k=20, frames dealt round-robin over the ranks
    (strong scaling), one pcr_sor_normals_batch call per rank."""
    import torch

    from pointclouds_rs_b200 import scenes

    mine = pdist.deal_frames(n_frames, rank, world)
    fr = [scenes.kitti_scene(seed=f, counts=scenes.KITTI_COUNTS["frame80k"]) for f in mine]
    off = np.cumsum([0] + [len(f) for f in fr]).astype(np.uint64)
    n = int(off[-1])
    pts = np.vstack(fr) if fr else np.zeros((0, 3), np.float32)
    ctx = pcr.Context(device=device)
    vp = np.zeros(3, np.float32)
    # pinned host buffers (SoA in, results out) and their device twins
    h_in = torch.from_numpy(np.ascontiguousarray(pts.T)).pin_memory() if n else torch.zeros((3, 1)).pin_memory()
    h_keep = torch.empty(max(n, 1), dtype=torch.uint8).pin_memory()
    h_nrm = torch.empty((3, max(n, 1)), dtype=torch.float32).pin_memory()
    kept = np.zeros(max(len(mine), 1), np.uint64)
    d_in = h_in.cuda()
    d_keep = torch.empty(max(n, 1), dtype=torch.uint8, device="cuda")
    d_nrm = torch.empty((3, max(n, 1)), dtype=torch.float32, device="cuda")
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")

    def host_call():
        if n:
            pcr.sor_normals_batch_raw(ctx, h_in[0].data_ptr(), h_in[1].data_ptr(), h_in[2].data_ptr(), n, off, K_SOR, STD_MUL, K_NORMALS, vp,
                                      h_keep.data_ptr(), h_nrm[0].data_ptr(), h_nrm[1].data_ptr(), h_nrm[2].data_ptr(), kept=kept)

    def dev_call():
        if n:
            pcr.sor_normals_batch_raw(ctx, d_in[0].data_ptr(), d_in[1].data_ptr(), d_in[2].data_ptr(), n, off, K_SOR, STD_MUL, K_NORMALS, vp,
                                      d_keep.data_ptr(), d_nrm[0].data_ptr(), d_nrm[1].data_ptr(), d_nrm[2].data_ptr(), device=True)
            ctx.synchronize()

    for _ in range(2):
        host_call()
        dev_call()
    _sync_all(torch, D)
    t_host, t_dev = [], []
    for _ in range(reps):
        flush.fill_(1)
        _sync_all(torch, D)
        t0 = time.perf_counter()
        host_call()
        t_host.append(time.perf_counter() - t0)
    for _ in range(reps):
        flush.fill_(2)
        _sync_all(torch, D)
        t0 = time.perf_counter()
        dev_call()
        t_dev.append(time.perf_counter() - t0)
    spread = {"host_api_ms": [round(t * 1e3, 3) for t in t_host], "device_ms": [round(t * 1e3, 3) for t in t_dev]}
    t_host, t_dev = float(np.median(t_host)) * reps, float(np.median(t_dev)) * reps  # (SURVEY 8d: the median of the repetitions)
    # both arms must agree (same kernels): the host arm's mask and normals against the device arm's
    same = True
    if n:
        same = bool(np.array_equal(h_keep[:n].numpy(), d_keep[:n].cpu().numpy()) and np.array_equal(h_nrm[:, :n].numpy(), d_nrm[:, :n].cpu().numpy()))
    t_host = pdist.max_over_ranks(D, t_host / reps, "cuda")
    t_dev = pdist.max_over_ranks(D, t_dev / reps, "cuda")
    n_all = pdist.sum_over_ranks(D, float(n), "cuda")
    same_all = pdist.sum_over_ranks(D, 0.0 if same else 1.0, "cuda") == 0.0
    ctx.close()
    return {
        "workload": "BASELINE configs[4]: 100 KITTI-shaped frames x 80 000 points, SOR k=10 + normals k=20, frames dealt round-robin, "
                    "one pcr_sor_normals_batch call per rank",
        "scaling": "strong", "frames": n_frames, "points": int(n_all), "frames_on_rank0": len(mine),
        "device": {"value": n_all / t_dev, "unit": UNIT, "ms": t_dev * 1e3, "timer": "wall clock around pcr_sor_normals_batch_dev + sync, inputs resident in HBM, max over ranks"},
        "host_api": {"value": n_all / t_host, "unit": UNIT, "ms": t_host * 1e3,
                     "h2d_bytes": 12 * int(n_all), "d2h_bytes": 13 * int(n_all),
                     "timer": "wall clock around pcr_sor_normals_batch (pinned host buffers, copies inside), max over ranks"},
        "host_and_device_results_identical": bool(same_all),
        "repetitions_rank0": spread, "statistic": "median of %d calls after 2 warm-up calls" % reps,
    }


def icp_measurement(pcr, pdist, D, device, rank, world):
    """BASELINE configs[3]: point-to-plane ICP, two synthetic scans of 1 M points, 30 iterations, the SOURCE sharded over
    the ranks; the library all-reduces the 30-double normal equations over NCCL every iteration."""
    import torch

    from pointclouds_rs_b200 import scenes

    tgt_np = scenes.aerial_scene(42, 0.415)
    R = scenes.rot_z(0.05)
    src_np = np.ascontiguousarray((tgt_np @ R.T + np.array([0.3, -0.2, 0.1], np.float32)).astype(np.float32))
    solo = pcr.Context(device=device)
    tgt = pcr.estimate_normals(pcr.PointCloud.from_numpy(tgt_np), 20, solo)
    full = pcr.PointCloud.from_numpy(src_np)
    ctx = pcr.Context(device=device)
    if world > 1:
        ctx.comm_init(pdist.share_unique_id(D, pcr.Context.unique_id, device="cuda"), rank, world)
    comm_kind = ctx.comm_kind
    # every world-th point: the generator emits terrain, then buildings, then trees, so contiguous ranges give the ranks
    # very different work (measured at 2 GPUs: 0.11 vs 0.23 ms of kernels per iteration, the faster rank waiting in the
    # all-reduce); which points a rank holds is the caller's choice, the result does not depend on it
    shard_np = np.ascontiguousarray(src_np[rank::world])
    b, e = 0, len(shard_np)
    shard = pcr.PointCloud.from_numpy(shard_np)
    for _ in range(2):
        pcr.icp_point_to_plane(shard, tgt, 30, 0.0, ctx=ctx)  # warm-up
    ctx.set_timing(True)
    ctx.get_timing()
    walls = []
    ICP_REPS = 5
    for _ in range(ICP_REPS):  # (SURVEY 8d: the median of the repetitions)
        _sync_all(torch, D)
        t0 = time.perf_counter()
        res = pcr.icp_point_to_plane(shard, tgt, 30, 0.0, ctx=ctx)
        walls.append(time.perf_counter() - t0)
    stage = ctx.get_timing()
    ctx.set_timing(False)
    wall_local = wall = float(np.median(walls))
    wall = pdist.max_over_ranks(D, wall, "cuda")
    step_ms, step_cnt = stage["icp_step"]      # (sums over the timed calls; used per iteration below)
    solve_ms, solve_cnt = stage["icp_solve"]
    one = pcr.icp_point_to_plane(full, tgt, 30, 0.0, ctx=solo)  # the unsharded run on this GPU
    v = torch.tensor([x for row in res.rotation for x in row] + list(res.translation) + [res.rmse, res.fitness, float(res.num_iterations)],
                     dtype=torch.float64, device="cuda")
    identical = True
    if D is not None:
        g = [torch.zeros_like(v) for _ in range(world)]
        D.all_gather(g, v)
        identical = all(torch.equal(x, g[0]) for x in g)
    close = bool(np.allclose(res.rotation, one.rotation, atol=1e-5) and np.allclose(res.translation, one.translation, atol=1e-5)
                 and abs(res.rmse - one.rmse) < 1e-5 and res.num_iterations == one.num_iterations)
    out = {
        "workload": "BASELINE configs[3]: point-to-plane ICP, two synthetic scans (aerial generator, scale 0.415), 30 iterations, tolerance 0; "
                    "source sharded over the ranks (every world-th point), target + grid + normals replicated",
        "scaling": "strong", "points": len(src_np), "source_points_on_rank0": e - b, "iterations": res.num_iterations,
        "ms_per_iter_e2e": wall * 1e3 / max(res.num_iterations, 1),
        "ms_per_iter_step_kernels_rank0": step_ms / max(step_cnt, 1),
        # reduce kernel + [all-reduce] + solve kernel: event time on the library's stream, so at N > 1 it contains the collective
        # AND the wait for the slowest rank to reach it
        "ms_per_iter_reduce_allreduce_solve_rank0": solve_ms / max(solve_cnt, 1),
        "ms_per_iter_loop_rank0": step_ms / max(step_cnt, 1) + solve_ms / max(solve_cnt, 1),  # the iteration itself: what sharding can shrink
        # what is not the iteration loop: upload of the shard and the (replicated) target + normals, target index build,
        # source binning, result download -- paid once per call whatever the number of ranks
        "ms_setup_and_host_rank0": wall_local * 1e3 - (step_ms + solve_ms) / ICP_REPS,
        "ms_per_call_rank0": [round(w * 1e3, 3) for w in walls], "statistic": "median of %d calls after 2 warm-up calls" % ICP_REPS,
        "collective": {"none": "none (one rank)",
                       "nccl": "ncclAllReduce of 30 f64 on the library's stream, every iteration",
                       "peer": "one-shot all-reduce of 30 f64 over NVLink peer memory (CUDA IPC blocks), fused into the reduction kernel, "
                               "every iteration; summed in rank order"}[comm_kind],
        "identical_on_all_ranks": bool(identical), "equals_unsharded": close,
        "rmse": res.rmse, "translation": res.translation,
    }
    ctx.close()
    solo.close()
    return out


def config3_measurement(pcr, pdist, D, device, rank, world, reps=3):
    """BASELINE configs[2]: aerial 241 K points -- normals k = 20, radius outlier removal (r = 2.0, 5 neighbours) and the
    radius-search CSR at r = 2.0, with the QUERIES sharded over the ranks (SURVEY 8e rows 1-2)."""
    import torch

    from pointclouds_rs_b200 import scenes

    pts = scenes.aerial_scene(42, 0.1)
    cloud = pcr.PointCloud.from_numpy(pts)
    solo = pcr.Context(device=device)
    ctx = pcr.Context(device=device)
    if world > 1:
        ctx.comm_init(pdist.share_unique_id(D, pcr.Context.unique_id, device="cuda"), rank, world)
        ctx.set_query_sharding(True)
    ref_n = pcr.normals_array(cloud, 20, ctx=solo)
    ref_keep, ref_kept, ref_mean, ref_stats = pcr.sor_mask(cloud, 10, 1.0, ctx=solo, want_mean=True)
    ref_ror, _ = pcr.ror_mask(cloud, 2.0, 5, ctx=solo)

    def timed(fn):
        fn()
        t = 0.0
        for _ in range(reps):
            _sync_all(torch, D)
            t0 = time.perf_counter()
            r = fn()
            t += time.perf_counter() - t0
        return pdist.max_over_ranks(D, t / reps, "cuda"), r

    t_n, nrm = timed(lambda: pcr.normals_array(cloud, 20, ctx=ctx))
    t_s, sor = timed(lambda: pcr.sor_mask(cloud, 10, 1.0, ctx=ctx, want_mean=True))
    t_r, ror = timed(lambda: pcr.ror_mask(cloud, 2.0, 5, ctx=ctx))
    # radius-search CSR: the caller shards the queries (contiguous range), the index is replicated
    b, e = pdist.split_range(len(pts), rank, world)
    tree = pcr.KdTree(cloud, 20, ctx=solo)
    t_c, csr = timed(lambda: tree.radius_search(pts[b:e], 2.0))
    total = pdist.sum_over_ranks(D, float(len(csr[1])), "cuda")
    ident = bool(np.array_equal(nrm.view(np.uint32), ref_n.view(np.uint32)) and np.array_equal(sor[0], ref_keep) and sor[1] == ref_kept
                 and np.array_equal(sor[2].view(np.uint32), ref_mean.view(np.uint32)) and np.array_equal(sor[3].view(np.uint32), ref_stats.view(np.uint32))
                 and np.array_equal(ror[0], ref_ror))
    ident = pdist.sum_over_ranks(D, 0.0 if ident else 1.0, "cuda") == 0.0
    n = len(pts)
    out = {
        "workload": "BASELINE configs[2]: aerial synthetic 241K pts: normals k=20, SOR k=10, radius outlier removal r=2.0 (5 neighbours), radius-search CSR r=2.0",
        "scaling": "strong", "points": n,
        "sharding": "queries: every rank holds the cloud and the index, searches its cell range of the sorted order, results merged with an integer "
                    "sum over NCCL (pcr_ctx_set_query_sharding); the CSR queries are split by the caller" if world > 1 else "one rank",
        "normals_k20": {"ms": t_n * 1e3, "value": n / t_n, "unit": UNIT},
        "sor_k10": {"ms": t_s * 1e3, "value": n / t_s, "unit": UNIT},
        "radius_outlier_r2": {"ms": t_r * 1e3, "value": n / t_r, "unit": UNIT},
        "radius_search_csr_r2": {"ms": t_c * 1e3, "value": n / t_c, "unit": UNIT, "neighbours_total": int(total)},
        "timer": "wall clock around the host-pointer C-ABI call (pageable numpy buffers, copies and the NCCL merge inside), max over ranks",
        "bit_identical_to_one_gpu": bool(ident),
    }
    del tree
    ctx.close()
    solo.close()
    return out


def frames_in_flight_measurement(pcr, device, h_raw, n_raw, h_ref, m_ref, flights=(2, 4), steps=60):
    """Secondary figure (NOT the headline): the same end-to-end step with several frames in flight.  One frame is
    latency-bound (short kernels, host round trips for counts), and contexts are independent, so T host threads --
    each with its own context, stream and pinned output block -- overlap their frames on the one GPU."""
    import torch

    def worker(ctx, out, n_steps, go, lens):
        go.wait()
        for _ in range(n_steps):
            d = pcr.DeviceCloud.upload_block(ctx, h_raw.data_ptr(), n_raw, n_raw, wait=False)
            v = d.voxel_downsample(VOXEL)
            o = v.sor_normals(K_SOR, STD_MUL, K_NORMALS)
            d.free()
            v.free()
            o.download_block(out.data_ptr(), n_raw, with_normals=True)
            lens.append(len(o))
            o.free()

    res = {"note": "T host threads x (context, stream), frame 0 and the calls of e2e; wall clock; results compared with the e2e arm"}
    for T in flights:
        ctxs = [pcr.Context(device=device) for _ in range(T)]
        outs = [torch.empty((6, n_raw), dtype=torch.float32).pin_memory() for _ in range(T)]
        for c in ctxs:
            c.set_frame_stream(True)
        dt, lens = 0.0, []
        for n_steps in (5, steps):  # warm-up, then timed
            go, lens = threading.Event(), []
            th = [threading.Thread(target=worker, args=(ctxs[t], outs[t], n_steps, go, lens)) for t in range(T)]
            for t in th:
                t.start()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            go.set()
            for t in th:
                t.join()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        same = all(m == m_ref for m in lens) and all(np.array_equal(o[:, :m_ref].numpy(), h_ref[:, :m_ref].numpy()) for o in outs)
        res[str(T)] = {"value": n_raw * steps * T / dt, "unit": UNIT, "ms_per_frame": dt / (steps * T) * 1e3, "identical_to_e2e": bool(same)}
        for c in ctxs:
            c.close()
    return res


if __name__ == "__main__":
    sys.exit(main())
