"""ICP started from a guess (the _init calls, DESIGN 3.4): its cost, multi-start and coarse-to-fine.

Workloads (scenes.kitti_sequence, 100 frames of 122 K points, voxel 0.2 on the device):
  identity_cost   point-to-plane ICP over the 99 consecutive pairs (30 iterations, tolerance 0): the batch _init call with
                  identity guesses against the plain batch call, on the same resident frames.  Outputs must be identical
                  bit for bit.
  multi_start     --ms-pairs consecutive pairs x --ms-guesses yaw hypotheses (rot_z(2 pi k / M)), point-to-plane, radius
                  1 m, 30 iterations: one icp_point_to_plane_batch(init=...) call against the workaround without it
                  (every source frame copied M times into a new buffer, the copies moved by apply_transform_batch, the
                  batch run from the identity, every result composed with its guess on the host).  Both arms start from
                  the same host arrays.  Reported: whether both keep the same hypothesis (best fitness) for every pair,
                  and the largest transform difference between the arms (the workaround rounds in another order).
  coarse_to_fine  the scenario of tests/test_icp_init.py over 100 frames of 20 K points (seed 11): a faster drive (1.5 m
                  and 0.08 rad per frame, three times the 0.5 m fine radius), point-to-point over the 99 pairs:
                  single-scale (radius 0.5, 30 iterations, tolerance 1e-6) against voxel 1.0, radius 5, 50 iterations,
                  then the full frames from that result.  Both arms start from the resident upload.  Reported: time,
                  and the relative-pose error of every pair against the generator (median, max, and the pairs within
                  5 cm and 5 mrad).  The generator turns about frame 0's origin, so later frames are far from their
                  sensor and the same yaw moves their points further: the pairs are not equally hard.
Every timed call is synchronous (host clock around the call and a synchronise).  The arms alternate in one process after
warm-up; the median and min / max over --reps repetitions are reported.  One JSON line; --out FILE also writes it there.
"""
import argparse
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
from pointclouds_rs_b200 import scenes  # noqa: E402

EYE12 = np.array([1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0], np.float32)


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
    """arms: {name: fn() -> outputs}.  Alternating repetitions after warm-up -> ({name: times ms}, {name: last outputs})."""
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


def row(name, ts, extra):
    r = {"row": name}
    r.update({f"{k}_ms": stats(v) for k, v in ts.items()})
    r.update(extra)
    print(json.dumps(r), file=sys.stderr)
    return r


def bits(res):
    return [(np.float32(r.rotation).tobytes(), np.float32(r.translation).tobytes(), np.float32(r.rmse).tobytes(),
             np.float32(r.fitness).tobytes(), r.num_iterations, r.converged) for r in res]


def t12(r):
    return np.concatenate([np.asarray(r.rotation, np.float32).reshape(9), np.asarray(r.translation, np.float32)])


def sequence(n, seed=7, counts=scenes.KITTI_COUNTS["frame122k"], **kw):
    seq = scenes.kitti_sequence(n, seed=seed, counts=counts, **kw)
    off = np.zeros(n + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in seq])
    return np.ascontiguousarray(np.vstack(seq), np.float32), off


def identity_cost(ctx, a):
    pts, off = sequence(a.frames)
    fr = pcr.DeviceFrames.from_numpy(pts, off, ctx=ctx).voxel_downsample(0.2).estimate_normals(15)
    pairs = np.c_[np.arange(1, a.frames), np.arange(a.frames - 1)]
    eye = np.tile(EYE12, (len(pairs), 1))
    kw = dict(max_iterations=30, tolerance=0.0)
    ts, o = timed({"init": lambda: fr.icp_point_to_plane(pairs, init=eye, **kw), "plain": lambda: fr.icp_point_to_plane(pairs, **kw)},
                  a.reps, a.warmup)
    return row("identity_cost", ts, {"pairs": len(pairs), "voxels_0.2": len(fr), "iterations": 30,
                                     "outputs_identical": bits(o["init"]) == bits(o["plain"])})


def multi_start(ctx, a):
    pts, off = sequence(a.ms_pairs + 1)
    fr = pcr.DeviceFrames.from_numpy(pts, off, ctx=ctx).voxel_downsample(0.2).estimate_normals(15)
    (vp, voff), vn = fr.to_numpy(), fr.normals_to_numpy()
    P, M = a.ms_pairs, a.ms_guesses
    pairs = np.repeat(np.c_[np.arange(1, P + 1), np.arange(P)], M, axis=0)  # pair p, guess k at row p * M + k
    guesses = np.stack([np.concatenate([scenes.rot_z(2 * np.pi * k / M).reshape(9), np.zeros(3, np.float32)]) for k in range(M)])
    inits = np.tile(guesses, (P, 1))
    kw = dict(max_iterations=30, tolerance=0.0, max_correspondence_distance=1.0)

    def with_init():
        return pcr.icp_point_to_plane_batch(vp, voff, pairs, vn, init=inits, ctx=ctx, **kw)

    def workaround():
        n_f = len(voff) - 1
        frames = [vp[int(voff[f]):int(voff[f + 1])] for f in range(n_f)]
        copies = [frames[s] for s, _ in pairs]
        all_f = frames + copies
        b_off = np.zeros(len(all_f) + 1, np.uint64)
        b_off[1:] = np.cumsum([len(f) for f in all_f])
        buf = np.vstack(all_f)
        moved = pcr.apply_transform_batch(buf, b_off, np.vstack([np.tile(EYE12, (n_f, 1)), inits]), ctx=ctx)
        nrm = np.vstack([vn, np.zeros((len(buf) - len(vn), 3), np.float32)])
        w_pairs = np.c_[n_f + np.arange(len(pairs)), pairs[:, 1]]
        res = pcr.icp_point_to_plane_batch(moved, b_off, w_pairs, nrm, ctx=ctx, **kw)
        out = []
        for j, r in enumerate(res):
            R, t = pcr.compose((inits[j, :9].reshape(3, 3), inits[j, 9:]), (r.rotation, r.translation))
            out.append((np.concatenate([R.reshape(9), t]), r.fitness))
        return out

    ts, o = timed({"init": with_init, "workaround": workaround}, a.reps, a.warmup)
    fit_i = np.array([r.fitness for r in o["init"]]).reshape(P, M)
    fit_w = np.array([f for _, f in o["workaround"]]).reshape(P, M)
    diff = max(float(np.abs(t12(r) - w).max()) for r, (w, _) in zip(o["init"], o["workaround"]))
    return row("multi_start", ts, {"pairs": P, "guesses": M, "registrations": P * M, "source_points": int(sum(voff[s + 1] - voff[s] for s, _ in pairs)),
                                   "same_hypotheses": bool(np.array_equal(fit_i.argmax(1), fit_w.argmax(1))),
                                   "best_hypothesis_counts": np.bincount(fit_i.argmax(1), minlength=M).tolist(),
                                   "max_transform_diff": diff})


def coarse_to_fine(ctx, a):
    step, yaw = np.array([1.5, 0.3, 0.0]), 0.08
    pts, off = sequence(a.frames, seed=11, counts=(17_600, 880, 145, 495), step=tuple(step), yaw=yaw)
    up = pcr.DeviceFrames.from_numpy(pts, off, ctx=ctx)
    pairs = np.c_[np.arange(1, a.frames), np.arange(a.frames - 1)]
    fine = dict(max_iterations=30, tolerance=1e-6, max_correspondence_distance=0.5)
    coarse = dict(max_iterations=50, tolerance=1e-6, max_correspondence_distance=5.0)

    def single():
        return up.icp_point_to_point(pairs, **fine)

    def c2f():
        c = up.voxel_downsample(1.0).icp_point_to_point(pairs, **coarse)
        return up.icp_point_to_point(pairs, init=c, **fine)

    ts, o = timed({"coarse_to_fine": c2f, "single_scale": single}, a.reps, a.warmup)
    Rt = scenes.rot_z(yaw).astype(np.float64)
    err = {}
    for k, res in o.items():
        te = [float(np.linalg.norm(np.asarray(r.translation) - scenes.rot_z(-yaw * i).astype(np.float64) @ step)) for i, r in enumerate(res)]
        re = [float(np.arccos(np.clip((np.trace(np.asarray(r.rotation, np.float64) @ Rt.T) - 1) / 2, -1, 1))) for r in res]
        err[k] = {"trans_err_m": {"median": round(float(np.median(te)), 5), "max": round(max(te), 5)},
                  "rot_err_rad": {"median": round(float(np.median(re)), 6), "max": round(max(re), 6)},
                  "pairs_within_5cm_5mrad": int(sum(t < 0.05 and r < 0.005 for t, r in zip(te, re))),
                  "first_pair_failing": next((i for i, (t, r) in enumerate(zip(te, re)) if not (t < 0.05 and r < 0.005)), None)}
    return row("coarse_to_fine", ts, {"pairs": len(pairs), "step_m": [1.5, 0.3, 0.0], "yaw_rad": yaw, "pose_error": err})


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--ms-pairs", type=int, default=20)
    ap.add_argument("--ms-guesses", type=int, default=12)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", default="identity_cost,multi_start,coarse_to_fine")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_icp_init: no CUDA device (the measurement needs a B200)")
    ctx = pcr.default_context()
    info = gpu_info()
    rows = []
    for name, fn in (("identity_cost", identity_cost), ("multi_start", multi_start), ("coarse_to_fine", coarse_to_fine)):
        if name in a.only.split(","):
            rows.append(fn(ctx, a))
            torch.cuda.empty_cache()
    s = json.dumps({"tool": "bench_icp_init", "gpu": info, "reps": a.reps, "warmup": a.warmup, "rows": rows})
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
