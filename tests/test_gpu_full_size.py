"""Parity at the FULL sizes BASELINE.json names (configs 3, 4, 5), against the oracle where it finishes
in seconds and through size-independent properties otherwise."""
import os

import numpy as np
import pytest

from pointclouds_rs_b200 import scenes

pytestmark = pytest.mark.gpu
T = max(1, min(32, os.cpu_count() or 1))


def _ang(a, b):
    a, b = a.astype(np.float64), b.astype(np.float64)
    return np.arctan2(np.linalg.norm(np.cross(a, b), axis=1), np.abs(np.sum(a * b, axis=1)))


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOUNDS_FILE = os.path.join(ROOT, "tests", "golden", "degenerate_normals.json")


def _bound(name, n):
    """Upper bound on the exactly-degenerate normals of config `name`: the count observed on a B200 and recorded in
    tests/golden/degenerate_normals.json (tracked), not a percentage."""
    import json

    with open(BOUNDS_FILE) as f:
        return int(json.load(f)["observed_on_b200"][name])


def _check_normals(pts, nrm, o, k, oracle, name):
    """<= 1e-4 rad (north_star) everywhere except on EXACTLY degenerate neighbourhoods.

    The aerial scene has wall points that share one coordinate exactly (x = cx + w/2 ...): their
    covariance has an exactly zero row, the Cardano eigenvalue is pure rounding noise (~1e-17), and
    whether `len2 < 1e-30` (estimate.rs:210) holds depends on the last ulp of f64 acos/cos -- which
    differs between CUDA and glibc (and Rust's libm).  Either branch is a legitimate execution of the
    reference code; such points are counted, must be rare, and must really be degenerate."""
    ang = _ang(nrm, o)
    bad = np.nonzero(ang > 1e-4)[0]
    print(f"{name}: {len(bad)} of {len(pts)} normals over 1e-4 rad")  # (pytest -s: the count to record in BOUNDS_FILE)
    assert len(bad) <= _bound(name, len(pts)), f"{len(bad)} normals over tolerance (recorded bound {_bound(name, len(pts))})"
    if len(bad):
        idx, _, _ = oracle.Tree(pts).knn_batch(pts[bad], k, threads=T)
        nb = pts[idx.astype(np.int64)]  # (n_bad, k, 3)
        degenerate = (nb.max(axis=1) == nb.min(axis=1)).any(axis=1)  # all neighbours share a coordinate exactly
        assert degenerate.all(), f"{int((~degenerate).sum())} non-degenerate normals differ, max {ang[bad][~degenerate].max()} rad"
    return len(bad)


def test_config3_aerial_241k_normals_and_radius(pcr, oracle):
    pts = scenes.aerial_scene(42, 0.1)
    assert len(pts) == 241_000
    cloud = pcr.PointCloud.from_numpy(pts)
    nrm = pcr.normals_array(cloud, 20)
    o = oracle.normals(pts, 20, threads=T)
    n_deg = _check_normals(pts, nrm, o, 20, oracle, "config3_aerial_241k_k20")
    print(f"config 3: {n_deg} exactly-degenerate wall normals took the other branch")
    assert np.allclose(np.linalg.norm(nrm, axis=1), 1.0, atol=1e-5)
    keep, kept = pcr.ror_mask(cloud, 2.0, 5)
    assert np.array_equal(keep, oracle.ror(pts, 2.0, 5, threads=T))
    tree = pcr.KdTree(cloud, 20)
    rng = np.random.default_rng(0)
    q = pts[rng.integers(0, len(pts), 3000)]
    off, idx = tree.radius_search(q, 2.0)
    otree = oracle.Tree(pts)
    assert np.array_equal(np.diff(off).astype(np.uint32), otree.radius_count_batch(q, 2.0, threads=T))
    for j in range(0, 3000, 97):
        assert np.array_equal(idx[off[j]:off[j + 1]], otree.radius_search(q[j], 2.0))
    ki, kd, kc = tree.knn(q, 20)
    oi, od, oc = otree.knn_batch(q, 20, threads=T)
    assert np.array_equal(ki, oi) and np.array_equal(kd.view(np.uint32), od.view(np.uint32))


def test_config4_icp_point_to_plane_1m_30_iterations(pcr, oracle):
    tgt = scenes.aerial_scene(42, 0.415)
    assert len(tgt) == 1_000_150
    src = oracle.apply_transform(tgt, scenes.rot_z(0.05), [0.3, -0.2, 0.1])
    tn = oracle.normals(tgt, 20, threads=T)
    t = pcr.PointCloud.from_numpy(tgt)
    gn = pcr.normals_array(t, 20)
    _check_normals(tgt, gn, tn, 20, oracle, "config4_aerial_1m_k20")
    t.normals = tn  # same normals on both sides: isolates the ICP loop
    res = pcr.icp_point_to_plane(pcr.PointCloud.from_numpy(src), t, max_iterations=30, tolerance=0.0)
    o = oracle.icp_point_to_plane(src, tgt, tn, 30, 0.0, threads=T)
    assert res.num_iterations == 30 == o.num_iterations and not res.converged
    # north_star tolerance: transforms within 1e-4 (rotation entries / translation in metres)
    assert np.abs(np.array(res.rotation) - o.rotation).max() < 1e-4
    assert np.abs(np.array(res.translation) - o.translation).max() < 1e-4
    assert abs(res.rmse - o.rmse) < 1e-4 * max(1.0, o.rmse) and abs(res.fitness - o.fitness) < 1e-6


def test_config5_batch_100_frames_8m_points(pcr, oracle):
    counts = scenes.KITTI_COUNTS["frame80k"]
    frames = [scenes.kitti_scene(seed, counts) for seed in range(100)]
    off = np.arange(101, dtype=np.uint64) * 80_000
    pts = np.vstack(frames)
    assert len(pts) == 8_000_000
    keep, nrm, kept = pcr.sor_normals_batch(pts, off, 10, 1.0, 20)
    # properties over all 8 M points
    assert kept.sum() == keep.sum() and (kept > 0.9 * 80_000).all() and (kept < 80_000).all()
    ln = np.linalg.norm(nrm, axis=1)
    assert np.allclose(ln[keep == 1], 1.0, atol=1e-5) and (ln[keep == 0] == 0).all()
    # exact comparison on a sample of frames
    for f in (0, 37, 99):
        sl = slice(int(off[f]), int(off[f + 1]))
        o_keep, _, _ = oracle.sor(frames[f], 10, 1.0, threads=T)
        assert np.array_equal(keep[sl], o_keep), f"frame {f}"
        sel = np.nonzero(o_keep)[0]
        assert _ang(nrm[sl][sel], oracle.normals(frames[f][sel], 20, threads=T)).max() < 1e-4
    # idempotence of the mask under frame order: a frame alone gives the same answer as in the batch
    k1, n1, c1 = pcr.sor_normals_batch(frames[5], np.array([0, 80_000], np.uint64), 10, 1.0, 20)
    sl = slice(int(off[5]), int(off[6]))
    assert np.array_equal(k1, keep[sl]) and np.array_equal(n1, nrm[sl])


def test_cpp_host_layer_runs(tmp_path):
    """include/pcr_b200.hpp (the C++ mirror of the Rust API) end to end on the device."""
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = tmp_path / "cpp_host_example"
    lib = os.path.join(root, "pointclouds_rs_b200", "lib")
    subprocess.check_call(["g++", "-std=c++17", "-I" + os.path.join(root, "include"), os.path.join(root, "examples", "cpp_host_example.cpp"),
                           "-L" + lib, "-lpcr_b200", "-Wl,-rpath," + lib, "-o", str(exe)])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "kept 5000 of 5001" in out.stdout, out.stdout
