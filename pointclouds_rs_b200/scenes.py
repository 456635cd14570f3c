"""Synthetic scenes of the shapes BASELINE.json names (numpy PCG64, seeded).

These restate the reference's demo generators so that bench.py, the tests and smoke() all see the
same inputs.  They are inputs, not algorithms: nothing here touches the KNN path.

  kitti_scene   <- examples/python/kitti_obstacle_detection.py:22-81 (same rng call order; counts scale)
  aerial_scene  <- examples/python/aerial_lidar.py:26-137
  hemisphere    <- tests/real_world_pipeline.rs:58-80 (ChaCha12 there; PCG64 here)
  uniform_cube  <- benches/bench_filters.rs:9-15 / bench_kdtree.rs:7-13
"""
from __future__ import annotations

import numpy as np

# (ground, per-car, pedestrian, noise) point counts
KITTI_COUNTS = {
    "demo68k": (60_000, 3_000, 500, 1_500),     # the reference demo, 68 000 points
    "frame122k": (108_000, 5_400, 900, 2_300),  # BASELINE config 2, 122 000 points
    "frame80k": (70_600, 3_530, 590, 1_750),    # BASELINE config 5, 80 000 points / frame
}


def kitti_scene(seed: int = 42, counts=KITTI_COUNTS["frame122k"]) -> np.ndarray:
    n_ground, n_car, n_ped, n_noise = counts
    rng = np.random.default_rng(seed)
    parts = []
    gx = rng.uniform(-30, 30, n_ground).astype(np.float32)
    gy = rng.uniform(-20, 20, n_ground).astype(np.float32)
    gz = rng.normal(0, 0.03, n_ground).astype(np.float32)
    parts.append(np.column_stack([gx, gy, gz]))
    for cx, cy, cz in ((8.0, 3.0, 0.8), (-5.0, -8.0, 0.8)):
        car = np.column_stack([
            rng.uniform(cx - 2.0, cx + 2.0, n_car),
            rng.uniform(cy - 0.9, cy + 0.9, n_car),
            rng.uniform(cz - 0.0, cz + 1.5, n_car),
        ]).astype(np.float32)
        parts.append(car)
    px, py, pz = 3.0, -2.0, 0.9
    ped = np.column_stack([
        rng.uniform(px - 0.25, px + 0.25, n_ped),
        rng.uniform(py - 0.25, py + 0.25, n_ped),
        rng.uniform(pz - 0.0, pz + 1.8, n_ped),
    ]).astype(np.float32)
    parts.append(ped)
    noise = np.column_stack([
        rng.uniform(-35, 35, n_noise),
        rng.uniform(-25, 25, n_noise),
        rng.uniform(-3, 8, n_noise),
    ]).astype(np.float32)
    parts.append(noise)
    return np.ascontiguousarray(np.vstack(parts), dtype=np.float32)


def kitti_points(counts) -> int:
    """Points of kitti_scene(seed, counts) (two cars)."""
    n_ground, n_car, n_ped, n_noise = counts
    return int(n_ground + 2 * n_car + n_ped + n_noise)


def kitti_sequence(n_frames: int, seed: int = 42, counts=KITTI_COUNTS["frame122k"], step=(0.4, 0.05, 0.0), yaw: float = 0.01,
                   jitter: float = 0.01) -> list:
    """A LiDAR drive through one KITTI-shaped scene: frame i sees a different random subset of kitti_points(counts) points
    of a 25 % denser scene, in the sensor frame of pose i (pose i+1 = pose i moved by `step` metres and turned by `yaw`
    radians about z), with Gaussian jitter.  Consecutive frames are a small rigid motion apart (odometry input)."""
    world = kitti_scene(seed, tuple(int(c * 1.25) for c in counts))
    n = kitti_points(counts)
    rng = np.random.default_rng(seed + 1)
    out = []
    for i in range(n_frames):
        idx = np.sort(rng.permutation(len(world))[:n])
        r = rot_z(-yaw * i).astype(np.float64)
        p = (world[idx].astype(np.float64) - np.asarray(step, np.float64) * i) @ r.T
        out.append(np.ascontiguousarray(p + rng.normal(0.0, jitter, (n, 3)), dtype=np.float32))
    return out


def aerial_scene(seed: int = 42, scale: float = 0.1) -> np.ndarray:
    """scale=0.1 -> 241 000 points (config 3); scale=0.415 -> 1 000 150 points (config 4)."""
    rng = np.random.default_rng(seed)
    parts = []
    area_x, area_y = 500.0, 500.0
    n_terrain = int(2_000_000 * scale)
    tx = rng.uniform(0, area_x, n_terrain).astype(np.float32)
    ty = rng.uniform(0, area_y, n_terrain).astype(np.float32)
    tz = (2.0 * np.sin(tx * 0.02) * np.cos(ty * 0.015) + rng.normal(0, 0.05, n_terrain)).astype(np.float32)
    parts.append(np.column_stack([tx, ty, tz]))
    buildings = [(100, 120, 30, 20, 12), (250, 300, 40, 40, 18), (350, 100, 25, 25, 8),
                 (400, 400, 50, 30, 15), (150, 350, 20, 20, 10)]
    n_per_building = int(50_000 * scale)
    for cx, cy, w, d, h in buildings:
        n_roof = int(n_per_building * 0.7)
        bx = rng.uniform(cx - w / 2, cx + w / 2, n_roof).astype(np.float32)
        by = rng.uniform(cy - d / 2, cy + d / 2, n_roof).astype(np.float32)
        bz = np.full(n_roof, h, dtype=np.float32) + rng.normal(0, 0.02, n_roof).astype(np.float32)
        parts.append(np.column_stack([bx, by, bz]))
        n_wall = n_per_building - n_roof
        side = rng.integers(0, 4, n_wall)
        wx = np.empty(n_wall, dtype=np.float32)
        wy = np.empty(n_wall, dtype=np.float32)
        wz = rng.uniform(0, h, n_wall).astype(np.float32)
        for i in range(n_wall):  # scalar draws, like the reference (keeps the rng stream identical)
            if side[i] == 0:
                wx[i] = rng.uniform(cx - w / 2, cx + w / 2)
                wy[i] = cy + d / 2
            elif side[i] == 1:
                wx[i] = rng.uniform(cx - w / 2, cx + w / 2)
                wy[i] = cy - d / 2
            elif side[i] == 2:
                wx[i] = cx + w / 2
                wy[i] = rng.uniform(cy - d / 2, cy + d / 2)
            else:
                wx[i] = cx - w / 2
                wy[i] = rng.uniform(cy - d / 2, cy + d / 2)
        parts.append(np.column_stack([wx, wy, wz]))
    trees = [(50, 50, 5, 0), (180, 200, 6, 0), (300, 450, 4, 0), (420, 250, 7, 0),
             (80, 400, 5, 0), (450, 50, 4, 0), (200, 80, 5, 0), (350, 350, 6, 0)]
    n_per_tree = int(20_000 * scale)
    for cx, cy, r, base in trees:
        n_canopy = int(n_per_tree * 0.8)
        count = 0
        canopy_pts = []
        while count < n_canopy:
            batch = 2 * n_canopy
            px = rng.uniform(-1, 1, batch)
            py = rng.uniform(-1, 1, batch)
            r2 = px ** 2 + py ** 2
            mask = r2 < 1.0
            px, py, r2 = px[mask], py[mask], r2[mask]
            pz = np.sqrt(1.0 - r2)
            pts = np.column_stack([
                (cx + px[:n_canopy - count] * r).astype(np.float32),
                (cy + py[:n_canopy - count] * r).astype(np.float32),
                (base + 4 + pz[:n_canopy - count] * r).astype(np.float32),
            ])
            canopy_pts.append(pts)
            count += len(pts)
        parts.append(np.vstack(canopy_pts)[:n_canopy])
        n_trunk = n_per_tree - n_canopy
        trunk_x = cx + rng.normal(0, 0.15, n_trunk).astype(np.float32)
        trunk_y = cy + rng.normal(0, 0.15, n_trunk).astype(np.float32)
        trunk_z = rng.uniform(base, base + 4, n_trunk).astype(np.float32)
        parts.append(np.column_stack([trunk_x, trunk_y, trunk_z]))
    return np.ascontiguousarray(np.vstack(parts), dtype=np.float32)


def hemisphere(n: int, seed: int = 99, radius: float = 5.0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    out = np.empty((n, 3), np.float32)
    got = 0
    while got < n:
        m = 2 * (n - got) + 16
        px = rng.uniform(-1.0, 1.0, m).astype(np.float32)
        py = rng.uniform(-1.0, 1.0, m).astype(np.float32)
        r2 = px * px + py * py
        ok = r2 < 1.0
        px, py, r2 = px[ok], py[ok], r2[ok]
        pz = np.sqrt(np.float32(1.0) - r2)
        take = min(n - got, len(px))
        out[got:got + take, 0] = px[:take] * np.float32(radius)
        out[got:got + take, 1] = py[:take] * np.float32(radius)
        out[got:got + take, 2] = pz[:take] * np.float32(radius)
        got += take
    return out


def uniform_cube(n: int, seed: int = 42, lo: float = 0.0, hi: float = 100.0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    return rng.uniform(lo, hi, (n, 3)).astype(np.float32)


def rot_z(angle: float) -> np.ndarray:
    c, s = np.float32(np.cos(np.float32(angle))), np.float32(np.sin(np.float32(angle)))
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]], np.float32)


def voxel_downsample_np(pts: np.ndarray, voxel_size: float) -> np.ndarray:
    """numpy restatement of voxel_downsample (crates/filters/src/voxel_downsample.rs:12-65): input
    preparation for BASELINE config 2 (it is not on the KNN path).  key = floor(p / voxel) as i32,
    per-voxel f32 sums in input order, mean = sum / count, output sorted by key."""
    if not np.isfinite(voxel_size) or voxel_size <= 0:
        raise ValueError("voxel_size must be > 0 and finite")
    pts = np.asarray(pts, np.float32).reshape(-1, 3)
    ok = np.isfinite(pts).all(axis=1)
    p = pts[ok]
    if len(p) == 0:
        return np.zeros((0, 3), np.float32)
    key = np.floor(p / np.float32(voxel_size)).astype(np.int64).clip(-2**31, 2**31 - 1)
    order = np.lexsort((np.arange(len(p)), key[:, 2], key[:, 1], key[:, 0]))  # key order, then input order
    ks = key[order]
    new = np.ones(len(p), bool)
    new[1:] = (ks[1:] != ks[:-1]).any(axis=1)
    seg = np.cumsum(new) - 1
    sums = np.zeros((seg[-1] + 1, 3), np.float32)
    np.add.at(sums, seg, p[order])  # unbuffered: sequential f32 adds in input order
    cnt = np.bincount(seg).astype(np.float32)
    return (sums / cnt[:, None]).astype(np.float32)


# ---------------------------------------------------------------------------------------------------
# Adversarial scenes for the exact KNN engine (tests/test_knn_routes.py).  Each one is built to reach a route or a branch
# of the level-0 self-query search that the gentle scenes above seldom reach: exact distance ties at the k-th place,
# duplicate points, candidate counts beyond what one cell tile can stage, k-th neighbours far outside the uniform-sheet
# model, queries on cell faces and degenerate (flat) grids.
# ---------------------------------------------------------------------------------------------------

def tie_grid(seed: int = 1, dims=(160, 160, 4), occupancy: float = 0.3) -> np.ndarray:
    """A random `occupancy` share of the integer box `dims`, rows shuffled, scaled by 2^-4 and offset by 4096.  Every
    coordinate, difference and d^2 is exact in f32, so equal distances are equal bits: most queries have a tie across the
    k-th place (the index breaks it).  The cell tile's ranking puts such ties in (d^2, index) order with its bubble pass
    (tile_fix), and the thread-per-query selection of external queries with its slow exact path (sel_exact_slow).  The
    tie groups stay within the tile's 32 slots for k <= 21, so the tile's exact-tie hand-back is left to dup_cloud."""
    rng = np.random.default_rng(seed)
    nx, ny, nz = dims
    sites = np.flatnonzero(rng.random(nx * ny * nz) < occupancy)
    rng.shuffle(sites)
    ijk = np.stack(np.unravel_index(sites, dims), 1).astype(np.float32)
    return np.ascontiguousarray(ijk * np.float32(1.0 / 16.0) + np.float32(4096.0), np.float32)


def dup_cloud(seed: int = 2, counts=(8_000, 400, 70, 500), max_copies: int = 6, n_big: int = 4, big_copies: int = 40,
              n_nonfinite: int = 7) -> np.ndarray:
    """A KITTI-shaped frame in which every point is repeated 1..max_copies times at scattered indices: groups of points at
    d^2 = 0 larger than a small k, whose members only the index tells apart.  `n_big` of the scattered noise points are
    repeated `big_copies` times: more candidates at d^2 = 0 than the cell tile's 32 slots, which it hands back to the warp
    kernels.  A few non-finite rows keep no list."""
    rng = np.random.default_rng(seed)
    base = kitti_scene(seed, counts)
    rep = rng.integers(1, max_copies + 1, len(base))
    rep[0] = max_copies  # (at least one group of the largest size)
    rep[len(base) - n_big:] = big_copies  # (the last rows of kitti_scene are its noise points)
    pts = np.repeat(base, rep, axis=0)
    pts = pts[rng.permutation(len(pts))]
    bad = rng.choice(len(pts), n_nonfinite, replace=False)
    pts[bad[0::3], 0] = np.nan
    pts[bad[1::3], 1] = np.inf
    pts[bad[2::3], 2] = -np.inf
    return np.ascontiguousarray(pts, np.float32)


def density_ramp(seed: int = 3, n_sheet: int = 30_000, ratio: float = 100.0, n_box: int = 1_500) -> np.ndarray:
    """A 40 x 10 m sheet whose density rises `ratio`-fold along x, plus three compact 0.3 m boxes.  One cell size serves
    the whole frame, so the candidates in a query's 27 cells run from a handful to thousands: past the tile kernel's
    dense-class bound (128), the selection histogram's (384) and what one sub-tile can stage (512 points), which forces
    the smaller sub-tile attempts and the dense class on the finer level."""
    rng = np.random.default_rng(seed)
    u = rng.random(n_sheet)
    x = 40.0 * np.log1p(u * (ratio - 1.0)) / np.log(ratio)  # density proportional to ratio^(x / 40)
    sheet = np.column_stack([x, rng.uniform(0.0, 10.0, n_sheet), rng.normal(0.0, 0.01, n_sheet)])
    parts = [sheet]
    for cx, cy in ((5.0, 5.0), (20.0, 2.0), (38.0, 8.0)):
        parts.append(np.column_stack([rng.uniform(cx, cx + 0.3, n_box), rng.uniform(cy, cy + 0.3, n_box), rng.uniform(0.1, 0.4, n_box)]))
    pts = np.vstack(parts)
    return np.ascontiguousarray(pts[rng.permutation(len(pts))], np.float32)


def wires(seed: int = 4, n_sheet: int = 20_000, n_wires: int = 6, spacing: float = 0.3, n_isolated: int = 40) -> np.ndarray:
    """Sparse polylines 3-6 m above a 20 x 20 m sheet, and isolated points tens of metres away.  A wire point's k-th
    neighbour lies k/2 spacings along the wire, far beyond what the sheet's density predicts (the selection's histogram
    has to widen); the isolated points have almost no candidates in their cells (the sparse class, searched on the
    coarser level) or need the coarser levels altogether."""
    rng = np.random.default_rng(seed)
    parts = [np.column_stack([rng.uniform(0.0, 20.0, n_sheet), rng.uniform(0.0, 20.0, n_sheet), rng.normal(0.0, 0.02, n_sheet)])]
    for _ in range(n_wires):
        a = np.append(rng.uniform(0.0, 20.0, 2), rng.uniform(3.0, 6.0))
        b = np.append(rng.uniform(0.0, 20.0, 2), rng.uniform(3.0, 6.0))
        m = max(2, int(np.linalg.norm(b - a) / spacing))
        t = np.linspace(0.0, 1.0, m)[:, None]
        parts.append(a + t * (b - a) + rng.normal(0.0, 0.005, (m, 3)))
    iso = rng.uniform(-60.0, 80.0, (n_isolated, 3))
    iso[:, 2] = rng.uniform(10.0, 40.0, n_isolated)
    parts.append(iso)
    pts = np.vstack(parts)
    return np.ascontiguousarray(pts[rng.permutation(len(pts))], np.float32)


def faces(seed: int = 5, n: int = 25_000, dims=(128, 128, 16)) -> np.ndarray:
    """Distinct random sites of the 2^-4 lattice in an 8 x 8 x 1 m box.  With a cell size of 0.25 (four lattice steps),
    a quarter of the coordinates lie exactly on a cell face on each axis, and candidates lie exactly at the ring bound of
    the search's stopping rule; d^2 is exact, so ties are exact too."""
    rng = np.random.default_rng(seed)
    sites = rng.choice(dims[0] * dims[1] * dims[2], n, replace=False)
    ijk = np.stack(np.unravel_index(sites, dims), 1).astype(np.float32)
    return np.ascontiguousarray(ijk * np.float32(1.0 / 16.0), np.float32)


def flat(seed: int = 6, n_sheet: int = 20_000, n_line: int = 2_000) -> np.ndarray:
    """An exactly planar sheet (z = 0) and an exactly straight line in the same plane: the grid has one cell along z, so
    every cube of cells is cut by the grid boundary."""
    rng = np.random.default_rng(seed)
    sheet = np.column_stack([rng.uniform(0.0, 20.0, n_sheet), rng.uniform(0.0, 20.0, n_sheet), np.zeros(n_sheet)])
    line = np.column_stack([rng.uniform(0.0, 30.0, n_line), np.full(n_line, -5.0), np.zeros(n_line)])
    pts = np.vstack([sheet, line])
    return np.ascontiguousarray(pts[rng.permutation(len(pts))], np.float32)


def straight_line(seed: int = 7, n: int = 3_000) -> np.ndarray:
    """Points of one exactly straight line along x: a grid of one cell on two axes."""
    rng = np.random.default_rng(seed)
    return np.ascontiguousarray(np.column_stack([rng.uniform(-10.0, 10.0, n), np.full(n, 2.5), np.full(n, -1.0)]), np.float32)


ADVERSARIAL = {
    "tie_grid": tie_grid,
    "dup_cloud": dup_cloud,
    "density_ramp": density_ramp,
    "wires": wires,
    "faces": faces,
    "flat": flat,
}


def adversarial_batch(seed: int = 8):
    """The adversarial scenes as frames of one batch, with the small frames a batch meets: 95, 96 and 97 points (either
    side of the size below which a frame is scanned whole), seven points (fewer than most k), one point, an empty frame and
    a straight line.  -> (points (N,3) f32, frame offsets (F+1,) u64)."""
    rng = np.random.default_rng(seed)
    frames = [f() for f in ADVERSARIAL.values()]
    frames += [uniform_cube(95, seed + 1, 0, 2), uniform_cube(96, seed + 2, 0, 2), uniform_cube(97, seed + 3, 0, 2),
               uniform_cube(7, seed + 4, 0, 1), uniform_cube(1, seed + 5), np.zeros((0, 3), np.float32), straight_line()]
    order = rng.permutation(len(frames))
    frames = [frames[i] for i in order]
    off = np.zeros(len(frames) + 1, np.uint64)
    off[1:] = np.cumsum([len(f) for f in frames])
    return np.ascontiguousarray(np.vstack(frames), np.float32), off
