"""The self-query KNN lists, route by route, against a brute-force reference and the CPU oracle.

Every level-0 route of the self-query search (cell tiles, their hand-back to the warp kernels, the dense class on the
finer level, the sparse class on the coarser one, the follow-up pass, the thread-per-query selection, the insertion and
shared-memory kernels) must return the same list: the K smallest (d^2, index) keys.  The consumers of these lists (SOR
mean distances, normals) cannot see which member of a tie group is in a list, so the lists themselves are compared here,
index for index, on scenes built to reach each route (pointclouds_rs_b200.scenes.ADVERSARIAL).

The CPU tests check the reference against the oracle and the scenes against the properties they are built to have.
"""
import functools
import math
import os

import numpy as np
import pytest

from pointclouds_rs_b200 import scenes

T = max(1, min(16, os.cpu_count() or 1))
KS = [2, 3, 11, 12, 13, 20, 21, 22, 24, 25, 32]
NONE = 0xFFFFFFFF


# ---- reference ------------------------------------------------------------------------------------------------

def _d2(pts, q):
    """f32 d^2 of the queries q (m,3) to every point, each operation rounded: ((dx*dx)+(dy*dy))+(dz*dz)."""
    dx = pts[None, :, 0] - q[:, None, 0]
    dy = pts[None, :, 1] - q[:, None, 1]
    dz = pts[None, :, 2] - q[:, None, 2]
    return (dx * dx + dy * dy) + dz * dz


def brute_keys(pts, queries, K, chunk=128):
    """The K smallest keys (d^2 bits << 32 | index) of every query, ascending; non-finite points are not candidates.
    -> (keys (m,K) u64, padded with all-ones, counts (m,))."""
    pts = np.asarray(pts, np.float32)
    queries = np.asarray(queries, np.float32).reshape(-1, 3)
    fin = np.flatnonzero(np.isfinite(pts).all(1))
    p, ids = pts[fin], fin.astype(np.uint64)
    kk = min(K, len(fin))
    out = np.full((len(queries), K), np.uint64(2**64 - 1), np.uint64)
    for s in range(0, len(queries), chunk):
        d2 = _d2(p, queries[s:s + chunk]).astype(np.float32)
        key = (d2.view(np.uint32).astype(np.uint64) << np.uint64(32)) | ids[None, :]
        if kk:
            part = np.partition(key, kk - 1, axis=1)[:, :kk] if kk < len(fin) else key
            out[s:s + chunk, :kk] = np.sort(part, axis=1)
    ok = np.isfinite(queries).all(1)
    out[~ok] = np.uint64(2**64 - 1)
    return out, np.where(ok, kk, 0)


def key_index(keys):
    idx = (keys & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    idx[keys == np.uint64(2**64 - 1)] = NONE
    return idx


def key_d2(keys):
    return (keys >> np.uint64(32)).astype(np.uint32).view(np.float32)


def sample_rows(n, m, seed=0):
    return np.sort(np.random.default_rng(seed).choice(n, min(n, m), replace=False))


@functools.lru_cache(maxsize=None)
def scene(name):
    return scenes.ADVERSARIAL[name]()


@functools.lru_cache(maxsize=None)
def batch():
    return scenes.adversarial_batch()


def engine_cell(pts, k_hint):
    """The cell size the index build starts from for a self-query search (grid_build.cu occupancy_target, initial_cell)."""
    p = pts[np.isfinite(pts).all(1)].astype(np.float64)
    target = min(64.0, max(2.0, (0.5 if k_hint <= 24 else 0.25) * k_hint))
    e = np.sort(p.max(0) - p.min(0))
    tiny = max(e[2] * 1e-6, 1e-30)
    vol = max(e[0], tiny) * max(e[1], tiny) * max(e[2], tiny)
    area = max(e[1], tiny) * max(e[2], tiny)
    return math.sqrt(math.sqrt(area * target / len(p)) * math.cbrt(vol * target / len(p)))


def cube_counts(pts, h):
    """Points in the 3x3x3 cells around every point's cell, for cells of size h from the box minimum."""
    p = pts[np.isfinite(pts).all(1)].astype(np.float64)
    c = np.floor((p - p.min(0)) / h).astype(np.int64)
    dims = c.max(0) + 3
    key = lambda a: ((a[:, 0] + 1) * dims[1] + a[:, 1] + 1) * dims[2] + a[:, 2] + 1
    cells, per = np.unique(key(c), return_counts=True)
    total = np.zeros(len(p), np.int64)
    for d in np.stack(np.meshgrid([-1, 0, 1], [-1, 0, 1], [-1, 0, 1]), -1).reshape(-1, 3):
        kk = key(c + d)
        at = np.searchsorted(cells, kk).clip(0, len(cells) - 1)
        total += np.where(cells[at] == kk, per[at], 0)
    return total


# ---- CPU: the reference and the scenes --------------------------------------------------------------------------

@pytest.mark.parametrize("name", list(scenes.ADVERSARIAL))
def test_reference_equals_oracle(oracle, name):
    pts = scene(name)
    rows = sample_rows(len(pts), 2000, 1)
    keys, cnt = brute_keys(pts, pts[rows], max(KS))
    tree = oracle.Tree(pts)
    for K in KS:  # (a top-K list under a total order is the prefix of the top-32 list)
        o_idx, o_dist, o_cnt = tree.knn_batch(pts[rows], K, threads=T)
        assert np.array_equal(o_cnt, np.minimum(cnt, K))
        for r in range(len(rows)):
            c = int(o_cnt[r])
            assert np.array_equal(o_idx[r, :c], key_index(keys[r, :c])), (name, K, rows[r])
            assert np.array_equal(o_dist[r, :c].view(np.uint32), np.sqrt(key_d2(keys[r, :c])).view(np.uint32))


def test_reference_equals_oracle_on_the_batch_layout(oracle):
    pts, off = batch()
    for f in range(len(off) - 1):
        fp = pts[off[f]:off[f + 1]]
        if len(fp) == 0:
            continue
        rows = sample_rows(len(fp), 300, f)
        keys, cnt = brute_keys(fp, fp[rows], max(KS))
        o_idx, _, o_cnt = oracle.Tree(fp).knn_batch(fp[rows], max(KS), threads=T)
        assert np.array_equal(o_cnt, cnt)
        for r in range(len(rows)):
            assert np.array_equal(o_idx[r, :o_cnt[r]], key_index(keys[r, :cnt[r]]))


def tie_share(pts, K, rows):
    """Share of the queries whose K-th and (K+1)-th smallest d^2 are equal: the index decides who is in the list."""
    keys, _ = brute_keys(pts, pts[rows], K + 1)
    d = key_d2(keys)
    return float(np.mean(d[:, K - 1] == d[:, K]))


def test_tie_grid_is_exact_and_tie_heavy():
    pts = scene("tie_grid")
    assert len(pts) > 30_000
    steps = (pts.astype(np.float64) - 4096.0) * 16.0
    assert np.array_equal(steps, np.round(steps)) and steps.min() >= 0 and steps.max() < 160
    assert len(np.unique(pts, axis=0)) == len(pts)
    rows = sample_rows(len(pts), 500, 2)
    d32 = _d2(pts, pts[rows[:50]])
    d64 = _d2(pts.astype(np.float64), pts[rows[:50]].astype(np.float64))
    assert np.array_equal(d32.astype(np.float64), d64)  # every d^2 is exact
    for K in (12, 25):
        assert tie_share(pts, K, rows) > 0.6, K
    # candidates at or below the K-th distance at K = 21, the largest K of the cell tiles: tie groups that run 8 or more
    # places past the K-th (deep ties for the bubble pass), but never past the tile's 32 slots (no exact-tie hand-back)
    d2 = np.sort(_d2(pts, pts[rows]).astype(np.float32), axis=1)
    at_or_below = np.sum(d2 <= d2[:, 20:21], axis=1)
    assert np.mean(at_or_below >= 21 + 8) > 0.01
    assert at_or_below.max() <= 32


def test_dup_cloud_has_large_scattered_duplicate_groups():
    pts = scene("dup_cloud")
    fin = np.isfinite(pts).all(1)
    assert (~fin).sum() == 7
    u, inv, cnt = np.unique(pts[fin], axis=0, return_inverse=True, return_counts=True)
    assert np.mean(cnt[inv.ravel()] > 3) > 0.3  # groups at d^2 = 0 larger than K = 2, 3
    assert np.sum(cnt == 6) > 1000 and np.sum(cnt == 40) == 4 and cnt.max() == 40  # ... and larger than 32
    n27 = cube_counts(pts, engine_cell(pts, 12))
    assert np.all(n27[cnt[inv.ravel()] == 40] <= 128)  # (the 40-fold groups are not dense: they run on the cell tiles)
    last = np.zeros(len(u), np.int64)
    order = np.flatnonzero(fin)
    np.maximum.at(last, inv.ravel(), order)
    first = np.full(len(u), len(pts))
    np.minimum.at(first, inv.ravel(), order)
    big = cnt >= 3
    assert np.median((last - first)[big]) > 1000  # members of a group are far apart in the index order


def test_density_ramp_crosses_the_tile_bounds():
    pts = scene("density_ramp")
    for K in (3, 12, 21):
        n27 = cube_counts(pts, engine_cell(pts, K))
        assert np.mean(n27 > 128) > 0.05, K   # dense class (tile bound)
        assert np.mean(n27 > 512) > 0.02, K   # more than one sub-tile can stage
        assert np.any((n27 > 384) & (n27 <= 512)), K
        assert np.mean(n27 <= 128) > 0.2, K   # ... while many queries stay normal


def test_wires_reach_far_and_isolated_points_are_sparse():
    pts = scene("wires")
    K = 12
    d = np.sqrt(key_d2(brute_keys(pts, pts, K)[0])[:, K - 1])
    on_sheet = np.abs(pts[:, 2]) < 0.2
    wire = (pts[:, 2] >= 2.5) & (pts[:, 2] <= 6.5) & (np.abs(pts[:, :2] - 10).max(1) <= 10)
    assert wire.sum() > 200
    assert np.median(d[wire]) > 4 * np.median(d[on_sheet])  # far outside the uniform-sheet model
    n27 = cube_counts(pts, engine_cell(pts, K))
    assert np.sum(n27 * 4 < K) >= 20  # the sparse class
    assert np.sum(d > 5.0) >= 20       # and k-th neighbours many cells away


def test_faces_sit_on_cell_faces():
    pts = scene("faces")
    assert len(np.unique(pts, axis=0)) == len(pts)
    on_face = (pts / np.float32(0.25)) == np.floor(pts / np.float32(0.25))
    assert on_face.mean(0).min() > 0.2
    assert tie_share(pts, 12, sample_rows(len(pts), 500, 3)) > 0.5


def test_flat_is_exactly_flat():
    pts = scene("flat")
    assert np.all(pts[:, 2] == 0)
    assert np.sum(pts[:, 1] == -5) == 2000
    line = scenes.straight_line()
    assert np.all(line[:, 1] == line[0, 1]) and np.all(line[:, 2] == line[0, 2])


def test_batch_layout_has_the_edge_frames():
    pts, off = batch()
    sizes = np.diff(off).astype(np.int64)
    for m in (0, 1, 7, 95, 96, 97):
        assert m in sizes
    assert len(pts) == off[-1]


# ---- GPU: the lists ---------------------------------------------------------------------------------------------

LIST_CASES = [("tie_grid", None), ("dup_cloud", None), ("density_ramp", None), ("wires", None), ("faces", None),
              ("faces", 0.25), ("flat", None)]


@pytest.fixture(scope="module")
def pinned_ctx(pcr):
    ctx = pcr.Context()
    ctx.set_cell_size(0.25)
    yield ctx
    ctx.close()


@functools.lru_cache(maxsize=None)
def oracle_lists(name, K, frame=None):
    from oracle import oracle as O

    if frame is None:
        pts = scene(name)
    else:
        pts, off = batch()
        pts = pts[off[frame]:off[frame + 1]]
    return O.Tree(pts).knn_batch(pts, K, threads=T)


def check_lists(pts, idx, cnt, o_idx, o_cnt, K, what, seed=0):
    """idx / cnt from the engine against the oracle on every point with a list, and the brute reference on a sample."""
    fin = np.isfinite(pts).all(1)
    assert np.all(cnt[~fin] == 0xFF), what
    has = cnt != 0xFF
    assert np.array_equal(cnt[has], o_cnt[has]), what
    for c in np.unique(cnt[has]):
        rows = np.flatnonzero(has & (cnt == c))
        bad = np.flatnonzero((idx[rows, :c] != o_idx[rows, :c]).any(1))
        assert len(bad) == 0, f"{what}: {len(bad)} lists differ, first point {rows[bad[0]]}: {idx[rows[bad[0]]]} vs {o_idx[rows[bad[0]]]}"
        assert np.all(idx[rows, c:] == NONE), what
    rows = sample_rows(len(pts), 150, seed)
    rows = rows[has[rows]]
    keys, b_cnt = brute_keys(pts, pts[rows], K)
    assert np.array_equal(cnt[rows], b_cnt), what
    assert np.array_equal(idx[rows], key_index(keys)), what
    return has[fin].mean() if fin.any() else 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("name,cell", LIST_CASES)
@pytest.mark.parametrize("K", KS)
def test_self_lists_single_frame(pcr, pinned_ctx, name, cell, K):
    pts = scene(name)
    idx, cnt, routes = pcr.debug_self_knn_lists(pts, [0, len(pts)], K, ctx=pinned_ctx if cell else None)
    o_idx, _, o_cnt = oracle_lists(name, K)
    share = check_lists(pts, idx, cnt, o_idx, o_cnt, K, f"{name} cell={cell} K={K}")
    assert share >= 0.9, f"only {share:.3f} of the finite points kept a list: {routes}"
    n_fin = int(np.isfinite(pts).all(1).sum())
    if K <= 21:  # the class split: normal, dense and sparse are disjoint; the rest (thin queries) run in the follow-up pass
        split = routes["normal"] + routes["dense"] + routes["sparse"]
        assert split <= n_fin <= split + routes["follow_up"], routes
    else:
        assert routes["normal"] == routes["dense"] == routes["sparse"] == routes["follow_up"] == routes["handed_back"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("K", KS)
def test_self_lists_batch(pcr, K):
    pts, off = batch()
    idx, cnt, routes = pcr.debug_self_knn_lists(pts, off, K)
    line = len(scenes.straight_line())
    for f in range(len(off) - 1):
        b, e = int(off[f]), int(off[f + 1])
        if b == e:
            continue
        o_idx, _, o_cnt = oracle_lists(None, K, f)
        share = check_lists(pts[b:e], idx[b:e], cnt[b:e], o_idx, o_cnt, K, f"frame {f} ({e - b} points) K={K}", seed=f)
        # (a straight line's 27 cells hold too few points for most of its queries: they go to the coarser levels, which keep
        # no list; its lists are checked where there are some, its other queries through KdTreeBatch below)
        assert share >= 0.9 or e - b == line, (f, share, routes)
    fin = np.isfinite(pts).all(1)
    assert np.mean(cnt[fin] != 0xFF) >= 0.9


@pytest.mark.gpu
def test_self_lists_arguments(pcr):
    from pointclouds_rs_b200 import _ffi

    pts = scene("flat")[:500]
    for K in (0, 1, 33):
        with pytest.raises(_ffi.PcrError) as e:
            pcr.debug_self_knn_lists(pts, [0, len(pts)], K)
        assert e.value.code == _ffi.PCR_ERR_UNSUPPORTED
    with pytest.raises(ValueError):
        pcr.debug_self_knn_lists(pts, [0, 300, 200], 8)
    idx, cnt, routes = pcr.debug_self_knn_lists(pts[:0], [0, 0], 8)
    assert idx.shape == (0, 8) and not any(routes.values())
    _, _, routes = pcr.debug_self_knn_lists(pts, [0, len(pts)], 22)
    assert routes["normal"] == routes["dense"] == routes["sparse"] == routes["follow_up"] == routes["handed_back"] == 0


@pytest.mark.gpu
def test_routes_are_reached(pcr, pinned_ctx):
    """Each level-0 route of the class split (K <= 21) runs on the scene built for it."""
    total = {}
    for name, cell in LIST_CASES:
        pts = scene(name)
        tot = None
        for K in (3, 12, 21):
            _, _, r = pcr.debug_self_knn_lists(pts, [0, len(pts)], K, ctx=pinned_ctx if cell else None)
            print(f"routes {name:12s} cell={cell} K={K:2d}: {r}")
            assert r["normal"] > 0, (name, K, r)
            tot = r if tot is None else {k: tot[k] + v for k, v in r.items()}
        total[(name, cell)] = tot
    assert total[("density_ramp", None)]["dense"] > 0
    assert total[("wires", None)]["sparse"] > 0 and total[("wires", None)]["deferred"] > 0
    assert sum(t["follow_up"] for t in total.values()) > 0
    # (the exact-tie hand-back needs more than 32 candidates below the tile's threshold: the 40-fold duplicates; the tie
    # groups of tie_grid stay within the 32 slots for K <= 21 and are put in index order by the tile's bubble pass)
    assert total[("dup_cloud", None)]["handed_back"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 12, 21, 25, 32])
def test_kdtree_batch_knn_on_the_batch_layout(pcr, oracle, k):
    """External queries against the batch index (no cell tiles for them): every frame's points as its queries, frame by
    frame bit-exact against the oracle, distances included."""
    pts, off = batch()
    idx, dist, cnt = pcr.KdTreeBatch(pts, off, k_hint=k).knn(pts, off, k)
    for f in range(len(off) - 1):
        b, e = int(off[f]), int(off[f + 1])
        if b == e:
            continue
        o_idx, o_dist, o_cnt = oracle.Tree(pts[b:e]).knn_batch(pts[b:e], k, threads=T)
        assert np.array_equal(cnt[b:e], o_cnt), f
        assert np.array_equal(idx[b:e], o_idx), f"frame {f}: first diff row {np.nonzero((idx[b:e] != o_idx).any(1))[0][:5]}"
        assert np.array_equal(dist[b:e].view(np.uint32), o_dist.view(np.uint32)), f
