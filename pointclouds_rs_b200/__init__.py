"""pointclouds_rs_b200 -- B200-native drop-in for the KNN hot path of pointclouds-rs ("pcrs").

The module mirrors the names and argument meaning of the reference's PyO3 module `pointclouds_rs`
(crates/python/src/lib.rs:12-49) for the functions that sit on the KNN path:

    PointCloud                                    crates/python/src/cloud.rs:10-88
    statistical_outlier_removal(cloud, k, std_mul)      crates/python/src/filters.rs:36-49
    radius_outlier_removal(cloud, radius, min_neighbors) crates/python/src/filters.rs:51-66
    estimate_normals(cloud, k)                          crates/python/src/normals.rs:4-10
    icp_point_to_point / icp_point_to_plane / apply_transform / IcpResult
                                                        crates/python/src/registration.rs:4-109
    KdTree (batched)                                    crates/spatial/src/kdtree.rs:14-164
    KdTreeBatch                                         KdTree over many frames per call, each frame searched alone

and for the steps either side of it (SURVEY.md section 8f):

    voxel_downsample(cloud, voxel_size)                 crates/python/src/filters.rs (voxel_downsample.rs:12-65)
    euclidean_cluster(cloud, threshold, min, max)       crates/segmentation/src/euclidean_cluster.rs:96-187
    ransac_plane(cloud, threshold, iterations)          crates/segmentation/src/ransac_plane.rs:56-129 (after the sampling step)
    DeviceCloud                                         a PointCloud that stays in HBM between the steps of a pipeline
    DeviceFrames                                        a batch of frames that stays in HBM between the batch calls
    apply_transform_batch / compose / chain_poses       apply_transform of many frames per call, RigidTransform::compose
                                                        (icp.rs:39-92), and the poses of an odometry chain

Everything runs through the C ABI (include/pcr_b200.h) of lib/libpcr_b200.so: hand-written sm_100a
CUDA, no PyTorch on the path, no CPU fallback.  Out of scope (DESIGN.md section 8): passthrough_filter and file IO.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import weakref
from typing import List, Optional, Sequence

import numpy as np

from . import _ffi
from ._ffi import PcrError  # noqa: F401

__all__ = [
    "PointCloud", "KdTree", "IcpResult", "Context",
    "statistical_outlier_removal", "radius_outlier_removal", "estimate_normals",
    "icp_point_to_point", "icp_point_to_plane", "apply_transform", "find_correspondences",
    "icp_point_to_point_batch", "icp_point_to_plane_batch", "voxel_downsample_batch", "estimate_normals_batch",
    "sor_normals_batch", "default_context", "PcrError", "euclidean_cluster", "voxel_downsample", "DeviceCloud", "ransac_plane", "PlaneResult",
    "ransac_plane_samples_batch", "ransac_plane_batch", "cluster_arrays_batch", "euclidean_cluster_batch",
    "DeviceFrames", "radius_outlier_removal_batch", "KdTreeBatch", "apply_transform_batch", "compose", "chain_poses",
]


def _p(a: Optional[np.ndarray], t):
    return a.ctypes.data_as(t) if a is not None else None


class Context:
    """Owns a pcr_ctx (device, stream, scratch).  One per host thread."""

    def __init__(self, device: Optional[int] = None, stream: Optional[int] = None):
        lib = _ffi.load()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
            if lib.pcr_device_count() and device >= lib.pcr_device_count():
                device = 0
        h = C.c_void_p()
        if stream is None:
            st = lib.pcr_ctx_create(device, C.byref(h))
        else:
            st = lib.pcr_ctx_create_on_stream(device, C.c_void_p(stream), C.byref(h))
        _ffi.check(st)
        self._h = h
        self.device = device
        self._clouds = weakref.WeakSet()  # live DeviceClouds: they must be freed before the context is destroyed

    def close(self):
        if getattr(self, "_h", None):
            for cl in list(getattr(self, "_clouds", ())):
                cl.free()
            _ffi.load().pcr_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        _ffi.check(_ffi.load().pcr_ctx_synchronize(self._h), self._h)

    @property
    def launch_count(self) -> int:
        return int(_ffi.load().pcr_ctx_launch_count(self._h))

    def set_timing(self, enable: bool):
        _ffi.check(_ffi.load().pcr_ctx_set_timing(self._h, 1 if enable else 0), self._h)

    def get_timing(self):
        """-> {tag: (milliseconds, spans)} accumulated since the previous call (synchronises)."""
        ms = (C.c_double * _ffi.PCR_NUM_TIMING_TAGS)()
        cnt = (C.c_uint64 * _ffi.PCR_NUM_TIMING_TAGS)()
        _ffi.check(_ffi.load().pcr_ctx_get_timing(self._h, ms, cnt), self._h)
        return {_ffi.TIMING_TAGS[i]: (ms[i], int(cnt[i])) for i in range(_ffi.PCR_NUM_TIMING_TAGS)}

    def set_frame_stream(self, enable: bool = True):
        """Consecutive clouds are frames of one sensor stream: reuse the probed cell size between similar frames."""
        _ffi.check(_ffi.load().pcr_ctx_set_frame_stream(self._h, 1 if enable else 0), self._h)

    def knn_counters(self) -> dict:
        """{queries, candidates}: work of the level-0 KNN kernel since the previous call (counted while timing is on)."""
        out = (C.c_uint64 * 2)()
        _ffi.check(_ffi.load().pcr_ctx_get_knn_counters(self._h, out), self._h)
        return {"queries": int(out[0]), "candidates": int(out[1])}

    def hint_stats(self) -> dict:
        """How often the frame-stream hints held (pcr_ctx_get_hint_stats)."""
        out = (C.c_uint64 * 8)()
        _ffi.check(_ffi.load().pcr_ctx_get_hint_stats(self._h, out), self._h)
        names = ("cell_size_reused", "cell_size_probed", "voxel_box_guess_held", "voxel_box_guess_missed", "coarser_level_ahead_needed",
                 "coarser_level_ahead_unneeded", "deferred_counts_not_awaited_zero", "deferred_counts_not_awaited_nonzero")
        return {k: int(v) for k, v in zip(names, out)}

    def set_query_sharding(self, enable: bool = True):
        """With a communicator (comm_init): SOR / normals / radius outlier removal of ONE cloud, given in full on every rank,
        search only this rank's share of the queries and merge the results over NCCL (SURVEY.md 8e)."""
        _ffi.check(_ffi.load().pcr_ctx_set_query_sharding(self._h, 1 if enable else 0), self._h)

    def debug_set_shard(self, rank: int, world_size: int):
        """Test hook (pcr_ctx_debug_set_shard): play one rank of a query-sharded call without a communicator."""
        _ffi.check(_ffi.load().pcr_ctx_debug_set_shard(self._h, int(rank), int(world_size)), self._h)

    def set_cell_size(self, cell: float):
        _ffi.check(_ffi.load().pcr_ctx_set_cell_size(self._h, float(cell)), self._h)

    # multi-GPU: the host exchanges the id (e.g. torch.distributed.broadcast_object_list)
    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(_ffi.PCR_UNIQUE_ID_BYTES)
        _ffi.check(_ffi.load().pcr_comm_unique_id(buf))
        return buf.raw

    def comm_init(self, uid: bytes, rank: int, world_size: int):
        buf = C.create_string_buffer(uid, _ffi.PCR_UNIQUE_ID_BYTES)
        _ffi.check(_ffi.load().pcr_ctx_comm_init(self._h, buf, rank, world_size), self._h)

    @property
    def comm_kind(self) -> str:
        """How the sharded ICP all-reduces its normal equations on this context: 'none', 'nccl' or 'peer' (NVLink peer memory)."""
        return ("none", "nccl", "peer")[_ffi.load().pcr_ctx_comm_kind(self._h)]


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context()
    return _default_ctx


def _soa(a: np.ndarray):
    x = np.ascontiguousarray(a[:, 0])
    y = np.ascontiguousarray(a[:, 1])
    z = np.ascontiguousarray(a[:, 2])
    return x, y, z


class PointCloud:
    """SoA point cloud (crates/core/src/cloud.rs:4-11) with the PyO3 class's surface."""

    def __init__(self):
        self.x = np.empty(0, np.float32)
        self.y = np.empty(0, np.float32)
        self.z = np.empty(0, np.float32)
        self.normals: Optional[np.ndarray] = None  # (N,3) f32
        self._nsoa = None  # (the array `normals` was when split, (nx, ny, nz)): the reference's Normals are SoA (cloud.rs:13-18)

    @staticmethod
    def _from_xyz(x, y, z, normals=None) -> "PointCloud":
        pc = PointCloud()
        pc.x, pc.y, pc.z = x, y, z
        pc.normals = normals
        return pc

    @staticmethod
    def from_numpy(array) -> "PointCloud":
        # crates/python/src/cloud.rs:25-37,91-137
        if not isinstance(array, np.ndarray) or array.dtype not in (np.float32, np.float64):
            raise TypeError("expected NumPy array with dtype float32 or float64, shape (N, 3)")
        if array.ndim != 2:
            raise TypeError("expected NumPy array with dtype float32 or float64, shape (N, 3)")
        if not array.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous (row-major). Use numpy.ascontiguousarray(arr) to convert.")
        if array.shape[1] != 3:
            raise ValueError("expected shape (N, 3)")
        a = array.astype(np.float32, copy=False)
        return PointCloud._from_xyz(*_soa(a))

    def _normals_soa(self):
        """nx, ny, nz as contiguous arrays, split once per normals array (a 1 M-point split costs more than an ICP setup)."""
        if self._nsoa is None or self._nsoa[0] is not self.normals:
            self._nsoa = (self.normals, _soa(np.asarray(self.normals, np.float32).reshape(-1, 3)))
        return self._nsoa[1]

    def to_numpy(self) -> np.ndarray:
        return np.stack([self.x, self.y, self.z], axis=1) if len(self.x) else np.zeros((0, 3), np.float32)

    def normals_to_numpy(self) -> Optional[np.ndarray]:
        """Superset of the reference surface (it has no accessor for normals)."""
        return None if self.normals is None else self.normals.copy()

    def len(self) -> int:
        return int(len(self.x))

    def is_empty(self) -> bool:
        return len(self.x) == 0

    def __len__(self) -> int:
        return int(len(self.x))

    def __repr__(self) -> str:
        return f"PointCloud(n={len(self.x)})"

    def select(self, indices: Sequence[int]) -> "PointCloud":
        idx = np.asarray(indices, dtype=np.int64).reshape(-1)
        n = len(self.x)
        bad = idx[(idx >= n) | (idx < 0)]
        if len(bad):
            raise IndexError(f"index {int(bad[0])} out of bounds for cloud with {n} points")
        nr = None if self.normals is None else self.normals[idx]
        return PointCloud._from_xyz(self.x[idx], self.y[idx], self.z[idx], nr)

    def select_inverse(self, indices: Sequence[int]) -> "PointCloud":
        idx = np.asarray(indices, dtype=np.int64).reshape(-1)
        n = len(self.x)
        bad = idx[(idx >= n) | (idx < 0)]
        if len(bad):
            raise IndexError(f"index {int(bad[0])} out of bounds for cloud with {n} points")
        keep = np.ones(n, bool)
        keep[idx] = False
        return self.select(np.nonzero(keep)[0])


class KdTree:
    """Batched form of pointclouds_spatial::KdTree: a uniform-grid index resident in HBM."""

    def __init__(self, cloud: PointCloud, k_hint: int = 0, ctx: Optional[Context] = None):
        self._ctx = ctx or default_context()
        lib = _ffi.load()
        h = C.c_void_p()
        self._n = len(cloud)
        st = lib.pcr_index_build(self._ctx._h, _p(cloud.x, _ffi.f32p), _p(cloud.y, _ffi.f32p), _p(cloud.z, _ffi.f32p),
                                 self._n, k_hint, C.byref(h))
        _ffi.check(st, self._ctx._h)
        self._h = h

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _ffi.load().pcr_index_free(self._h)
                self._h = None
        except Exception:
            pass

    def len(self) -> int:
        return int(_ffi.load().pcr_index_len(self._h))

    __len__ = len

    def is_empty(self) -> bool:
        return self.len() == 0

    def info(self):
        cell = C.c_float()
        dims = (C.c_int32 * 3)()
        n_idx = C.c_size_t()
        _ffi.check(_ffi.load().pcr_index_info(self._h, C.byref(cell), dims, C.byref(n_idx)))
        return {"cell_size": cell.value, "dims": list(dims), "n_indexed": n_idx.value}

    def knn(self, queries: np.ndarray, k: int):
        """-> (idx (nq,k) u32, dist (nq,k) f32, counts (nq,) u32); rows padded with UINT32_MAX / inf."""
        q = np.ascontiguousarray(np.asarray(queries, np.float32).reshape(-1, 3))
        qx, qy, qz = _soa(q)
        nq = len(qx)
        idx = np.full((nq, max(k, 0)), 0xFFFFFFFF, np.uint32)
        dist = np.full((nq, max(k, 0)), np.inf, np.float32)
        cnt = np.zeros(nq, np.uint32)
        st = _ffi.load().pcr_knn(self._h, _p(qx, _ffi.f32p), _p(qy, _ffi.f32p), _p(qz, _ffi.f32p), nq, k,
                                 _p(idx, _ffi.u32p), _p(dist, _ffi.f32p), _p(cnt, _ffi.u32p))
        _ffi.check(st, self._ctx._h)
        return idx, dist, cnt

    def knn_indices(self, queries: np.ndarray, k: int):
        q = np.ascontiguousarray(np.asarray(queries, np.float32).reshape(-1, 3))
        qx, qy, qz = _soa(q)
        nq = len(qx)
        idx = np.full((nq, max(k, 0)), 0xFFFFFFFF, np.uint32)
        cnt = np.zeros(nq, np.uint32)
        st = _ffi.load().pcr_knn(self._h, _p(qx, _ffi.f32p), _p(qy, _ffi.f32p), _p(qz, _ffi.f32p), nq, k,
                                 _p(idx, _ffi.u32p), None, _p(cnt, _ffi.u32p))
        _ffi.check(st, self._ctx._h)
        return idx, cnt

    def radius_count(self, queries: np.ndarray, radius: float) -> np.ndarray:
        q = np.ascontiguousarray(np.asarray(queries, np.float32).reshape(-1, 3))
        qx, qy, qz = _soa(q)
        cnt = np.zeros(len(qx), np.uint32)
        st = _ffi.load().pcr_radius_count(self._h, _p(qx, _ffi.f32p), _p(qy, _ffi.f32p), _p(qz, _ffi.f32p), len(qx),
                                          float(radius), _p(cnt, _ffi.u32p))
        _ffi.check(st, self._ctx._h)
        return cnt

    def radius_search(self, queries: np.ndarray, radius: float):
        """CSR: (offsets (nq+1,) u64, idx u32) with every row ascending by index (kdtree.rs:132)."""
        q = np.ascontiguousarray(np.asarray(queries, np.float32).reshape(-1, 3))
        qx, qy, qz = _soa(q)
        nq = len(qx)
        off = np.zeros(nq + 1, np.uint64)
        total = C.c_size_t()
        cap = max(16 * nq, 1024)
        lib = _ffi.load()
        for _ in range(2):
            idx = np.empty(cap, np.uint32)
            st = lib.pcr_radius_search(self._h, _p(qx, _ffi.f32p), _p(qy, _ffi.f32p), _p(qz, _ffi.f32p), nq, float(radius),
                                       _p(off, _ffi.u64p), _p(idx, _ffi.u32p), cap, C.byref(total))
            if st == _ffi.PCR_ERR_CAPACITY:
                cap = int(total.value)
                continue
            _ffi.check(st, self._ctx._h)
            return off, idx[: total.value].copy()
        raise PcrError(_ffi.PCR_ERR_CAPACITY, "radius_search: capacity retry failed")

    def find_correspondences(self, source: PointCloud, max_distance: float = math.inf):
        ns = len(source)
        si = np.empty(max(ns, 1), np.uint32)
        ti = np.empty(max(ns, 1), np.uint32)
        dd = np.empty(max(ns, 1), np.float32)
        m = C.c_size_t()
        st = _ffi.load().pcr_find_correspondences(self._h, _p(source.x, _ffi.f32p), _p(source.y, _ffi.f32p), _p(source.z, _ffi.f32p),
                                                  ns, float(max_distance), _p(si, _ffi.u32p), _p(ti, _ffi.u32p), _p(dd, _ffi.f32p),
                                                  C.byref(m))
        _ffi.check(st, self._ctx._h)
        return si[: m.value].copy(), ti[: m.value].copy(), dd[: m.value].copy()


def find_correspondences(source: PointCloud, target_tree: KdTree, max_distance: float = math.inf):
    return target_tree.find_correspondences(source, max_distance)


# ---------------------------------------------------------------------------------------------------
# filters
# ---------------------------------------------------------------------------------------------------

def sor_mask(cloud: PointCloud, k: int, std_mul: float, ctx: Optional[Context] = None, want_mean: bool = False):
    """keep mask (u8), kept count, [mean distances], (mean, std, threshold)."""
    ctx = ctx or default_context()
    if not math.isfinite(std_mul) or std_mul < 0.0:  # crates/python/src/filters.rs:42-46
        raise ValueError("std_mul must be >= 0 and finite")
    n = len(cloud)
    keep = np.zeros(max(n, 1), np.uint8)
    kept = C.c_size_t()
    mean_d = np.empty(max(n, 1), np.float32) if want_mean else None
    stats = np.zeros(3, np.float32)
    st = _ffi.load().pcr_sor(ctx._h, _p(cloud.x, _ffi.f32p), _p(cloud.y, _ffi.f32p), _p(cloud.z, _ffi.f32p), n, k, float(std_mul),
                             _p(keep, _ffi.u8p), C.byref(kept), _p(mean_d, _ffi.f32p), _p(stats, _ffi.f32p))
    _ffi.check(st, ctx._h)
    return keep[:n], int(kept.value), (mean_d[:n] if want_mean else None), stats


def statistical_outlier_removal(cloud: PointCloud, k: int, std_mul: float, ctx: Optional[Context] = None) -> PointCloud:
    keep, _, _, _ = sor_mask(cloud, k, std_mul, ctx)
    return cloud.select(np.nonzero(keep)[0])  # statistical_outlier.rs:68


def voxel_downsample(cloud: PointCloud, voxel_size: float, ctx: Optional[Context] = None) -> PointCloud:
    """crates/python/src/filters.rs:4-13 (ValueError unless voxel_size > 0 and finite)."""
    ctx = ctx or default_context()
    if not math.isfinite(voxel_size) or voxel_size <= 0.0:
        raise ValueError("voxel_size must be > 0 and finite")
    n = len(cloud)
    ox, oy, oz = (np.zeros(max(n, 1), np.float32) for _ in range(3))
    m = C.c_size_t()
    st = _ffi.load().pcr_voxel_downsample(ctx._h, _p(cloud.x, _ffi.f32p), _p(cloud.y, _ffi.f32p), _p(cloud.z, _ffi.f32p), n,
                                          float(voxel_size), _p(ox, _ffi.f32p), _p(oy, _ffi.f32p), _p(oz, _ffi.f32p), C.byref(m))
    _ffi.check(st, ctx._h)
    k = int(m.value)
    return PointCloud._from_xyz(ox[:k].copy(), oy[:k].copy(), oz[:k].copy())


def ror_mask(cloud: PointCloud, radius: float, min_neighbors: int, ctx: Optional[Context] = None):
    ctx = ctx or default_context()
    if not math.isfinite(radius) or radius <= 0.0:  # crates/python/src/filters.rs:57-61
        raise ValueError("radius must be > 0 and finite")
    n = len(cloud)
    keep = np.zeros(max(n, 1), np.uint8)
    kept = C.c_size_t()
    st = _ffi.load().pcr_radius_outlier(ctx._h, _p(cloud.x, _ffi.f32p), _p(cloud.y, _ffi.f32p), _p(cloud.z, _ffi.f32p), n,
                                        float(radius), int(min_neighbors), _p(keep, _ffi.u8p), C.byref(kept))
    _ffi.check(st, ctx._h)
    return keep[:n], int(kept.value)


def radius_outlier_removal(cloud: PointCloud, radius: float, min_neighbors: int, ctx: Optional[Context] = None) -> PointCloud:
    keep, _ = ror_mask(cloud, radius, min_neighbors, ctx)
    return cloud.select(np.nonzero(keep)[0])


# ---------------------------------------------------------------------------------------------------
# segmentation
# ---------------------------------------------------------------------------------------------------

def euclidean_cluster(cloud: PointCloud, distance_threshold: float, min_size: int, max_size: int,
                      ctx: Optional[Context] = None) -> List[List[int]]:
    """crates/python/src/segmentation.rs:4-17 -> list of index lists (largest cluster first)."""
    ctx = ctx or default_context()
    n = len(cloud)
    off = np.zeros(n + 1, np.uint32)
    idx = np.zeros(max(n, 1), np.uint32)
    nc = C.c_size_t()
    st = _ffi.load().pcr_euclidean_cluster(ctx._h, _p(cloud.x, _ffi.f32p), _p(cloud.y, _ffi.f32p), _p(cloud.z, _ffi.f32p), n,
                                           float(distance_threshold), int(min_size), int(max_size), _p(off, _ffi.u32p),
                                           _p(idx, _ffi.u32p), C.byref(nc))
    _ffi.check(st, ctx._h)
    return [idx[off[c]:off[c + 1]].tolist() for c in range(int(nc.value))]


class PlaneResult:
    """crates/python/src/segmentation.rs:19-36."""

    def __init__(self, normal, d, inliers):
        self.normal = [float(v) for v in normal]
        self.d = float(d)
        self.inliers = inliers

    def __repr__(self) -> str:
        return f"PlaneResult(normal={self.normal}, d={self.d:.4f}, inliers={len(self.inliers)})"


def draw_plane_samples(n: int, iterations: int, seed=None) -> np.ndarray:
    """The reference's sample_three_distinct (ransac_plane.rs:140-163) with numpy's generator: same procedure,
    NOT the same stream as Rust's StdRng (ChaCha12).  A Rust host passes its own triples to the C ABI."""
    rng = np.random.default_rng(seed)
    out = []
    if n < 3:
        return np.zeros((0, 3), np.uint32)
    for _ in range(int(iterations)):
        i0 = int(rng.integers(n))
        i1, tries = int(rng.integers(n)), 0
        while i1 == i0 and tries <= 100:
            i1, tries = int(rng.integers(n)), tries + 1
        if i1 == i0:
            continue
        i2, tries = int(rng.integers(n)), 0
        while i2 in (i0, i1) and tries <= 100:
            i2, tries = int(rng.integers(n)), tries + 1
        if i2 in (i0, i1):
            continue
        out.append((i0, i1, i2))
    return np.asarray(out, np.uint32).reshape(-1, 3)


def ransac_plane_samples(cloud: PointCloud, distance_threshold: float, samples, ctx: Optional[Context] = None) -> PlaneResult:
    """ransac_plane_seeded (ransac_plane.rs:56-129) for given index triples."""
    ctx = ctx or default_context()
    n = len(cloud)
    smp = np.ascontiguousarray(np.asarray(samples, np.uint32).reshape(-1, 3))
    if len(smp) and int(smp.max()) >= n:
        raise IndexError(f"sample index {int(smp.max())} out of bounds for cloud with {n} points")
    model = np.zeros(4, np.float32)
    inl = np.zeros(max(n, 1), np.uint32)
    k = C.c_size_t()
    st = _ffi.load().pcr_ransac_plane_samples(ctx._h, _p(cloud.x, _ffi.f32p), _p(cloud.y, _ffi.f32p), _p(cloud.z, _ffi.f32p), n,
                                              float(distance_threshold), _p(smp, _ffi.u32p), len(smp), _p(model, _ffi.f32p),
                                              _p(inl, _ffi.u32p), C.byref(k))
    _ffi.check(st, ctx._h)
    return PlaneResult(model[:3], model[3], inl[:int(k.value)].tolist())


def ransac_plane(cloud: PointCloud, distance_threshold: float, iterations: int, ctx: Optional[Context] = None) -> PlaneResult:
    """crates/python/src/segmentation.rs:42-55: a random seed per call, like the reference's ransac_plane (:36-43)."""
    return ransac_plane_samples(cloud, distance_threshold, draw_plane_samples(len(cloud), iterations), ctx)


def cluster_arrays(cloud: PointCloud, distance_threshold: float, min_size: int, max_size: int, ctx: Optional[Context] = None):
    """Same call, CSR form (offsets, indices) without building Python lists."""
    ctx = ctx or default_context()
    n = len(cloud)
    off = np.zeros(n + 1, np.uint32)
    idx = np.zeros(max(n, 1), np.uint32)
    nc = C.c_size_t()
    st = _ffi.load().pcr_euclidean_cluster(ctx._h, _p(cloud.x, _ffi.f32p), _p(cloud.y, _ffi.f32p), _p(cloud.z, _ffi.f32p), n,
                                           float(distance_threshold), int(min_size), int(max_size), _p(off, _ffi.u32p),
                                           _p(idx, _ffi.u32p), C.byref(nc))
    _ffi.check(st, ctx._h)
    k = int(nc.value)
    return off[:k + 1].copy(), idx[:int(off[k])].copy()


# ---------------------------------------------------------------------------------------------------
# normals
# ---------------------------------------------------------------------------------------------------

def normals_array(cloud: PointCloud, k: int, viewpoint=(0.0, 0.0, 0.0), ctx: Optional[Context] = None) -> np.ndarray:
    """estimate_normals_with_viewpoint -> (N,3) f32 (empty if the cloud is empty or k == 0)."""
    ctx = ctx or default_context()
    n = len(cloud)
    if n == 0 or k == 0:
        return np.zeros((0, 3), np.float32)
    vp = np.asarray(viewpoint, np.float32).reshape(3)
    nx = np.empty(n, np.float32)
    ny = np.empty(n, np.float32)
    nz = np.empty(n, np.float32)
    st = _ffi.load().pcr_estimate_normals(ctx._h, _p(cloud.x, _ffi.f32p), _p(cloud.y, _ffi.f32p), _p(cloud.z, _ffi.f32p), n, k,
                                          _p(vp, _ffi.f32p), _p(nx, _ffi.f32p), _p(ny, _ffi.f32p), _p(nz, _ffi.f32p))
    _ffi.check(st, ctx._h)
    return np.stack([nx, ny, nz], axis=1)


def estimate_normals(cloud: PointCloud, k: int, ctx: Optional[Context] = None) -> PointCloud:
    """Returns a copy of the cloud with normals attached (crates/python/src/normals.rs:4-10)."""
    nr = normals_array(cloud, k, (0.0, 0.0, 0.0), ctx)
    return PointCloud._from_xyz(cloud.x.copy(), cloud.y.copy(), cloud.z.copy(), nr)


# ---------------------------------------------------------------------------------------------------
# registration
# ---------------------------------------------------------------------------------------------------

class IcpResult:
    def __init__(self, r: _ffi.IcpResultC):
        self.converged = bool(r.converged)
        self.fitness = float(np.float32(r.fitness))
        self.rmse = float(np.float32(r.rmse))
        self.num_iterations = int(r.num_iterations)
        self.translation = [float(v) for v in r.translation]
        rot = [float(v) for v in r.rotation]
        self.rotation = [rot[0:3], rot[3:6], rot[6:9]]

    def __repr__(self) -> str:
        return f"IcpResult(converged={str(self.converged).lower()}, rmse={self.rmse:.6f}, iterations={self.num_iterations})"


def _icp_params(max_iterations, tolerance, max_correspondence_distance):
    # crates/python/src/registration.rs:67-72,85
    if math.isnan(tolerance) or tolerance < 0:
        raise ValueError("tolerance must be >= 0")
    if math.isnan(max_correspondence_distance) or max_correspondence_distance < 0:
        raise ValueError("max_correspondence_distance must be >= 0")
    return _ffi.IcpParams(int(max_iterations), float(tolerance), float(max_correspondence_distance))


def icp_point_to_point(source: PointCloud, target: PointCloud, max_iterations: int = 50, tolerance: float = 1e-5,
                       max_correspondence_distance: float = math.inf, ctx: Optional[Context] = None) -> IcpResult:
    ctx = ctx or default_context()
    p = _icp_params(max_iterations, tolerance, max_correspondence_distance)
    res = _ffi.IcpResultC()
    st = _ffi.load().pcr_icp_point_to_point(ctx._h, _p(source.x, _ffi.f32p), _p(source.y, _ffi.f32p), _p(source.z, _ffi.f32p),
                                            len(source), _p(target.x, _ffi.f32p), _p(target.y, _ffi.f32p), _p(target.z, _ffi.f32p),
                                            len(target), C.byref(p), C.byref(res))
    _ffi.check(st, ctx._h)
    return IcpResult(res)


def icp_point_to_plane(source: PointCloud, target: PointCloud, max_iterations: int = 50, tolerance: float = 1e-5,
                       max_correspondence_distance: float = math.inf, ctx: Optional[Context] = None) -> IcpResult:
    ctx = ctx or default_context()
    if target.normals is None:  # crates/python/src/registration.rs:66-71
        raise ValueError("target cloud must have normals for point-to-plane ICP. Use estimate_normals(target, k) first.")
    p = _icp_params(max_iterations, tolerance, max_correspondence_distance)
    nx, ny, nz = target._normals_soa()
    res = _ffi.IcpResultC()
    st = _ffi.load().pcr_icp_point_to_plane(ctx._h, _p(source.x, _ffi.f32p), _p(source.y, _ffi.f32p), _p(source.z, _ffi.f32p),
                                            len(source), _p(target.x, _ffi.f32p), _p(target.y, _ffi.f32p), _p(target.z, _ffi.f32p),
                                            len(target), _p(nx, _ffi.f32p), _p(ny, _ffi.f32p), _p(nz, _ffi.f32p), len(nx),
                                            C.byref(p), C.byref(res))
    _ffi.check(st, ctx._h)
    return IcpResult(res)


def apply_transform(cloud: PointCloud, rotation, translation, ctx: Optional[Context] = None) -> PointCloud:
    """R*p + t for every point; the result carries xyz only (icp.rs:77-92)."""
    ctx = ctx or default_context()
    n = len(cloud)
    r = np.ascontiguousarray(np.asarray(rotation, np.float32).reshape(9))
    t = np.ascontiguousarray(np.asarray(translation, np.float32).reshape(3))
    ox = np.empty(n, np.float32)
    oy = np.empty(n, np.float32)
    oz = np.empty(n, np.float32)
    st = _ffi.load().pcr_apply_transform(ctx._h, _p(cloud.x, _ffi.f32p), _p(cloud.y, _ffi.f32p), _p(cloud.z, _ffi.f32p), n,
                                         _p(r, _ffi.f32p), _p(t, _ffi.f32p), _p(ox, _ffi.f32p), _p(oy, _ffi.f32p), _p(oz, _ffi.f32p))
    _ffi.check(st, ctx._h)
    return PointCloud._from_xyz(ox, oy, oz)


def _batch_frames(points, frame_offsets):
    """Checks and converts the frame buffer of a batch call: (N,3) f32 rows, frames back to back, u64 offsets."""
    pts = np.asarray(points)
    if pts.ndim != 2 or pts.shape[1] != 3:
        raise ValueError("points must have shape (N, 3)")
    n = len(pts)
    off = np.asarray(frame_offsets).reshape(-1)
    if len(off) == 0 or off.dtype.kind not in "iu":
        raise ValueError("frame_offsets must be n_frames + 1 integers")
    if off[0] != 0 or off[-1] != n or np.any(np.diff(off) < 0):
        raise ValueError(f"frame_offsets must be non-decreasing from 0 to the number of points ({n})")
    return np.ascontiguousarray(pts, np.float32), np.ascontiguousarray(off, np.uint64)


def _frame_transforms(transforms, n_frames: int) -> np.ndarray:
    """Checks and converts one rigid transform per frame -> (F, 12) f32 rows: row-major rotation, then translation.
    (F, 3, 4) is read as [R | t] per frame."""
    t = np.asarray(transforms)
    if t.ndim == 3 and t.shape[1:] == (3, 4):
        t = np.concatenate([t[:, :, :3].reshape(-1, 9), t[:, :, 3]], axis=1)
    if t.ndim != 2 or t.shape[1] != 12 or t.dtype.kind not in "iuf":
        raise ValueError(f"transforms must have shape (F, 12) or (F, 3, 4); got {t.shape}")
    if len(t) != n_frames:
        raise ValueError(f"expected one transform per frame ({n_frames} frames), got {len(t)}")
    return np.ascontiguousarray(t, np.float32)


def _transform12(rotation, translation) -> np.ndarray:
    return np.concatenate([np.asarray(rotation, np.float32).reshape(9), np.asarray(translation, np.float32).reshape(3)])


def compose(first, then):
    """RigidTransform::compose (icp.rs:52-73): the transform that applies `first`, then `then`.  Args: (R, t) pairs;
    -> (R (3,3) f32, t (3,) f32) with R = then.R @ first.R and t = then.R @ first.t + then.t, in the reference's f32
    operation order (no FMA)."""
    a, b, out = _transform12(*first), _transform12(*then), np.empty(12, np.float32)
    _ffi.check(_ffi.load().pcr_transform_compose(_p(a, _ffi.f32p), _p(b, _ffi.f32p), _p(out, _ffi.f32p)))
    return out[:9].reshape(3, 3), out[9:].copy()


def chain_poses(relative) -> np.ndarray:
    """Poses of an odometry chain -> (n + 1, 12) f32, the layout apply_transform_batch takes.  `relative`: the n
    IcpResults of the CONSECUTIVE pairs (i + 1, i) in order (relative[i] takes frame i + 1 into frame i's coordinates),
    or their transforms as apply_transform_batch takes them: (n, 12) rows (row-major R, then t) or (n, 3, 4) [R | t].
    pose[0] is the identity and pose[i + 1] = compose(relative[i], pose[i]): the transform that takes frame i + 1 into
    frame 0's coordinates.  Other pairings are not chains and give meaningless poses."""
    if isinstance(relative, np.ndarray):
        rel = relative
    else:
        rel = [_transform12(r.rotation, r.translation) if isinstance(r, IcpResult) else r for r in relative]
        rel = np.asarray(rel) if rel else np.zeros((0, 12), np.float32)
    rel = _frame_transforms(rel, len(rel) if rel.ndim else 0)
    poses = np.zeros((len(rel) + 1, 12), np.float32)
    poses[0, [0, 4, 8]] = 1.0
    lib = _ffi.load()
    for i in range(len(rel)):
        _ffi.check(lib.pcr_transform_compose(_p(rel[i], _ffi.f32p), _p(poses[i], _ffi.f32p), _p(poses[i + 1], _ffi.f32p)))
    return poses


def apply_transform_batch(points: np.ndarray, frame_offsets: Sequence[int], transforms, ctx: Optional[Context] = None) -> np.ndarray:
    """apply_transform of every frame of a batch in one call.  points: (N,3), frame f = rows [frame_offsets[f],
    frame_offsets[f+1]); transforms: (F, 12) (row-major R, then t) or (F, 3, 4) [R | t], one per frame.  -> (N,3) f32,
    frame f's rows bit for bit what apply_transform returns for the frame alone with transform f."""
    pts, off = _batch_frames(points, frame_offsets)
    tr = _frame_transforms(transforms, len(off) - 1)
    ctx = ctx or default_context()
    x, y, z = _soa(pts)
    n = len(pts)
    ox, oy, oz = (np.empty(max(n, 1), np.float32) for _ in range(3))
    st = _ffi.load().pcr_apply_transform_batch(ctx._h, _p(x, _ffi.f32p), _p(y, _ffi.f32p), _p(z, _ffi.f32p), _p(off, _ffi.u64p), len(off) - 1,
                                               _p(tr, _ffi.f32p), _p(ox, _ffi.f32p), _p(oy, _ffi.f32p), _p(oz, _ffi.f32p))
    _ffi.check(st, ctx._h)
    return np.stack([ox[:n], oy[:n], oz[:n]], axis=1)


def _icp_batch_arrays(points, frame_offsets, pairs):
    """Checks and converts the frame buffer of a batched ICP: (N,3) f32 rows, u64 offsets, (P,2) u32 pairs."""
    pts, off = _batch_frames(points, frame_offsets)
    nf = len(off) - 1
    pr = np.asarray(pairs)
    if pr.size == 0:
        pr = pr.reshape(0, 2)
    if pr.ndim != 2 or pr.shape[1] != 2 or (len(pr) and pr.dtype.kind not in "iu"):
        raise ValueError("pairs must be an integer array of shape (P, 2): (source frame, target frame)")
    if len(pr) and (pr.min() < 0 or pr.max() >= nf):
        raise ValueError(f"pairs hold a frame id outside [0, {nf})")
    return pts, off, np.ascontiguousarray(pr, np.uint32)


def icp_point_to_point_batch(points: np.ndarray, frame_offsets: Sequence[int], pairs, max_iterations: int = 50,
                             tolerance: float = 1e-5, max_correspondence_distance: float = math.inf,
                             ctx: Optional[Context] = None) -> List[IcpResult]:
    """Point-to-point ICP of many frame pairs in one call.  points: (N,3), every frame back to back, frame f = rows
    [frame_offsets[f], frame_offsets[f+1]); pairs: (P,2), pair p registers frame pairs[p][0] (source) onto frame
    pairs[p][1] (target).  -> one IcpResult per pair, each what icp_point_to_point returns for those two clouds."""
    p = _icp_params(max_iterations, tolerance, max_correspondence_distance)
    pts, off, pr = _icp_batch_arrays(points, frame_offsets, pairs)
    ctx = ctx or default_context()
    x, y, z = _soa(pts)
    res = (_ffi.IcpResultC * max(len(pr), 1))()
    st = _ffi.load().pcr_icp_point_to_point_batch(ctx._h, _p(x, _ffi.f32p), _p(y, _ffi.f32p), _p(z, _ffi.f32p), _p(off, _ffi.u64p),
                                                  len(off) - 1, _p(pr, _ffi.u32p), len(pr), C.byref(p), res)
    _ffi.check(st, ctx._h)
    return [IcpResult(res[i]) for i in range(len(pr))]


def icp_point_to_plane_batch(points: np.ndarray, frame_offsets: Sequence[int], pairs, normals: Optional[np.ndarray],
                             max_iterations: int = 50, tolerance: float = 1e-5, max_correspondence_distance: float = math.inf,
                             ctx: Optional[Context] = None) -> List[IcpResult]:
    """Point-to-plane form of icp_point_to_point_batch.  normals: (N,3), one per row of `points` (only the rows of
    target frames are read)."""
    if normals is None:  # crates/python/src/registration.rs:66-71
        raise ValueError("point-to-plane ICP needs the targets' normals. Use estimate_normals first.")
    p = _icp_params(max_iterations, tolerance, max_correspondence_distance)
    pts, off, pr = _icp_batch_arrays(points, frame_offsets, pairs)
    nrm = np.asarray(normals)
    if nrm.ndim != 2 or nrm.shape[1] != 3 or len(nrm) != len(pts):
        raise ValueError(f"normals must have shape ({len(pts)}, 3), one per point; got {nrm.shape}")
    ctx = ctx or default_context()
    x, y, z = _soa(pts)
    nx, ny, nz = _soa(np.ascontiguousarray(nrm, np.float32))
    res = (_ffi.IcpResultC * max(len(pr), 1))()
    st = _ffi.load().pcr_icp_point_to_plane_batch(ctx._h, _p(x, _ffi.f32p), _p(y, _ffi.f32p), _p(z, _ffi.f32p), _p(off, _ffi.u64p),
                                                  len(off) - 1, _p(nx, _ffi.f32p), _p(ny, _ffi.f32p), _p(nz, _ffi.f32p), len(nx),
                                                  _p(pr, _ffi.u32p), len(pr), C.byref(p), res)
    _ffi.check(st, ctx._h)
    return [IcpResult(res[i]) for i in range(len(pr))]



# ---------------------------------------------------------------------------------------------------
# device-resident clouds (superset of the reference surface: the same calls without the PCIe round
# trips between the steps of a pipeline)
# ---------------------------------------------------------------------------------------------------

class DeviceCloud:
    """A PointCloud that lives in HBM.  Every filter returns a new DeviceCloud; nothing crosses PCIe
    until to_numpy() / normals_to_numpy() / the cluster index lists / the ICP result."""

    def __init__(self, handle, ctx: Context):
        self._h = handle
        self._ctx = ctx
        ctx._clouds.add(self)

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    @staticmethod
    def from_numpy(array, ctx: Optional[Context] = None) -> "DeviceCloud":
        """(N, 3) float32 / float64, C-contiguous (crates/python/src/cloud.rs:25-37).  A float32 array crosses PCIe as it is
        and is split into SoA on the device (pcr_cloud_upload_rows): splitting 122 K points with numpy costs more than the
        whole voxel -> SOR -> normals pipeline."""
        if isinstance(array, np.ndarray) and array.dtype == np.float32 and array.ndim == 2 and array.shape[1] == 3 and array.flags["C_CONTIGUOUS"]:
            ctx = ctx or default_context()
            h = C.c_void_p()
            _ffi.check(_ffi.load().pcr_cloud_upload_rows(ctx._h, array.ctypes.data, len(array), C.byref(h)), ctx._h)
            return DeviceCloud(h, ctx)
        return DeviceCloud.from_cloud(PointCloud.from_numpy(array), ctx)  # (same checks and errors as the host class)

    @staticmethod
    def from_cloud(cloud: PointCloud, ctx: Optional[Context] = None) -> "DeviceCloud":
        ctx = ctx or default_context()
        h = C.c_void_p()
        st = _ffi.load().pcr_cloud_upload(ctx._h, cloud.x.ctypes.data, cloud.y.ctypes.data, cloud.z.ctypes.data, len(cloud), C.byref(h))
        _ffi.check(st, ctx._h)
        return DeviceCloud(h, ctx)

    @staticmethod
    def upload_raw(ctx: Context, x_ptr: int, y_ptr: int, z_ptr: int, n: int) -> "DeviceCloud":
        """Upload from raw host addresses (e.g. pinned buffers)."""
        h = C.c_void_p()
        _ffi.check(_ffi.load().pcr_cloud_upload(ctx._h, x_ptr, y_ptr, z_ptr, n, C.byref(h)), ctx._h)
        return DeviceCloud(h, ctx)

    @staticmethod
    def upload_block(ctx: Context, ptr: int, stride: int, n: int, wait: bool = True) -> "DeviceCloud":
        """Upload x | y | z from ONE host block (rows `stride` floats apart): a single strided transfer.
        wait=False does not wait for the copy (pinned block, left unchanged until a result that depends on the
        cloud has come back): the next steps queue right behind it."""
        h = C.c_void_p()
        lib = _ffi.load()
        fn = lib.pcr_cloud_upload_block if wait else lib.pcr_cloud_upload_block_nowait
        _ffi.check(fn(ctx._h, ptr, stride, n, C.byref(h)), ctx._h)
        return DeviceCloud(h, ctx)

    def download_block(self, ptr: int, stride: int, with_normals: bool = False):
        """Download x | y | z [| nx | ny | nz] into ONE host block (rows `stride` floats apart)."""
        _ffi.check(_ffi.load().pcr_cloud_download_block(self._h, ptr, stride, 1 if with_normals else 0), self._ctx._h)

    def download_raw(self, x_ptr: int, y_ptr: int, z_ptr: int, nx_ptr: int = 0, ny_ptr: int = 0, nz_ptr: int = 0):
        """Download into raw host addresses (arrays of len()); normals too if the three pointers are given."""
        _ffi.check(_ffi.load().pcr_cloud_download(self._h, x_ptr, y_ptr, z_ptr), self._ctx._h)
        if nx_ptr:
            _ffi.check(_ffi.load().pcr_cloud_download_normals(self._h, nx_ptr, ny_ptr, nz_ptr), self._ctx._h)

    def free(self):
        h, self._h = getattr(self, "_h", None), None
        if h and self._ctx._h:  # a closed context has already freed its clouds
            _ffi.load().pcr_cloud_free(h)

    def _new(self, fn, *args) -> "DeviceCloud":
        h = C.c_void_p()
        _ffi.check(fn(self._h, *args, C.byref(h)), self._ctx._h)
        return DeviceCloud(h, self._ctx)

    def len(self) -> int:
        return int(_ffi.load().pcr_cloud_len(self._h))

    __len__ = len

    def is_empty(self) -> bool:
        return self.len() == 0

    def has_normals(self) -> bool:
        return bool(_ffi.load().pcr_cloud_has_normals(self._h))

    def __repr__(self) -> str:
        return f"DeviceCloud(n={self.len()}, normals={self.has_normals()})"

    def to_numpy(self) -> np.ndarray:
        out = np.empty((self.len(), 3), np.float32)  # (interleaved on the device: one contiguous transfer)
        _ffi.check(_ffi.load().pcr_cloud_download_rows(self._h, out.ctypes.data, None), self._ctx._h)
        return out

    def normals_to_numpy(self) -> Optional[np.ndarray]:
        if not self.has_normals():
            return None
        out = np.empty((self.len(), 3), np.float32)
        _ffi.check(_ffi.load().pcr_cloud_download_rows(self._h, None, out.ctypes.data), self._ctx._h)
        return out

    def to_cloud(self) -> PointCloud:
        a = self.to_numpy()
        return PointCloud._from_xyz(*_soa(a), self.normals_to_numpy())

    def select(self, indices: Sequence[int]) -> "DeviceCloud":
        idx = np.asarray(indices, dtype=np.int64).reshape(-1)
        n = self.len()
        bad = idx[(idx >= n) | (idx < 0)]
        if len(bad):
            raise IndexError(f"index {int(bad[0])} out of bounds for cloud with {n} points")
        i32 = np.ascontiguousarray(idx, np.uint32)
        return self._new(_ffi.load().pcr_cloud_select, _p(i32, _ffi.u32p), len(i32))

    def voxel_downsample(self, voxel_size: float) -> "DeviceCloud":
        if not math.isfinite(voxel_size) or voxel_size <= 0.0:
            raise ValueError("voxel_size must be > 0 and finite")
        return self._new(_ffi.load().pcr_cloud_voxel_downsample, float(voxel_size))

    def statistical_outlier_removal(self, k: int, std_mul: float) -> "DeviceCloud":
        if not math.isfinite(std_mul) or std_mul < 0.0:  # crates/python/src/filters.rs:42-46
            raise ValueError("std_mul must be >= 0 and finite")
        return self._new(_ffi.load().pcr_cloud_statistical_outlier_removal, int(k), float(std_mul))

    def radius_outlier_removal(self, radius: float, min_neighbors: int) -> "DeviceCloud":
        if not math.isfinite(radius) or radius <= 0.0:
            raise ValueError("radius must be > 0 and finite")
        return self._new(_ffi.load().pcr_cloud_radius_outlier_removal, float(radius), int(min_neighbors))

    def estimate_normals(self, k: int, viewpoint=(0.0, 0.0, 0.0)) -> "DeviceCloud":
        vp = np.asarray(viewpoint, np.float32)
        return self._new(_ffi.load().pcr_cloud_estimate_normals, int(k), _p(vp, _ffi.f32p))

    def sor_normals(self, k_sor: int, std_mul: float, k_normals: int, viewpoint=(0.0, 0.0, 0.0)) -> "DeviceCloud":
        """statistical_outlier_removal(k_sor, std_mul) then estimate_normals(k_normals) on the kept points, one index."""
        vp = np.asarray(viewpoint, np.float32)
        return self._new(_ffi.load().pcr_cloud_sor_normals, int(k_sor), float(std_mul), int(k_normals), _p(vp, _ffi.f32p))

    def euclidean_cluster(self, distance_threshold: float, min_size: int, max_size: int) -> List[List[int]]:
        n = self.len()
        off = np.zeros(n + 1, np.uint32)
        idx = np.zeros(max(n, 1), np.uint32)
        nc = C.c_size_t()
        st = _ffi.load().pcr_cloud_euclidean_cluster(self._h, float(distance_threshold), int(min_size), int(max_size), _p(off, _ffi.u32p),
                                                     _p(idx, _ffi.u32p), C.byref(nc))
        _ffi.check(st, self._ctx._h)
        return [idx[off[c]:off[c + 1]].tolist() for c in range(int(nc.value))]

    def ransac_plane_samples(self, distance_threshold: float, samples) -> "PlaneResult":
        n = self.len()
        smp = np.ascontiguousarray(np.asarray(samples, np.uint32).reshape(-1, 3))
        if len(smp) and int(smp.max()) >= n:
            raise IndexError(f"sample index {int(smp.max())} out of bounds for cloud with {n} points")
        model = np.zeros(4, np.float32)
        inl = np.zeros(max(n, 1), np.uint32)
        k = C.c_size_t()
        st = _ffi.load().pcr_cloud_ransac_plane_samples(self._h, float(distance_threshold), _p(smp, _ffi.u32p), len(smp),
                                                        _p(model, _ffi.f32p), _p(inl, _ffi.u32p), C.byref(k))
        _ffi.check(st, self._ctx._h)
        return PlaneResult(model[:3], model[3], inl[:int(k.value)].tolist())

    def ransac_plane(self, distance_threshold: float, iterations: int) -> "PlaneResult":
        return self.ransac_plane_samples(distance_threshold, draw_plane_samples(self.len(), iterations))

    def apply_transform(self, rotation, translation) -> "DeviceCloud":
        r = np.ascontiguousarray(np.asarray(rotation, np.float32).reshape(9))
        t = np.ascontiguousarray(np.asarray(translation, np.float32).reshape(3))
        return self._new(_ffi.load().pcr_cloud_apply_transform, _p(r, _ffi.f32p), _p(t, _ffi.f32p))

    def icp_point_to_point(self, target: "DeviceCloud", max_iterations: int = 50, tolerance: float = 1e-5,
                           max_correspondence_distance: float = math.inf) -> "IcpResult":
        prm = _icp_params(max_iterations, tolerance, max_correspondence_distance)
        res = _ffi.IcpResultC()
        _ffi.check(_ffi.load().pcr_cloud_icp_point_to_point(self._h, target._h, C.byref(prm), C.byref(res)), self._ctx._h)
        return IcpResult(res)

    def icp_point_to_plane(self, target: "DeviceCloud", max_iterations: int = 50, tolerance: float = 1e-5,
                           max_correspondence_distance: float = math.inf) -> "IcpResult":
        prm = _icp_params(max_iterations, tolerance, max_correspondence_distance)
        res = _ffi.IcpResultC()
        _ffi.check(_ffi.load().pcr_cloud_icp_point_to_plane(self._h, target._h, C.byref(prm), C.byref(res)), self._ctx._h)
        return IcpResult(res)

# ---------------------------------------------------------------------------------------------------
# multi-frame batch (BASELINE config 5)
# ---------------------------------------------------------------------------------------------------

def sor_normals_batch(points: np.ndarray, frame_offsets: Sequence[int], k_sor: int, std_mul: float, k_normals: int,
                      viewpoint=(0.0, 0.0, 0.0), ctx: Optional[Context] = None):
    """points: (N,3) f32 of all frames back to back. -> (keep u8 (N,), normals (N,3), kept per frame)."""
    ctx = ctx or default_context()
    pts = np.ascontiguousarray(np.asarray(points, np.float32).reshape(-1, 3))
    off = np.ascontiguousarray(np.asarray(frame_offsets, np.uint64))
    nf = len(off) - 1
    n = len(pts)
    vp = np.asarray(viewpoint, np.float32).reshape(3)
    keep = np.empty(max(n, 1), np.uint8)            # (every entry is written: removed points get keep 0 and a zero normal)
    nrm = np.empty((max(n, 1), 3), np.float32) if k_normals else np.zeros((max(n, 1), 3), np.float32)
    kept = np.zeros(max(nf, 1), np.uint64)
    # the rows go to the device as they are (pcr_sor_normals_batch_rows): numpy's split of 8 M points into SoA and back
    # cost 90 of the 103 ms this call took, the work itself 11
    st = _ffi.load().pcr_sor_normals_batch_rows(ctx._h, _p(pts, _ffi.f32p), _p(off, _ffi.u64p), nf, k_sor, float(std_mul), k_normals,
                                                _p(vp, _ffi.f32p), _p(keep, _ffi.u8p), _p(nrm, _ffi.f32p), _p(kept, _ffi.u64p))
    _ffi.check(st, ctx._h)
    return keep[:n], nrm[:n], kept[:nf]


def voxel_downsample_batch(points: np.ndarray, frame_offsets: Sequence[int], voxel_size: float, ctx: Optional[Context] = None):
    """voxel_downsample of every frame of a batch in one call.  points: (N,3), frame f = rows [frame_offsets[f],
    frame_offsets[f+1]).  -> (voxels (M,3) f32, offsets (F+1,) u64): frame f's voxels are rows [offsets[f], offsets[f+1]),
    bit for bit what voxel_downsample returns for the frame alone; the offsets can be passed to the other batch calls."""
    pts, off = _batch_frames(points, frame_offsets)
    if not math.isfinite(voxel_size) or voxel_size <= 0.0:
        raise ValueError("voxel_size must be > 0 and finite")
    ctx = ctx or default_context()
    x, y, z = _soa(pts)
    n = len(pts)
    ox, oy, oz = (np.zeros(max(n, 1), np.float32) for _ in range(3))
    out_off = np.zeros(len(off), np.uint64)
    st = _ffi.load().pcr_voxel_downsample_batch(ctx._h, _p(x, _ffi.f32p), _p(y, _ffi.f32p), _p(z, _ffi.f32p), _p(off, _ffi.u64p), len(off) - 1,
                                                float(voxel_size), _p(ox, _ffi.f32p), _p(oy, _ffi.f32p), _p(oz, _ffi.f32p), _p(out_off, _ffi.u64p))
    _ffi.check(st, ctx._h)
    m = int(out_off[-1])
    return np.stack([ox[:m], oy[:m], oz[:m]], axis=1), out_off


def estimate_normals_batch(points: np.ndarray, frame_offsets: Sequence[int], k: int, viewpoint=(0.0, 0.0, 0.0),
                           ctx: Optional[Context] = None) -> np.ndarray:
    """estimate_normals_with_viewpoint of every frame of a batch in one call, each frame searched only within itself.
    -> (N,3) f32, frame f's rows bit for bit what normals_array returns for the frame alone ((0,3) if k == 0)."""
    pts, off = _batch_frames(points, frame_offsets)
    ctx = ctx or default_context()
    n = len(pts)
    if n == 0 or k == 0:
        return np.zeros((0, 3), np.float32)
    vp = np.asarray(viewpoint, np.float32).reshape(3)
    x, y, z = _soa(pts)
    nx, ny, nz = (np.empty(n, np.float32) for _ in range(3))
    st = _ffi.load().pcr_estimate_normals_batch(ctx._h, _p(x, _ffi.f32p), _p(y, _ffi.f32p), _p(z, _ffi.f32p), _p(off, _ffi.u64p), len(off) - 1,
                                                k, _p(vp, _ffi.f32p), _p(nx, _ffi.f32p), _p(ny, _ffi.f32p), _p(nz, _ffi.f32p))
    _ffi.check(st, ctx._h)
    return np.stack([nx, ny, nz], axis=1)


def _frame_samples(samples, off):
    """Checks and stacks the per-frame triples of a batched RANSAC: one (m_f, 3) integer array of frame-LOCAL indices per
    frame -> (triples (M, 3) u32, sample offsets (F+1,) u64)."""
    nf = len(off) - 1
    if isinstance(samples, (str, bytes)) or not hasattr(samples, "__len__") or len(samples) != nf:
        raise ValueError(f"samples must hold one (m, 3) array of triples per frame ({nf} frames)")
    parts, s_off = [], np.zeros(nf + 1, np.uint64)
    for f, smp in enumerate(samples):
        a = np.asarray(smp)
        if a.size == 0:
            a = a.reshape(0, 3)
        if a.ndim != 2 or a.shape[1] != 3 or (len(a) and a.dtype.kind not in "iu"):
            raise ValueError(f"samples[{f}] must be an integer array of shape (m, 3)")
        n_f = int(off[f + 1] - off[f])
        if len(a) and (int(a.min()) < 0 or int(a.max()) >= n_f):
            bad = int(a.min()) if int(a.min()) < 0 else int(a.max())
            raise IndexError(f"frame {f}: sample index {bad} out of bounds for a frame with {n_f} points")
        parts.append(a.astype(np.uint32))
        s_off[f + 1] = s_off[f] + len(a)
    smp = np.ascontiguousarray(np.vstack(parts) if parts else np.zeros((0, 3), np.uint32), np.uint32)
    return smp, s_off


def ransac_plane_samples_batch(points: np.ndarray, frame_offsets: Sequence[int], distance_threshold: float, samples,
                               ctx: Optional[Context] = None):
    """ransac_plane_samples of every frame of a batch in one call.  points: (N,3), frame f = rows [frame_offsets[f],
    frame_offsets[f+1]); samples: one (m_f, 3) array of frame-local index triples per frame.  -> (models (F,4) f32
    [nx, ny, nz, d], inliers u32, inlier_offsets (F+1,) u64): frame f's model and its ascending frame-local inliers
    inliers[inlier_offsets[f]:inlier_offsets[f+1]] are bit for bit what ransac_plane_samples returns for the frame alone."""
    pts, off = _batch_frames(points, frame_offsets)
    smp, s_off = _frame_samples(samples, off)
    ctx = ctx or default_context()
    x, y, z = _soa(pts)
    n, nf = len(pts), len(off) - 1
    models = np.zeros((max(nf, 1), 4), np.float32)
    inl = np.zeros(max(n, 1), np.uint32)
    inl_off = np.zeros(nf + 1, np.uint64)
    st = _ffi.load().pcr_ransac_plane_samples_batch(ctx._h, _p(x, _ffi.f32p), _p(y, _ffi.f32p), _p(z, _ffi.f32p), _p(off, _ffi.u64p), nf,
                                                    float(distance_threshold), _p(smp, _ffi.u32p), _p(s_off, _ffi.u64p),
                                                    _p(models, _ffi.f32p), _p(inl, _ffi.u32p), _p(inl_off, _ffi.u64p))
    _ffi.check(st, ctx._h)
    return models[:nf], inl[:int(inl_off[-1])].copy(), inl_off


def ransac_plane_batch(points: np.ndarray, frame_offsets: Sequence[int], distance_threshold: float, iterations: int, seed=None,
                       ctx: Optional[Context] = None):
    """ransac_plane of every frame of a batch: frame f's triples are draw_plane_samples(n_f, iterations, [seed, f]) (a
    fresh random draw per frame when seed is None).  -> as ransac_plane_samples_batch."""
    _, off = _batch_frames(points, frame_offsets)
    samples = [draw_plane_samples(int(off[f + 1] - off[f]), iterations, None if seed is None else [seed, f]) for f in range(len(off) - 1)]
    return ransac_plane_samples_batch(points, off, distance_threshold, samples, ctx)


def cluster_arrays_batch(points: np.ndarray, frame_offsets: Sequence[int], distance_threshold: float, min_size: int, max_size: int,
                         ctx: Optional[Context] = None):
    """euclidean_cluster of every frame of a batch in one call, CSR form.  -> (cluster_offsets (F+1,) u64, offsets u32,
    indices u32): frame f's clusters are c in [cluster_offsets[f], cluster_offsets[f+1]), cluster c is the frame-local
    indices[offsets[c]:offsets[c+1]], in the order cluster_arrays returns for the frame alone."""
    pts, off = _batch_frames(points, frame_offsets)
    ctx = ctx or default_context()
    x, y, z = _soa(pts)
    n, nf = len(pts), len(off) - 1
    offsets = np.zeros(n + 1, np.uint32)
    idx = np.zeros(max(n, 1), np.uint32)
    c_off = np.zeros(nf + 1, np.uint64)
    st = _ffi.load().pcr_euclidean_cluster_batch(ctx._h, _p(x, _ffi.f32p), _p(y, _ffi.f32p), _p(z, _ffi.f32p), _p(off, _ffi.u64p), nf,
                                                 float(distance_threshold), int(min_size), int(max_size), _p(offsets, _ffi.u32p),
                                                 _p(idx, _ffi.u32p), _p(c_off, _ffi.u64p))
    _ffi.check(st, ctx._h)
    k = int(c_off[-1])
    return c_off, offsets[:k + 1].copy(), idx[:int(offsets[k])].copy()


def euclidean_cluster_batch(points: np.ndarray, frame_offsets: Sequence[int], distance_threshold: float, min_size: int, max_size: int,
                            ctx: Optional[Context] = None) -> List[List[List[int]]]:
    """-> one list of index lists per frame, each what euclidean_cluster returns for the frame alone."""
    c_off, offsets, idx = cluster_arrays_batch(points, frame_offsets, distance_threshold, min_size, max_size, ctx)
    return [[idx[offsets[c]:offsets[c + 1]].tolist() for c in range(int(c_off[f]), int(c_off[f + 1]))] for f in range(len(c_off) - 1)]


def sor_normals_batch_raw(ctx: Context, x, y, z, n: int, frame_offsets: np.ndarray, k_sor: int, std_mul: float,
                          k_normals: int, viewpoint: np.ndarray, keep, nx, ny, nz, kept=None, device: bool = False):
    """Thin call for benchmarks: x..nz are raw addresses (ints).  device=True -> *_dev entry point
    (device pointers, nothing copied, asynchronous on the context's stream)."""
    lib = _ffi.load()
    nf = len(frame_offsets) - 1
    if device:
        st = lib.pcr_sor_normals_batch_dev(ctx._h, x, y, z, _p(frame_offsets, _ffi.u64p), nf, k_sor, float(std_mul), k_normals,
                                           _p(viewpoint, _ffi.f32p), keep, nx, ny, nz)
    else:
        cast = lambda a, t: C.cast(C.c_void_p(a), t)
        st = lib.pcr_sor_normals_batch(ctx._h, cast(x, _ffi.f32p), cast(y, _ffi.f32p), cast(z, _ffi.f32p),
                                       _p(frame_offsets, _ffi.u64p), nf, k_sor, float(std_mul), k_normals,
                                       _p(viewpoint, _ffi.f32p), cast(keep, _ffi.u8p), cast(nx, _ffi.f32p), cast(ny, _ffi.f32p),
                                       cast(nz, _ffi.f32p), _p(kept, _ffi.u64p) if kept is not None else None)
    _ffi.check(st, ctx._h)


def radius_outlier_removal_batch(points: np.ndarray, frame_offsets: Sequence[int], radius: float, min_neighbors: int,
                                 ctx: Optional[Context] = None):
    """radius_outlier_removal's mask for every frame of a batch in one call, each point counting only the points of its
    own frame.  -> (keep u8 (N,), kept per frame (F,) u64): frame f's bytes are what ror_mask returns for the frame alone."""
    pts, off = _batch_frames(points, frame_offsets)
    if not math.isfinite(radius) or radius <= 0.0:  # crates/python/src/filters.rs:57-61
        raise ValueError("radius must be > 0 and finite")
    ctx = ctx or default_context()
    x, y, z = _soa(pts)
    n, nf = len(pts), len(off) - 1
    keep = np.zeros(max(n, 1), np.uint8)
    kept = np.zeros(max(nf, 1), np.uint64)
    st = _ffi.load().pcr_radius_outlier_batch(ctx._h, _p(x, _ffi.f32p), _p(y, _ffi.f32p), _p(z, _ffi.f32p), _p(off, _ffi.u64p), nf,
                                              float(radius), int(min_neighbors), _p(keep, _ffi.u8p), _p(kept, _ffi.u64p))
    _ffi.check(st, ctx._h)
    return keep[:n], kept[:nf]


def _frame_lists(lists, off):
    """Checks and stacks one frame-local index list per frame -> (indices u32, list offsets (F+1,) u64); IndexError names
    the frame of an index outside it."""
    nf = len(off) - 1
    if isinstance(lists, (str, bytes)) or not hasattr(lists, "__len__") or len(lists) != nf:
        raise ValueError(f"expected one index list per frame ({nf} frames)")
    parts, l_off = [], np.zeros(nf + 1, np.uint64)
    for f, lst in enumerate(lists):
        a = np.asarray(lst)
        if a.size == 0:
            a = a.reshape(0).astype(np.int64)
        if a.ndim != 1 or a.dtype.kind not in "iu":
            raise ValueError(f"lists[{f}] must be a 1-D integer array")
        n_f = int(off[f + 1] - off[f])
        if len(a) and (int(a.min()) < 0 or int(a.max()) >= n_f):
            bad = int(a.min()) if int(a.min()) < 0 else int(a.max())
            raise IndexError(f"frame {f}: index {bad} out of bounds for a frame with {n_f} points")
        parts.append(a.astype(np.uint32))
        l_off[f + 1] = l_off[f] + len(a)
    idx = np.ascontiguousarray(np.concatenate(parts) if parts else np.zeros(0, np.uint32), np.uint32)
    return idx, l_off


class DeviceFrames:
    """A batch of frames that lives in HBM: the frame-batch counterpart of DeviceCloud.  Every method runs the batch core
    of the matching *_batch call and returns a new DeviceFrames (or host results); frame f of a result is what the
    DeviceCloud method returns for frame f alone.  Indices in and out are frame-local."""

    def __init__(self, handle, ctx: Context):
        self._h = handle
        self._ctx = ctx
        ctx._clouds.add(self)

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    @staticmethod
    def from_numpy(points, frame_offsets: Sequence[int], ctx: Optional[Context] = None) -> "DeviceFrames":
        """points: (N, 3), frame f = rows [frame_offsets[f], frame_offsets[f+1]).  The rows cross PCIe as they are and are
        split into SoA on the device."""
        pts, off = _batch_frames(points, frame_offsets)
        if len(off) < 2:
            raise ValueError("a batch holds at least one frame")
        ctx = ctx or default_context()
        h = C.c_void_p()
        _ffi.check(_ffi.load().pcr_frames_upload_rows(ctx._h, pts.ctypes.data, _p(off, _ffi.u64p), len(off) - 1, C.byref(h)), ctx._h)
        return DeviceFrames(h, ctx)

    def free(self):
        h, self._h = getattr(self, "_h", None), None
        if h and self._ctx._h:  # a closed context has already freed its batches
            _ffi.load().pcr_frames_free(h)

    def _new(self, fn, *args) -> "DeviceFrames":
        h = C.c_void_p()
        _ffi.check(fn(self._h, *args, C.byref(h)), self._ctx._h)
        return DeviceFrames(h, self._ctx)

    @property
    def n_frames(self) -> int:
        return int(_ffi.load().pcr_frames_count(self._h))

    @property
    def offsets(self) -> np.ndarray:
        off = np.zeros(self.n_frames + 1, np.uint64)
        _ffi.check(_ffi.load().pcr_frames_offsets(self._h, _p(off, _ffi.u64p)), self._ctx._h)
        return off

    def len(self) -> int:
        return int(_ffi.load().pcr_frames_len(self._h))

    __len__ = len

    def has_normals(self) -> bool:
        return bool(_ffi.load().pcr_frames_has_normals(self._h))

    def __repr__(self) -> str:
        return f"DeviceFrames(frames={self.n_frames}, n={self.len()}, normals={self.has_normals()})"

    def frame(self, f: int) -> DeviceCloud:
        """Frame f as a DeviceCloud (a device copy, normals carried)."""
        if not 0 <= int(f) < self.n_frames:
            raise IndexError(f"frame {f} out of range ({self.n_frames} frames)")
        h = C.c_void_p()
        _ffi.check(_ffi.load().pcr_frames_frame(self._h, int(f), C.byref(h)), self._ctx._h)
        return DeviceCloud(h, self._ctx)

    def merge(self) -> DeviceCloud:
        """All frames as one DeviceCloud, in frame order, normals carried (a device copy): the map of an odometry chain
        once every frame is in one frame's coordinates (apply_transform), ready for voxel_downsample."""
        h = C.c_void_p()
        _ffi.check(_ffi.load().pcr_frames_merge(self._h, C.byref(h)), self._ctx._h)
        return DeviceCloud(h, self._ctx)

    def apply_transform(self, transforms) -> "DeviceFrames":
        """Frame f moved by transforms[f]: (F, 12) (row-major R, then t, as chain_poses returns them) or (F, 3, 4) [R | t].
        The result carries xyz only (icp.rs:91) and the same offsets."""
        tr = _frame_transforms(transforms, self.n_frames)
        return self._new(_ffi.load().pcr_frames_apply_transform, _p(tr, _ffi.f32p))

    def to_numpy(self):
        """-> (points (N, 3) f32, offsets (F+1,) u64), one download."""
        out = np.empty((self.len(), 3), np.float32)
        _ffi.check(_ffi.load().pcr_frames_download_rows(self._h, out.ctypes.data, None), self._ctx._h)
        return out, self.offsets

    def normals_to_numpy(self) -> Optional[np.ndarray]:
        if not self.has_normals():
            return None
        out = np.empty((self.len(), 3), np.float32)
        _ffi.check(_ffi.load().pcr_frames_download_rows(self._h, None, out.ctypes.data), self._ctx._h)
        return out

    def _select(self, lists, invert: int) -> "DeviceFrames":
        idx, l_off = _frame_lists(lists, self.offsets)
        return self._new(_ffi.load().pcr_frames_select, _p(idx, _ffi.u32p), _p(l_off, _ffi.u64p), invert)

    def select(self, lists) -> "DeviceFrames":
        """lists: one frame-local index array per frame; frame f keeps its listed points in list order (duplicates too)."""
        return self._select(lists, 0)

    def select_inverse(self, lists) -> "DeviceFrames":
        """Frame f keeps the points its list does not name, in their order."""
        return self._select(lists, 1)

    def voxel_downsample(self, voxel_size: float) -> "DeviceFrames":
        if not math.isfinite(voxel_size) or voxel_size <= 0.0:
            raise ValueError("voxel_size must be > 0 and finite")
        return self._new(_ffi.load().pcr_frames_voxel_downsample, float(voxel_size))

    def statistical_outlier_removal(self, k: int, std_mul: float) -> "DeviceFrames":
        if not math.isfinite(std_mul) or std_mul < 0.0:  # crates/python/src/filters.rs:42-46
            raise ValueError("std_mul must be >= 0 and finite")
        return self._new(_ffi.load().pcr_frames_statistical_outlier_removal, int(k), float(std_mul))

    def radius_outlier_removal(self, radius: float, min_neighbors: int) -> "DeviceFrames":
        if not math.isfinite(radius) or radius <= 0.0:
            raise ValueError("radius must be > 0 and finite")
        return self._new(_ffi.load().pcr_frames_radius_outlier_removal, float(radius), int(min_neighbors))

    def estimate_normals(self, k: int, viewpoint=(0.0, 0.0, 0.0)) -> "DeviceFrames":
        vp = np.asarray(viewpoint, np.float32).reshape(3)
        return self._new(_ffi.load().pcr_frames_estimate_normals, int(k), _p(vp, _ffi.f32p))

    def sor_normals(self, k_sor: int, std_mul: float, k_normals: int, viewpoint=(0.0, 0.0, 0.0)) -> "DeviceFrames":
        if not math.isfinite(std_mul) or std_mul < 0.0:
            raise ValueError("std_mul must be >= 0 and finite")
        vp = np.asarray(viewpoint, np.float32).reshape(3)
        return self._new(_ffi.load().pcr_frames_sor_normals, int(k_sor), float(std_mul), int(k_normals), _p(vp, _ffi.f32p))

    def ransac_plane_samples(self, distance_threshold: float, samples, outliers: bool = False):
        """samples: one (m_f, 3) array of frame-local triples per frame.  -> one PlaneResult per frame, and with
        outliers=True also the DeviceFrames of every frame's select_inverse(inliers), built on the device."""
        off = self.offsets
        smp, s_off = _frame_samples(samples, off)
        nf = len(off) - 1
        models = np.zeros((nf, 4), np.float32)
        inl = np.zeros(max(int(off[-1]), 1), np.uint32)
        inl_off = np.zeros(nf + 1, np.uint64)
        h = C.c_void_p()
        st = _ffi.load().pcr_frames_ransac_plane_samples(self._h, float(distance_threshold), _p(smp, _ffi.u32p), _p(s_off, _ffi.u64p),
                                                         _p(models, _ffi.f32p), _p(inl, _ffi.u32p), _p(inl_off, _ffi.u64p),
                                                         C.byref(h) if outliers else None)
        _ffi.check(st, self._ctx._h)
        res = [PlaneResult(models[f, :3], models[f, 3], inl[int(inl_off[f]):int(inl_off[f + 1])].tolist()) for f in range(nf)]
        return (res, DeviceFrames(h, self._ctx)) if outliers else res

    def ransac_plane(self, distance_threshold: float, iterations: int, seed=None, outliers: bool = False):
        """Frame f's triples are draw_plane_samples(n_f, iterations, [seed, f]), as ransac_plane_batch draws them."""
        off = self.offsets
        samples = [draw_plane_samples(int(off[f + 1] - off[f]), iterations, None if seed is None else [seed, f]) for f in range(len(off) - 1)]
        return self.ransac_plane_samples(distance_threshold, samples, outliers)

    def cluster_arrays(self, distance_threshold: float, min_size: int, max_size: int):
        """-> (cluster_offsets (F+1,) u64, offsets u32, indices u32), as cluster_arrays_batch."""
        n, nf = self.len(), self.n_frames
        offsets = np.zeros(n + 1, np.uint32)
        idx = np.zeros(max(n, 1), np.uint32)
        c_off = np.zeros(nf + 1, np.uint64)
        st = _ffi.load().pcr_frames_euclidean_cluster(self._h, float(distance_threshold), int(min_size), int(max_size), _p(offsets, _ffi.u32p),
                                                      _p(idx, _ffi.u32p), _p(c_off, _ffi.u64p))
        _ffi.check(st, self._ctx._h)
        k = int(c_off[-1])
        return c_off, offsets[:k + 1].copy(), idx[:int(offsets[k])].copy()

    def euclidean_cluster(self, distance_threshold: float, min_size: int, max_size: int) -> List[List[List[int]]]:
        """-> one list of index lists per frame, each what DeviceCloud.euclidean_cluster returns for the frame alone."""
        c_off, offsets, idx = self.cluster_arrays(distance_threshold, min_size, max_size)
        return [[idx[offsets[c]:offsets[c + 1]].tolist() for c in range(int(c_off[f]), int(c_off[f + 1]))] for f in range(len(c_off) - 1)]

    def _icp(self, fn, pairs, max_iterations, tolerance, max_correspondence_distance) -> List[IcpResult]:
        prm = _icp_params(max_iterations, tolerance, max_correspondence_distance)
        nf = self.n_frames
        pr = np.asarray(pairs)
        if pr.size == 0:
            pr = pr.reshape(0, 2)
        if pr.ndim != 2 or pr.shape[1] != 2 or (len(pr) and pr.dtype.kind not in "iu"):
            raise ValueError("pairs must be an integer array of shape (P, 2): (source frame, target frame)")
        if len(pr) and (pr.min() < 0 or pr.max() >= nf):
            raise ValueError(f"pairs hold a frame id outside [0, {nf})")
        pr = np.ascontiguousarray(pr, np.uint32)
        res = (_ffi.IcpResultC * max(len(pr), 1))()
        _ffi.check(fn(self._h, _p(pr, _ffi.u32p), len(pr), C.byref(prm), res), self._ctx._h)
        return [IcpResult(res[i]) for i in range(len(pr))]

    def icp_point_to_point(self, pairs, max_iterations: int = 50, tolerance: float = 1e-5,
                           max_correspondence_distance: float = math.inf) -> List[IcpResult]:
        """pairs: (P, 2) frame ids, pair p registers frame pairs[p][0] onto frame pairs[p][1] -> one IcpResult per pair."""
        return self._icp(_ffi.load().pcr_frames_icp_point_to_point, pairs, max_iterations, tolerance, max_correspondence_distance)

    def icp_point_to_plane(self, pairs, max_iterations: int = 50, tolerance: float = 1e-5,
                           max_correspondence_distance: float = math.inf) -> List[IcpResult]:
        """Point-to-plane form; the batch must carry normals (estimate_normals / sor_normals)."""
        if not self.has_normals():  # crates/python/src/registration.rs:66-71
            raise ValueError("point-to-plane ICP needs frames with normals. Use estimate_normals first.")
        return self._icp(_ffi.load().pcr_frames_icp_point_to_plane, pairs, max_iterations, tolerance, max_correspondence_distance)


def _query_frames(queries, query_offsets, n_frames: int):
    """Checks and converts the queries of a KdTreeBatch call: (nq,3) rows, frames back to back, one frame per index frame."""
    q, off = _batch_frames(queries, query_offsets)
    if len(off) - 1 != n_frames:
        raise ValueError(f"query_offsets describe {len(off) - 1} frames, the index holds {n_frames}")
    return _soa(q), off


class KdTreeBatch:
    """KdTree over many frames at once: frame f = rows [frame_offsets[f], frame_offsets[f+1]) of the points, queried with
    frames of queries back to back, query frame f searched in index frame f only.  Frame f's results are what
    KdTree(frame f).<method>(queries of frame f) returns; indices in and out are frame-local.  The index stays in HBM
    (cell table and grid levels included) until the object is freed."""

    def __init__(self, points, frame_offsets: Sequence[int], k_hint: int = 0, ctx: Optional[Context] = None, _handle=None):
        if _handle is not None:
            self._ctx = ctx
            self._h, self._off = _handle, np.ascontiguousarray(frame_offsets, np.uint64)
        else:
            pts, off = _batch_frames(points, frame_offsets)
            if len(off) < 2:
                raise ValueError("a batch index holds at least one frame")
            self._ctx = ctx or default_context()
            x, y, z = _soa(pts)
            h = C.c_void_p()
            _ffi.check(_ffi.load().pcr_index_build_batch(self._ctx._h, _p(x, _ffi.f32p), _p(y, _ffi.f32p), _p(z, _ffi.f32p), _p(off, _ffi.u64p),
                                                         len(off) - 1, int(k_hint), C.byref(h)), self._ctx._h)
            self._h, self._off = h, off
        self._ctx._clouds.add(self)

    @staticmethod
    def from_device_frames(frames: "DeviceFrames", k_hint: int = 0) -> "KdTreeBatch":
        """The index of a DeviceFrames batch, built from its device arrays (no host copy of the points)."""
        off = frames.offsets
        ptrs = [C.c_void_p() for _ in range(6)]
        lib = _ffi.load()
        _ffi.check(lib.pcr_frames_device_pointers(frames._h, *(C.byref(p) for p in ptrs)), frames._ctx._h)
        h = C.c_void_p()
        _ffi.check(lib.pcr_index_build_batch_dev(frames._ctx._h, ptrs[0], ptrs[1], ptrs[2], _p(off, _ffi.u64p), len(off) - 1, int(k_hint),
                                                 C.byref(h)), frames._ctx._h)
        return KdTreeBatch(None, off, ctx=frames._ctx, _handle=h)

    def free(self):
        h, self._h = getattr(self, "_h", None), None
        if h and self._ctx._h:  # a closed context has already freed its indexes
            _ffi.load().pcr_index_free(h)

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    @property
    def n_frames(self) -> int:
        return len(self._off) - 1

    @property
    def offsets(self) -> np.ndarray:
        return self._off.copy()

    def len(self) -> int:
        return int(_ffi.load().pcr_index_len(self._h))

    __len__ = len

    def __repr__(self) -> str:
        return f"KdTreeBatch(frames={self.n_frames}, n={self.len()})"

    def _knn(self, queries, query_offsets, k: int, want_dist: bool):
        (qx, qy, qz), off = _query_frames(queries, query_offsets, self.n_frames)
        nq = len(qx)
        idx = np.full((nq, max(k, 0)), 0xFFFFFFFF, np.uint32)
        dist = np.full((nq, max(k, 0)), np.inf, np.float32) if want_dist else None
        cnt = np.zeros(nq, np.uint32)
        st = _ffi.load().pcr_knn_batch(self._h, _p(qx, _ffi.f32p), _p(qy, _ffi.f32p), _p(qz, _ffi.f32p), _p(off, _ffi.u64p), self.n_frames,
                                       int(k), _p(idx, _ffi.u32p), _p(dist, _ffi.f32p), _p(cnt, _ffi.u32p))
        _ffi.check(st, self._ctx._h)
        return idx, dist, cnt

    def knn(self, queries, query_offsets: Sequence[int], k: int):
        """-> (idx (nq,k) u32, dist (nq,k) f32, counts (nq,) u32), rows as KdTree.knn, indices frame-local."""
        return self._knn(queries, query_offsets, k, True)

    def knn_indices(self, queries, query_offsets: Sequence[int], k: int):
        idx, _, cnt = self._knn(queries, query_offsets, k, False)
        return idx, cnt

    def radius_count(self, queries, query_offsets: Sequence[int], radius: float) -> np.ndarray:
        (qx, qy, qz), off = _query_frames(queries, query_offsets, self.n_frames)
        cnt = np.zeros(len(qx), np.uint32)
        st = _ffi.load().pcr_radius_count_batch(self._h, _p(qx, _ffi.f32p), _p(qy, _ffi.f32p), _p(qz, _ffi.f32p), _p(off, _ffi.u64p),
                                                self.n_frames, float(radius), _p(cnt, _ffi.u32p))
        _ffi.check(st, self._ctx._h)
        return cnt

    def radius_search(self, queries, query_offsets: Sequence[int], radius: float):
        """CSR over all queries: (offsets (nq+1,) u64, idx u32), every row frame-local and ascending (kdtree.rs:132)."""
        (qx, qy, qz), off = _query_frames(queries, query_offsets, self.n_frames)
        nq = len(qx)
        r_off = np.zeros(nq + 1, np.uint64)
        total = C.c_size_t()
        cap = max(16 * nq, 1024)
        lib = _ffi.load()
        for _ in range(2):
            idx = np.empty(cap, np.uint32)
            st = lib.pcr_radius_search_batch(self._h, _p(qx, _ffi.f32p), _p(qy, _ffi.f32p), _p(qz, _ffi.f32p), _p(off, _ffi.u64p), self.n_frames,
                                             float(radius), _p(r_off, _ffi.u64p), _p(idx, _ffi.u32p), cap, C.byref(total))
            if st == _ffi.PCR_ERR_CAPACITY:
                cap = int(total.value)
                continue
            _ffi.check(st, self._ctx._h)
            return r_off, idx[: total.value].copy()
        raise PcrError(_ffi.PCR_ERR_CAPACITY, "radius_search: capacity retry failed")

    def find_correspondences(self, queries, query_offsets: Sequence[int], max_distance: float = math.inf):
        """-> (src_idx u32, tgt_idx u32, dist f32, corr_offsets (F+1,) u64): frame f's pairs are [corr_offsets[f],
        corr_offsets[f+1]), as KdTree(frame f).find_correspondences(queries of frame f) returns them."""
        (qx, qy, qz), off = _query_frames(queries, query_offsets, self.n_frames)
        ns = len(qx)
        si, ti = np.empty(max(ns, 1), np.uint32), np.empty(max(ns, 1), np.uint32)
        dd = np.empty(max(ns, 1), np.float32)
        c_off = np.zeros(self.n_frames + 1, np.uint64)
        st = _ffi.load().pcr_find_correspondences_batch(self._h, _p(qx, _ffi.f32p), _p(qy, _ffi.f32p), _p(qz, _ffi.f32p), _p(off, _ffi.u64p),
                                                        self.n_frames, float(max_distance), _p(si, _ffi.u32p), _p(ti, _ffi.u32p),
                                                        _p(dd, _ffi.f32p), _p(c_off, _ffi.u64p))
        _ffi.check(st, self._ctx._h)
        m = int(c_off[-1])
        return si[:m].copy(), ti[:m].copy(), dd[:m].copy(), c_off
