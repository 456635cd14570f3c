"""ctypes binding of lib/libpcr_b200.so (the C ABI declared in include/pcr_b200.h).

There is no CPU fallback: if the shared library has not been built, or no B200 is visible, the
calls raise.  Build with `python __graft_entry__.py build` (or `make -C pointclouds_rs_b200/csrc`).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PCR_LIB_OVERRIDE") or os.path.join(_HERE, "lib", "libpcr_b200.so")  # override: A/B builds

PCR_OK = 0
PCR_ERR_INVALID_ARG = 1
PCR_ERR_NORMALS_MISMATCH = 2
PCR_ERR_CUDA = 3
PCR_ERR_NCCL = 4
PCR_ERR_OOM = 5
PCR_ERR_NO_DEVICE = 6
PCR_ERR_UNSUPPORTED = 7
PCR_ERR_CAPACITY = 8
PCR_MAX_K = 1024
PCR_UNIQUE_ID_BYTES = 128
PCR_NUM_TIMING_TAGS = 8
TIMING_TAGS = ("build", "knn", "knn_deferred", "sor_stats", "icp_step", "icp_solve", "knn_normals", "other")

f32p = C.POINTER(C.c_float)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int32)
szp = C.POINTER(C.c_size_t)
vp = C.c_void_p


class IcpParams(C.Structure):
    _fields_ = [("max_iterations", C.c_uint64), ("tolerance", C.c_float), ("max_correspondence_distance", C.c_float)]


class IcpResultC(C.Structure):
    _fields_ = [
        ("rotation", C.c_float * 9),
        ("translation", C.c_float * 3),
        ("fitness", C.c_float),
        ("rmse", C.c_float),
        ("converged", C.c_int32),
        ("num_iterations", C.c_uint64),
    ]


class PcrError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"pcr_b200 error {code}: {message}")
        self.code = code
        self.message = message


# name -> (restype, argtypes); exactly the symbols include/pcr_b200.h declares
SIGNATURES = {
    "pcr_version": (C.c_int, []),
    "pcr_device_count": (C.c_int, []),
    "pcr_ctx_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "pcr_ctx_create_on_stream": (C.c_int, [C.c_int, vp, C.POINTER(vp)]),
    "pcr_ctx_destroy": (None, [vp]),
    "pcr_ctx_synchronize": (C.c_int, [vp]),
    "pcr_last_error": (C.c_char_p, [vp]),
    "pcr_ctx_launch_count": (C.c_uint64, [vp]),
    "pcr_ctx_set_cell_size": (C.c_int, [vp, C.c_float]),
    "pcr_ctx_set_frame_stream": (C.c_int, [vp, C.c_int]),
    "pcr_ctx_get_hint_stats": (C.c_int, [vp, u64p]),
    "pcr_ctx_get_knn_counters": (C.c_int, [vp, u64p]),
    "pcr_ctx_set_query_sharding": (C.c_int, [vp, C.c_int]),
    "pcr_ctx_debug_set_shard": (C.c_int, [vp, C.c_int, C.c_int]),
    "pcr_ctx_set_timing": (C.c_int, [vp, C.c_int]),
    "pcr_ctx_get_timing": (C.c_int, [vp, C.POINTER(C.c_double), u64p]),
    "pcr_comm_unique_id": (C.c_int, [vp]),
    "pcr_ctx_comm_init": (C.c_int, [vp, vp, C.c_int, C.c_int]),
    "pcr_ctx_comm_rank": (C.c_int, [vp]),
    "pcr_ctx_comm_size": (C.c_int, [vp]),
    "pcr_ctx_comm_kind": (C.c_int, [vp]),
    "pcr_index_build": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, C.c_size_t, C.POINTER(vp)]),
    "pcr_index_build_dev": (C.c_int, [vp, vp, vp, vp, C.c_size_t, C.c_size_t, C.POINTER(vp)]),
    "pcr_index_free": (None, [vp]),
    "pcr_index_len": (C.c_size_t, [vp]),
    "pcr_index_info": (C.c_int, [vp, f32p, i32p, szp]),
    "pcr_knn": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, C.c_size_t, u32p, f32p, u32p]),
    "pcr_knn_dev": (C.c_int, [vp, vp, vp, vp, C.c_size_t, C.c_size_t, vp, vp, vp]),
    "pcr_radius_count": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, C.c_float, u32p]),
    "pcr_radius_search": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, C.c_float, u64p, u32p, C.c_size_t, szp]),
    "pcr_index_build_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, C.c_size_t, C.POINTER(vp)]),
    "pcr_index_build_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, C.c_size_t, C.POINTER(vp)]),
    "pcr_knn_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, C.c_size_t, u32p, f32p, u32p]),
    "pcr_knn_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, C.c_size_t, vp, vp, vp]),
    "pcr_radius_count_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, C.c_float, u32p]),
    "pcr_radius_count_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, C.c_float, vp]),
    "pcr_radius_search_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, C.c_float, u64p, u32p, C.c_size_t, szp]),
    "pcr_find_correspondences_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, C.c_float, u32p, u32p, f32p, u64p]),
    "pcr_sor": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, C.c_size_t, C.c_float, u8p, szp, f32p, f32p]),
    "pcr_sor_dev": (C.c_int, [vp, vp, vp, vp, C.c_size_t, C.c_size_t, C.c_float, vp, vp]),
    "pcr_radius_outlier": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, C.c_float, C.c_size_t, u8p, szp]),
    "pcr_estimate_normals": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, C.c_size_t, f32p, f32p, f32p, f32p]),
    "pcr_estimate_normals_dev": (C.c_int, [vp, vp, vp, vp, C.c_size_t, C.c_size_t, f32p, vp, vp, vp]),
    "pcr_find_correspondences": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, C.c_float, u32p, u32p, f32p, szp]),
    "pcr_apply_transform": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, f32p, f32p, f32p, f32p, f32p]),
    "pcr_icp_point_to_point": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, f32p, f32p, f32p, C.c_size_t, C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
    "pcr_icp_point_to_plane": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, f32p, f32p, f32p, C.c_size_t, f32p, f32p, f32p, C.c_size_t, C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
    "pcr_icp_point_to_point_dev": (C.c_int, [vp, vp, vp, vp, C.c_size_t, vp, vp, vp, C.c_size_t, C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
    "pcr_icp_point_to_plane_dev": (C.c_int, [vp, vp, vp, vp, C.c_size_t, vp, vp, vp, C.c_size_t, vp, vp, vp, C.c_size_t, C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
    "pcr_icp_point_to_point_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, u32p, C.c_size_t, C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
    "pcr_icp_point_to_plane_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, f32p, f32p, f32p, C.c_size_t, u32p, C.c_size_t,
                                               C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
    "pcr_icp_point_to_point_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, u32p, C.c_size_t, C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
    "pcr_icp_point_to_plane_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, vp, vp, vp, C.c_size_t, u32p, C.c_size_t,
                                                   C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
    "pcr_voxel_downsample": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, C.c_float, f32p, f32p, f32p, szp]),
    "pcr_voxel_downsample_dev": (C.c_int, [vp, vp, vp, vp, C.c_size_t, C.c_float, vp, vp, vp, szp]),
    "pcr_voxel_downsample_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, C.c_float, f32p, f32p, f32p, u64p]),
    "pcr_voxel_downsample_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, C.c_float, vp, vp, vp, u64p]),
    "pcr_estimate_normals_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, C.c_size_t, f32p, f32p, f32p, f32p]),
    "pcr_estimate_normals_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, C.c_size_t, f32p, vp, vp, vp]),
    "pcr_euclidean_cluster": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, C.c_float, C.c_size_t, C.c_size_t, u32p, u32p, szp]),
    "pcr_cluster_labels_dev": (C.c_int, [vp, vp, vp, vp, C.c_size_t, C.c_float, vp]),
    "pcr_radius_outlier_dev": (C.c_int, [vp, vp, vp, vp, C.c_size_t, C.c_float, C.c_size_t, vp]),
    "pcr_cloud_upload": (C.c_int, [vp, vp, vp, vp, C.c_size_t, C.POINTER(vp)]),
    "pcr_cloud_upload_block": (C.c_int, [vp, vp, C.c_size_t, C.c_size_t, C.POINTER(vp)]),
    "pcr_cloud_upload_block_nowait": (C.c_int, [vp, vp, C.c_size_t, C.c_size_t, C.POINTER(vp)]),
    "pcr_cloud_download_block": (C.c_int, [vp, vp, C.c_size_t, C.c_int]),
    "pcr_cloud_free": (None, [vp]),
    "pcr_cloud_len": (C.c_size_t, [vp]),
    "pcr_cloud_has_normals": (C.c_int, [vp]),
    "pcr_cloud_download": (C.c_int, [vp, vp, vp, vp]),
    "pcr_cloud_download_normals": (C.c_int, [vp, vp, vp, vp]),
    "pcr_cloud_upload_rows": (C.c_int, [vp, vp, C.c_size_t, C.POINTER(vp)]),
    "pcr_cloud_download_rows": (C.c_int, [vp, vp, vp]),
    "pcr_cloud_device_pointers": (C.c_int, [vp] + [C.POINTER(vp)] * 6),
    "pcr_cloud_select": (C.c_int, [vp, u32p, C.c_size_t, C.POINTER(vp)]),
    "pcr_cloud_voxel_downsample": (C.c_int, [vp, C.c_float, C.POINTER(vp)]),
    "pcr_cloud_statistical_outlier_removal": (C.c_int, [vp, C.c_size_t, C.c_float, C.POINTER(vp)]),
    "pcr_cloud_radius_outlier_removal": (C.c_int, [vp, C.c_float, C.c_size_t, C.POINTER(vp)]),
    "pcr_cloud_estimate_normals": (C.c_int, [vp, C.c_size_t, f32p, C.POINTER(vp)]),
    "pcr_cloud_sor_normals": (C.c_int, [vp, C.c_size_t, C.c_float, C.c_size_t, f32p, C.POINTER(vp)]),
    "pcr_cloud_euclidean_cluster": (C.c_int, [vp, C.c_float, C.c_size_t, C.c_size_t, u32p, u32p, szp]),
    "pcr_cloud_apply_transform": (C.c_int, [vp, f32p, f32p, C.POINTER(vp)]),
    "pcr_cloud_icp_point_to_point": (C.c_int, [vp, vp, C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
    "pcr_cloud_icp_point_to_plane": (C.c_int, [vp, vp, C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
    "pcr_ransac_plane_samples": (C.c_int, [vp, f32p, f32p, f32p, C.c_size_t, C.c_float, u32p, C.c_size_t, f32p, u32p, szp]),
    "pcr_cloud_ransac_plane_samples": (C.c_int, [vp, C.c_float, u32p, C.c_size_t, f32p, u32p, szp]),
    "pcr_ransac_plane_samples_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, C.c_float, u32p, u64p, f32p, u32p, u64p]),
    "pcr_ransac_plane_samples_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, C.c_float, u32p, u64p, f32p, vp, u64p]),
    "pcr_euclidean_cluster_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, C.c_float, C.c_size_t, C.c_size_t, u32p, u32p, u64p]),
    "pcr_euclidean_cluster_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, C.c_float, C.c_size_t, C.c_size_t, vp, vp, u64p]),
    "pcr_cluster_labels_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, C.c_float, vp]),
    "pcr_sor_normals_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, C.c_size_t, C.c_float, C.c_size_t, f32p, u8p, f32p, f32p, f32p, u64p]),
    "pcr_sor_normals_batch_rows": (C.c_int, [vp, f32p, u64p, C.c_size_t, C.c_size_t, C.c_float, C.c_size_t, f32p, u8p, f32p, u64p]),
    "pcr_sor_normals_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, C.c_size_t, C.c_float, C.c_size_t, f32p, vp, vp, vp, vp]),
    "pcr_radius_outlier_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, C.c_float, C.c_size_t, u8p, u64p]),
    "pcr_radius_outlier_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, C.c_float, C.c_size_t, vp]),
    "pcr_frames_upload": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, C.POINTER(vp)]),
    "pcr_frames_upload_rows": (C.c_int, [vp, vp, u64p, C.c_size_t, C.POINTER(vp)]),
    "pcr_frames_free": (None, [vp]),
    "pcr_frames_len": (C.c_size_t, [vp]),
    "pcr_frames_count": (C.c_size_t, [vp]),
    "pcr_frames_offsets": (C.c_int, [vp, u64p]),
    "pcr_frames_has_normals": (C.c_int, [vp]),
    "pcr_frames_device_pointers": (C.c_int, [vp] + [C.POINTER(vp)] * 6),
    "pcr_frames_download": (C.c_int, [vp, vp, vp, vp, vp, vp, vp]),
    "pcr_frames_download_rows": (C.c_int, [vp, vp, vp]),
    "pcr_frames_frame": (C.c_int, [vp, C.c_size_t, C.POINTER(vp)]),
    "pcr_frames_merge": (C.c_int, [vp, C.POINTER(vp)]),
    "pcr_frames_apply_transform": (C.c_int, [vp, f32p, C.POINTER(vp)]),
    "pcr_apply_transform_batch": (C.c_int, [vp, f32p, f32p, f32p, u64p, C.c_size_t, f32p, f32p, f32p, f32p]),
    "pcr_apply_transform_batch_dev": (C.c_int, [vp, vp, vp, vp, u64p, C.c_size_t, f32p, vp, vp, vp]),
    "pcr_transform_compose": (C.c_int, [f32p, f32p, f32p]),
    "pcr_frames_select": (C.c_int, [vp, u32p, u64p, C.c_int, C.POINTER(vp)]),
    "pcr_frames_voxel_downsample": (C.c_int, [vp, C.c_float, C.POINTER(vp)]),
    "pcr_frames_statistical_outlier_removal": (C.c_int, [vp, C.c_size_t, C.c_float, C.POINTER(vp)]),
    "pcr_frames_radius_outlier_removal": (C.c_int, [vp, C.c_float, C.c_size_t, C.POINTER(vp)]),
    "pcr_frames_estimate_normals": (C.c_int, [vp, C.c_size_t, f32p, C.POINTER(vp)]),
    "pcr_frames_sor_normals": (C.c_int, [vp, C.c_size_t, C.c_float, C.c_size_t, f32p, C.POINTER(vp)]),
    "pcr_frames_ransac_plane_samples": (C.c_int, [vp, C.c_float, u32p, u64p, f32p, u32p, u64p, C.POINTER(vp)]),
    "pcr_frames_euclidean_cluster": (C.c_int, [vp, C.c_float, C.c_size_t, C.c_size_t, u32p, u32p, u64p]),
    "pcr_frames_icp_point_to_point": (C.c_int, [vp, u32p, C.c_size_t, C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
    "pcr_frames_icp_point_to_plane": (C.c_int, [vp, u32p, C.c_size_t, C.POINTER(IcpParams), C.POINTER(IcpResultC)]),
}

_lib = None


def load():
    """Load the shared library (raises if it has not been built -- no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA extension first "
                "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback."
            )
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the ABI is incomplete
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def last_error(ctx=None) -> str:
    msg = load().pcr_last_error(ctx)
    return msg.decode(errors="replace") if msg else "unknown error"


def check(status: int, ctx=None):
    if status != PCR_OK:
        msg = last_error(ctx)
        if status == PCR_ERR_INVALID_ARG or status == PCR_ERR_NORMALS_MISMATCH:
            raise ValueError(msg)  # the reference's Python layer maps these to ValueError
        raise PcrError(status, msg)
