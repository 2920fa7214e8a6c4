"""ctypes binding of libnornic_knn.so — every symbol include/nornic_knn.h declares.

The product path fails loudly when the CUDA library is missing: there is no CPU fallback anywhere in
this package (the CPU oracle lives under oracle/ and is test infrastructure only)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnornic_knn.so")


class CudaBuffer(C.Structure):
    # pkg/gpu/cuda/cuda_bridge.go:132-136
    _fields_ = [("data", C.c_void_p), ("size", C.c_size_t), ("memory_type", C.c_int)]


class NkStats(C.Structure):
    _fields_ = [
        ("rows", C.c_uint64), ("searches", C.c_uint64), ("queries", C.c_uint64), ("kernel_launches", C.c_uint64),
        ("bytes_h2d", C.c_uint64), ("bytes_d2h", C.c_uint64), ("bytes_scanned", C.c_uint64),
        ("n_devices", C.c_uint32), ("dim", C.c_uint32),
    ]


_vp, _i, _u, _u64, _sz = C.c_void_p, C.c_int, C.c_uint, C.c_uint64, C.c_size_t
_fp = C.POINTER(C.c_float)
_up = C.POINTER(C.c_uint32)
_bufp = C.POINTER(CudaBuffer)

# name -> (restype, argtypes).  Keep in lock-step with include/nornic_knn.h (tests/test_abi.py checks).
SIGNATURES = {
    # ---- legacy ABI (cuda_bridge.go:20-375)
    "cuda_set_error": (None, [C.c_char_p]),
    "cuda_get_last_error": (C.c_char_p, []),
    "cuda_clear_error": (None, []),
    "cuda_get_device_count": (_i, []),
    "cuda_is_available": (_i, []),
    "cuda_create_device": (_vp, [_i]),
    "cuda_release_device": (None, [_vp]),
    "cuda_device_name": (C.c_char_p, [_i]),
    "cuda_device_memory": (_sz, [_i]),
    "cuda_device_compute_capability": (_i, [_i]),
    "cuda_create_buffer": (_bufp, [_vp, _vp, _sz, _i]),
    "cuda_release_buffer": (None, [_bufp]),
    "cuda_buffer_data": (_vp, [_bufp]),
    "cuda_buffer_size": (_sz, [_bufp]),
    "cuda_buffer_copy_to_host": (_i, [_bufp, _vp, _sz]),
    "cuda_compute_norms": (_i, [_vp, _bufp, _bufp, _u, _u]),
    "cuda_normalize_vectors": (_i, [_vp, _bufp, _u, _u]),
    "cuda_cosine_similarity": (_i, [_vp, _bufp, _bufp, _bufp, _u, _u, _i]),
    "cuda_topk": (_i, [_vp, _bufp, _vp, _vp, _u, _u]),
    # ---- fused batched API
    "nk_last_error": (C.c_char_p, []),
    "nk_version": (C.c_char_p, []),
    "nk_index_create": (_vp, [C.POINTER(C.c_int), _i, C.c_uint32, _i, _i]),
    "nk_index_release": (None, [_vp]),
    "nk_index_upload": (_i, [_vp, _vp, _u64]),
    "nk_index_append": (_i, [_vp, _vp, _u64]),
    "nk_index_update_row": (_i, [_vp, _u64, _vp]),
    "nk_index_remove_swap": (_i, [_vp, _u64]),
    "nk_index_fill_uniform": (_i, [_vp, _u64, _u64]),
    "nk_index_set_row_base": (_i, [_vp, _u64]),
    "nk_index_attach_device_rows": (_i, [_vp, _vp, _u64]),
    "nk_index_set_path": (_i, [_vp, _i]),
    "nk_index_rows": (_u64, [_vp]),
    "nk_index_stats": (_i, [_vp, C.POINTER(NkStats)]),
    "nk_index_last_path": (_i, [_vp]),
    "nk_index_debug_flags": (_i, [_vp, C.POINTER(C.c_int)]),
    "nk_index_enable_timing": (_i, [_vp, _i]),
    "nk_index_scan_time_ms": (_i, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "nk_index_read_rows": (_i, [_vp, _u64, _u64, _vp]),
    "nk_search": (_i, [_vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp]),
    "nk_search_device": (_i, [_vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp, _vp]),
    "nk_search_keys_device": (_i, [_vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp]),
    "nk_merge_keys_device": (_i, [_i, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _i, _vp, _vp, _vp]),
    "nk_score_subset": (_i, [_vp, _vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp]),
    "nk_index_set_row_mask": (_i, [_vp, _vp, _u64]),
    "nk_index_upload_from_f32": (_i, [_vp, _vp, _u64]),
    "nk_blob_vectors": (_i, [_vp, C.c_size_t, _vp, _vp, _vp]),
    "nk_index_assign_nearest": (_i, [_vp, _vp, C.c_uint32, _i, _vp, _vp]),
    "nk_index_cluster_means": (_i, [_vp, _vp, C.c_uint32, _vp, _vp]),
    "nk_index_kmeanspp": (_i, [_vp, C.c_uint32, _u64, _vp, _vp, _vp, _vp]),
    "nk_fill_uniform_device": (_i, [_i, _vp, _u64, C.c_uint32, _u64, _u64, _vp]),
    "nk_index_fill_clustered": (_i, [_vp, _u64, _u64, C.c_uint32, C.c_float, _i]),
    "nk_index_refresh_shadow": (_i, [_vp]),
    "nk_index_set_metric": (_i, [_vp, _i]),
    "nk_index_set_min_score": (_i, [_vp, C.c_float]),
    "nk_index_debug_counters": (_i, [_vp, C.POINTER(C.c_uint64)]),
    "nk_debug_filter_dump": (_i, [_vp, _vp, C.c_uint32, _i, _vp, _vp]),
    "nk_index_status": (_i, [_vp, _vp]),
    "nk_index_set_row_groups": (_i, [_vp, _vp, _u64, C.c_uint32]),
    "nk_search_groups": (_i, [_vp, _vp, C.c_uint32, _vp, _vp, _vp]),
    "nk_index_set_clusters": (_i, [_vp, _vp, C.c_uint32, _vp, _u64]),
    "nk_search_clusters": (_i, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _vp, _vp, _vp]),
    "nk_search_clusters_device": (_i, [_vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _vp, _vp, _vp, _vp]),
    "nk_comm_create": (_vp, [_i, _i, _i, _sz]),
    "nk_comm_export": (_i, [_vp, _vp]),
    "nk_comm_connect": (_i, [_vp, _vp]),
    "nk_comm_connect_local": (_i, [C.POINTER(_vp), _i]),
    "nk_comm_status": (_i, [_vp, _vp]),
    "nk_comm_release": (None, [_vp]),
    "nk_comm_exchange_merge": (_i, [_vp, _vp, C.c_uint32, C.c_uint32, _i, _vp, _vp, _vp]),
    "nk_search_sharded_device": (_i, [_vp, _vp, _vp, C.c_uint32, C.c_uint32, _vp, _vp, _vp]),
}

_lib = None


def load() -> C.CDLL:
    """Load the CUDA library; raise (never fall back) if it is missing or fails to load."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m nornicdb_b200.build` "
            "(or __graft_entry__.build()).  There is no CPU fallback in this package.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    msg = load().nk_last_error()
    return msg.decode("utf-8", "replace") if msg else ""
