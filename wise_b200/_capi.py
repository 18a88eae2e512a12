"""ctypes binding of libwiseb200.so (include/wise_b200.h).

This is the only place the shared library is loaded.  There is deliberately no fallback: if the
library is missing, or a compute call is made without a B200, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WISE_B200_LIB") or os.path.join(_HERE, "libwiseb200.so")

WB_MAX_K = 2048

_f32p = C.POINTER(C.c_float)
_i64p = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)
_vp = C.c_void_p

# name -> (restype, argtypes); mirrors include/wise_b200.h one to one (tests check this).
SIGNATURES = {
    "wb_last_error": (C.c_char_p, []),
    "wb_version": (C.c_char_p, []),
    "wb_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "wb_flat_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(_vp)]),
    "wb_ivf_create": (C.c_int, [C.c_int, C.c_int64, C.c_int, C.POINTER(_vp)]),
    "wb_free": (C.c_int, [_vp]),
    "wb_dim": (C.c_int64, [_vp]),
    "wb_ntotal": (C.c_int64, [_vp]),
    "wb_is_trained": (C.c_int, [_vp]),
    "wb_nlist": (C.c_int64, [_vp]),
    "wb_is_ivf": (C.c_int, [_vp]),
    "wb_reserve": (C.c_int, [_vp, C.c_int64]),
    "wb_capacity": (C.c_int, [_vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "wb_add_with_ids": (C.c_int, [_vp, C.c_int64, _vp, _vp]),
    "wb_add_with_ids_dev": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp]),
    "wb_pinned_alloc": (C.c_int, [C.c_int64, C.POINTER(_vp)]),
    "wb_pinned_free": (C.c_int, [_vp]),
    "wb_add_with_ids_pinned": (C.c_int, [_vp, C.c_int64, _vp, _vp, C.c_int]),
    "wb_ivf_add_preassigned_pinned": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, C.c_int]),
    "wb_add_slot_wait": (C.c_int, [_vp, C.c_int]),
    "wb_sync": (C.c_int, [_vp]),
    "wb_ivf_train": (C.c_int, [_vp, C.c_int64, _vp, C.c_int, C.c_int64]),
    "wb_ivf_set_centroids": (C.c_int, [_vp, _vp]),
    "wb_ivf_get_centroids": (C.c_int, [_vp, _vp]),
    "wb_ivf_mark_trained": (C.c_int, [_vp]),
    "wb_ivf_set_spherical": (C.c_int, [_vp, C.c_int]),
    "wb_kmeans_assign_dev": (C.c_int, [_vp, C.c_int64, _vp, _vp, C.POINTER(C.c_double), _vp]),
    "wb_kmeans_assign_fast_dev": (C.c_int, [_vp, C.c_int64, _vp, _vp, C.POINTER(C.c_double), _vp]),
    "wb_kmeans_accumulate_dev": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp]),
    "wb_kmeans_update_dev": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int64, C.POINTER(C.c_int64), _vp]),
    "wb_search": (C.c_int, [_vp, C.c_int64, _vp, C.c_int64, C.c_int64, _vp, _vp]),
    "wb_search_dev": (C.c_int, [_vp, C.c_int64, _vp, C.c_int64, C.c_int64, _vp, _vp, _vp]),
    "wb_filter_create_ids": (C.c_int, [_vp, C.c_int64, _vp, C.c_int, C.POINTER(_vp)]),
    "wb_filter_create_range": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int, C.POINTER(_vp)]),
    "wb_filter_count": (C.c_int64, [_vp]),
    "wb_filter_free": (C.c_int, [_vp]),
    "wb_search_filtered": (C.c_int, [_vp, _vp, C.c_int64, _vp, C.c_int64, C.c_int64, _vp, _vp]),
    "wb_search_filtered_dev": (C.c_int, [_vp, _vp, C.c_int64, _vp, C.c_int64, C.c_int64, _vp, _vp, _vp]),
    "wb_range_search": (C.c_int, [_vp, _vp, C.c_int64, _vp, C.c_float, C.c_int64, _vp, C.POINTER(_vp)]),
    "wb_range_search_dev": (C.c_int, [_vp, _vp, C.c_int64, _vp, C.c_float, C.c_int64, _vp, C.POINTER(_vp), _vp]),
    "wb_range_result_copy": (C.c_int, [_vp, _vp, _vp]),
    "wb_range_result_copy_dev": (C.c_int, [_vp, _vp, _vp, _vp]),
    "wb_range_result_free": (C.c_int, [_vp]),
    "wb_range_merge_dev": (C.c_int, [C.c_int, C.c_int64, C.c_int64, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "wb_exch_search_filtered": (C.c_int, [_vp, _vp, _vp, C.c_int64, _vp, C.c_int64, C.c_int64, _vp, _vp]),
    "wb_exch_search_filtered_dev": (C.c_int, [_vp, _vp, _vp, C.c_int64, _vp, C.c_int64, C.c_int64, _vp, _vp, _vp]),
    "wb_merge_topk_dev":(C.c_int, [C.c_int, C.c_int64, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp, _vp]),
    "wb_exch_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int64, C.POINTER(_vp)]),
    "wb_exch_local_handle": (C.c_int, [_vp, _vp]),
    "wb_exch_open_peers": (C.c_int, [_vp, _vp]),
    "wb_exch_merge_dev": (C.c_int, [_vp, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp, _vp]),
    "wb_exch_search": (C.c_int, [_vp, _vp, C.c_int64, _vp, C.c_int64, C.c_int64, _vp, _vp]),
    "wb_exch_search_dev": (C.c_int, [_vp, _vp, C.c_int64, _vp, C.c_int64, C.c_int64, _vp, _vp, _vp]),
    "wb_exch_launch_count": (C.c_int64, [_vp]),
    "wb_exch_status": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "wb_exch_free": (C.c_int, [_vp]),
    "wb_group_create": (C.c_int, [C.c_int, _vp, C.c_int64, C.c_int64, C.POINTER(_vp)]),
    "wb_group_search": (C.c_int, [_vp, _vp, C.c_int64, _vp, C.c_int64, C.c_int64, _vp, _vp]),
    "wb_group_search_dev": (C.c_int, [_vp, _vp, C.c_int64, _vp, C.c_int64, C.c_int64, _vp, _vp, _vp]),
    "wb_group_free": (C.c_int, [_vp]),
    "wb_reconstruct_batch": (C.c_int, [_vp, C.c_int64, _vp, _vp]),
    "wb_lookup_ids": (C.c_int, [_vp, C.c_int64, _vp, _vp]),
    "wb_export_rows": (C.c_int, [_vp, C.c_int64, C.c_int64, _vp, _vp, _vp]),
    "wb_ivf_add_preassigned": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp]),
    "wb_ivf_finalize": (C.c_int, [_vp]),
    "wb_ivf_list_offsets": (C.c_int, [_vp, _vp, C.POINTER(C.c_int)]),
    "wb_tar_scan": (C.c_int, [C.c_char_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "wb_tar_read": (C.c_int, [C.c_char_p, C.c_int64, C.c_int64, _vp, _vp, C.POINTER(C.c_int64)]),
    "wb_tf32_peak": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "wb_storage": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(C.c_int64)]),
    "wb_launch_count": (C.c_int64, [_vp]),
    "wb_ivf_fused_searches": (C.c_int64, [_vp]),
    "wb_scan_plan": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int, C.c_int64, _i32p]),
    "wb_phase_stamps": (C.c_int, [_vp, _vp, C.c_int]),
    "wb_gemm_stats": (C.c_int, [_vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "wb_flat_bf16_stats": (C.c_int, [_vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "wb_flat_image_bytes": (C.c_int64, [_vp]),
    "wb_set_timing": (C.c_int, [_vp, C.c_int]),
    "wb_last_scan_ms": (C.c_float, [_vp]),
    "wb_scan_ms_history": (C.c_int, [_vp, _f32p, C.c_int]),
}

_lib = None


def lib() -> C.CDLL:
    """Load libwiseb200.so once; raise (never fall back) if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C wise_b200/csrc`. wise_b200 has no CPU or PyTorch fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError here == header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().wb_last_error()
        raise RuntimeError((msg or b"unknown wise_b200 error").decode("utf-8", "replace"))


def ptr(a) -> int | None:
    """Address of a numpy array / torch tensor / None as a plain integer."""
    if a is None:
        return None
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    try:  # writable contiguous numpy array: the buffer protocol is twice as fast as ndarray.ctypes (3 pointers per search)
        return C.addressof(C.c_char.from_buffer(a))
    except (TypeError, ValueError):  # read-only, empty or strided: the slow, general way
        return a.ctypes.data
