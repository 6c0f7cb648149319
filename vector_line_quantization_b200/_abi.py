"""ctypes binding of lib/libvlq_b200.so (the C-ABI of include/vlq_b200.h).

The library is the product: if it is missing or cannot be loaded this module raises -- there is no CPU fallback.
All compute entry points take raw DEVICE pointers (ints here); `check()` maps non-zero return codes to VlqError.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libvlq_b200.so")

_p = C.c_void_p
_i = C.c_int
_l = C.c_int64
_z = C.c_size_t
_f = C.c_float

# name -> (restype, argtypes); kept in the order of include/vlq_b200.h
SIGNATURES = {
    "vlq_error_string": (C.c_char_p, [_i]),
    "vlq_version": (C.c_char_p, []),
    "vlq_launch_count": (C.c_uint64, []),
    "vlq_row_norms": (_i, [_p, _l, _i, _p, _p]),
    "vlq_l2_assign": (_i, [_p, _l, _i, _p, _p, _i, _i, _p, _p, _p]),
    "vlq_tc_supported": (_i, [_i, _i]),
    "vlq_tc_cent_pack_bytes": (_z, [_i, _i]),
    "vlq_tc_pack_centroids": (_i, [_p, _p, _i, _i, _f, _p, _p]),
    "vlq_l2_tc_workspace_bytes": (_z, [_l, _i, _i]),
    "vlq_l2_assign_tc": (_i, [_p, _l, _i, _p, _f, _i, _i, _p, _p, _p, _z, _p]),
    "vlq_tc_num_buckets": (_i, [_i]),
    "vlq_l2_distances_tc": (_i, [_p, _l, _i, _p, _f, _i, _p, _l, _p, _p, _z, _p]),
    "vlq_l2_bucket_min_tc": (_i, [_p, _l, _i, _p, _f, _i, _p, _p, _z, _p]),
    "vlq_l2_distances": (_i, [_p, _l, _i, _p, _p, _i, _p, _l, _p]),
    "vlq_select_rows": (_i, [_p, _l, _i, _l, _i, _p, _p, _p, _p]),
    "vlq_knn_graph_workspace_bytes": (_z, [_i, _i]),
    "vlq_knn_graph": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _z, _p]),
    "vlq_line_encode": (_i, [_p, _l, _i, _p, _p, _p, _p, _i, _p, _i, _p, _i, _p, _p, _p, _p, _p, _p, _p]),
    "vlq_lambda_quantize": (_i, [_p, _l, _p, _i, _p, _p]),
    "vlq_line_residual": (_i, [_p, _l, _i, _p, _p, _p, _p, _p, _i, _p, _p]),
    "vlq_build_lists_workspace_bytes": (_z, [_l, _l]),
    "vlq_build_lists": (_i, [_l, _i, _l, _p, _p, _p, _p, _p, _l, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _z, _p]),
    "vlq_remove_ids_workspace_bytes": (_z, [_l, _l]),
    "vlq_remove_ids_plan": (_i, [_l, _l, _p, _p, _l, _l, _p, _l, _p, _p, _z, _p]),
    "vlq_remove_ids_apply": (_i, [_l, _i, _l, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _z, _p]),
    "vlq_build_lists_aux": (_i, [_l, _i, _i, _l, _p, _p, _p, _p, _p, _p, _l, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p,
                                 _p, _p, _z, _p]),
    "vlq_remove_ids_apply_aux": (_i, [_l, _i, _i, _l, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _z, _p]),
    "vlq_lookup_ids": (_i, [_l, _p, _l, _p, _l, _p, _p, _p]),
    "vlq_decode_entries": (_i, [_l, _p, _l, _p, _p, _p, _p, _i, _i, _p, _p, _p, _i, _p, _i, _p, _p, _p]),
    "vlq_imi_decode_entries": (_i, [_l, _p, _p, _p, _p, _i, _i, _p, _p, _p, _i, _p, _p, _p]),
    "vlq_refine_encode": (_i, [_p, _l, _i, _p, _p, _p, _i, _p, _p, _p, _i, _p, _i, _p, _i, _p, _p, _p]),
    "vlq_refine_topk": (_i, [_p, _l, _i, _p, _i, _i, _l, _p, _p, _p, _p, _p, _i, _p, _p, _p, _i, _p, _i, _p, _i, _p, _p,
                             _p]),
    "vlq_refine_decode": (_i, [_l, _p, _l, _p, _p, _p, _p, _p, _i, _i, _p, _p, _p, _i, _p, _i, _p, _i, _p, _p, _p]),
    "vlq_filter_kappa": (_i, [_l, _p, _p, _l, _l, _p, _l, _p, _l, _i, _p, _p]),
    "vlq_filter_results": (_i, [_l, _i, _p, _p, _p]),
    "vlq_recompute_kappa": (_i, [_l, _l, _p, _p, _p, _p, _i, _p, _i, _p, _p, _i, _p, _p]),
    "vlq_select_lines": (_i, [_p, _l, _l, _p, _i, _p, _p, _i, _i, _p, _p, _p, _p]),
    "vlq_coarse_select_lines": (_i, [_p, _l, _l, _p, _i, _i, _i, _p, _p, _i, _i, _p, _p, _p, _p, _p]),
    "vlq_coarse_exact_supported": (_i, [_i, _i, _i, _i, _i]),
    "vlq_coarse_exact_preferred": (_i, [_i, _i, _i, _i, _i]),
    "vlq_coarse_select_lines_exact": (_i, [_p, _l, _i, _p, _p, _p, _i, _i, _i, _p, _p, _i, _i, _p, _p, _p, _p, _p]),
    "vlq_coarse_route": (_i, [_i, _i, _i, _i, _i, _i]),
    "vlq_coarse_lines_workspace_bytes": (_z, [_l, _i, _i, _i, _i, _i, _i]),
    "vlq_coarse_lines": (_i, [_p, _l, _i, _p, _p, _p, _f, _i, _i, _p, _p, _i, _i, _p, _p, _p, _p, _p, _z, _p]),
    "vlq_gather_candidates": (_i, [_p, _l, _i, _p, _p, _l, _p, _p]),
    "vlq_scan_topk_workspace_bytes": (_z, [_l, _i]),
    "vlq_scan_topk": (_i, [_p, _l, _i, _p, _i, _p, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _i, _i, _i, _p, _p, _p, _z, _p]),
    "vlq_range_workspace_bytes": (_z, [_l, _i, _i, _i]),
    "vlq_range_count": (_i, [_p, _l, _i, _p, _i, _p, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _i, _p, _f, _p, _p, _z, _p]),
    "vlq_range_gather": (_i, [_p, _l, _i, _p, _i, _p, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _i, _p, _f, _p, _p, _l, _l,
                              _p, _p, _p, _z, _p]),
    "vlq_line_encode_pq4": (_i, [_p, _l, _i, _p, _p, _p, _p, _i, _p, _i, _p, _i, _p, _p, _p, _p, _p, _p, _p]),
    "vlq_scan_topk_pq4": (_i, [_p, _l, _i, _p, _i, _p, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p, _i, _i, _i, _p, _p, _p,
                               _z, _p]),
    "vlq_range_count_pq4": (_i, [_p, _l, _i, _p, _i, _p, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _i, _p, _f, _p, _p, _z,
                                 _p]),
    "vlq_range_gather_pq4": (_i, [_p, _l, _i, _p, _i, _p, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _i, _p, _f, _p, _p, _l,
                                  _l, _p, _p, _p, _z, _p]),
    "vlq_decode_entries_pq4": (_i, [_l, _p, _l, _p, _p, _p, _p, _i, _i, _p, _p, _p, _i, _p, _i, _p, _p, _p]),
    "vlq_recompute_kappa_pq4": (_i, [_l, _l, _p, _p, _p, _p, _i, _p, _i, _p, _p, _i, _p, _p]),
    "vlq_merge_topk": (_i, [_p, _p, _i, _l, _i, _p, _p, _p]),
    "vlq_merge_topk_peers": (_i, [_p, _z, _z, _i, _l, _i, _p, _p, _p]),
    "vlq_gather_peer_slices": (_i, [_p, _i, _i, _p, _i, _l, _l, _p]),
    "vlq_km_update_workspace_bytes": (_z, [_l, _i]),
    "vlq_km_update": (_i, [_p, _l, _i, _p, _i, _p, _p, _p, _z, _p]),
    "vlq_copy_columns": (_i, [_p, _l, _l, _i, _i, _p, _p]),
    "vlq_imi_top_cells": (_i, [_p, _p, _p, _p, _l, _i, _i, _i, _p, _p, _p]),
    "vlq_imi_encode": (_i, [_p, _l, _i, _p, _p, _p, _p, _i, _p, _i, _p, _p, _p, _p]),
    "vlq_gather_rows": (_i, [_p, _i, _p, _l, _p, _p]),
    "vlq_u8_to_f32": (_i, [_p, _l, _p, _p]),
    "vlq_iota_i64": (_i, [_p, _l, _l, _p]),
    "vlq_i32_to_i64": (_i, [_p, _l, _p, _p]),
    "vlq_shift_ids": (_i, [_p, _l, _l, _p]),
    "vlq_device_count": (_i, [C.POINTER(_i)]),
    "vlq_set_device": (_i, [_i]),
    "vlq_get_device": (_i, [C.POINTER(_i)]),
    "vlq_mem_info": (_i, [C.POINTER(_z), C.POINTER(_z)]),
    "vlq_malloc": (_i, [C.POINTER(_p), _z]),
    "vlq_free": (_i, [_p]),
    "vlq_malloc_host": (_i, [C.POINTER(_p), _z]),
    "vlq_free_host": (_i, [_p]),
    "vlq_memcpy_h2d": (_i, [_p, _p, _z, _p]),
    "vlq_memcpy_d2h": (_i, [_p, _p, _z, _p]),
    "vlq_memcpy_d2d": (_i, [_p, _p, _z, _p]),
    "vlq_memset": (_i, [_p, _i, _z, _p]),
    "vlq_pointer_is_device": (_i, [_p]),
    "vlq_pointer_device": (_i, [_p, C.POINTER(_i)]),
    "vlq_enable_peer_access": (_i, [_i]),
    "vlq_stream_create": (_i, [C.POINTER(_p)]),
    "vlq_stream_destroy": (_i, [_p]),
    "vlq_stream_synchronize": (_i, [_p]),
    "vlq_stream_wait": (_i, [_p, _p]),
    "vlq_event_create": (_i, [_p]),
    "vlq_event_destroy": (_i, [_p]),
    "vlq_event_record": (_i, [_p, _p]),
    "vlq_stream_wait_event": (_i, [_p, _p]),
}


class VlqError(RuntimeError):
    def __init__(self, code, where):
        self.code = code
        msg = lib().vlq_error_string(code)
        super().__init__("%s failed: %s (code %d)" % (where, msg.decode() if msg else "?", code))


_lib = None


def lib():
    """Load (once) and return the CUDA library; raises if it is absent -- never falls back to a CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "%s is missing: build it with `python -m vector_line_quantization_b200.build` "
                "(the VLQ hot path has no CPU fallback)" % LIB_PATH)
        handle = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError here means header and library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(code, where="vlq call"):
    if code != 0:
        raise VlqError(code, where)


def call(name, *args):
    """Invoke a C-ABI function that returns an int status and raise on failure."""
    check(getattr(lib(), name)(*args), name)
