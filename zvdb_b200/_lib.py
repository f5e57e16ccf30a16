"""ctypes binding of libzvdb_b200.so (the C ABI in include/zvdb_b200.h).

Loading fails loudly when the library is missing: there is no Python or CPU fallback for any
entry point.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ZVDB_B200_LIB points the binding at another build of the same library (A/B runs of kernel variants)
LIB_PATH = os.environ.get("ZVDB_B200_LIB") or os.path.join(_HERE, "lib", "libzvdb_b200.so")

OK, ERR_OOM, ERR_NODE_NOT_FOUND, ERR_DIM_MISMATCH, ERR_CUDA, ERR_INVALID, ERR_UNSUPPORTED = range(7)
METRIC_L2, METRIC_COSINE, METRIC_DOT = 0, 1, 2
STORAGE_F32, STORAGE_F16, STORAGE_SQ8 = 0, 1, 2
INVALID_ID = 0xFFFFFFFFFFFFFFFF

_u32, _u64, _i32, _i64, _vp = C.c_uint32, C.c_uint64, C.c_int, C.c_int64, C.c_void_p
_pf, _pu32, _pu64, _pi32 = C.POINTER(C.c_float), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)

# name -> (restype, argtypes); mirrors include/zvdb_b200.h one to one
SIGNATURES = {
    "zvdb_create": (_i32, [C.POINTER(_vp), _u32, _u32, _u32, _i32, _i32]),
    "zvdb_destroy": (None, [_vp]),
    "zvdb_set_level_seed": (_i32, [_vp, _u64]),
    "zvdb_insert": (_i32, [_vp, _pf, _u32]),
    "zvdb_insert_batch": (_i32, [_vp, _pf, _u64, _u32, _pi32]),
    "zvdb_insert_typed": (_i32, [_vp, _vp, _u32, _i32]),
    "zvdb_insert_batch_typed": (_i32, [_vp, _vp, _u64, _u32, _i32, _pi32]),
    "zvdb_search_typed": (_i32, [_vp, _vp, _u32, _i32, _u32, _pu64, _pf, _pu32]),
    "zvdb_search_batch_typed": (_i32, [_vp, _vp, _u64, _u32, _i32, _u32, _u32, _vp, _vp, _vp]),
    "zvdb_dtype": (_i32, [_vp]),
    "zvdb_get_point_typed": (_vp, [_vp, _u64]),
    "zvdb_count": (_u64, [_vp]),
    "zvdb_dim": (_u32, [_vp]),
    "zvdb_max_level": (_u32, [_vp]),
    "zvdb_entry_point": (_i64, [_vp]),
    "zvdb_get_point": (_pf, [_vp, _u64]),
    "zvdb_get_connections": (_i32, [_vp, _u64, _u32, _pu64, _u32, _pu32]),
    "zvdb_node_level": (C.c_int32, [_vp, _u64]),
    "zvdb_export_layer": (_i32, [_vp, _u32, _pu32, _pu32]),
    "zvdb_load_graph": (_i32, [_vp, _pf, _u64, _u32, _pu64, _pu32, _u64]),
    "zvdb_build_from_candidates": (_i32, [_vp, _pf, _u64, _u32, _vp, _u32, _i32]),
    "zvdb_append_batch": (_i32, [_vp, _pf, _u64, _u32, _u32, _u32]),
    "zvdb_set_descent": (_i32, [_vp, _i32]),
    "zvdb_descent_start": (_i64, [_vp]),
    "zvdb_set_storage": (_i32, [_vp, _i32]),
    "zvdb_storage": (_i32, [_vp]),
    "zvdb_storage_codebook": (_i32, [_vp, _pf, _pf, _u32]),
    "zvdb_export_upper_layers": (_i32, [_vp, _vp, _vp, _vp, _pu64]),
    "zvdb_load_upper_layers": (_i32, [_vp, _vp, _vp, _u64, _u64]),
    "zvdb_save": (_i32, [_vp, C.c_char_p]),
    "zvdb_load": (_i32, [_vp, C.c_char_p]),
    "zvdb_alloc_host": (_vp, [C.c_size_t]),
    "zvdb_free_host": (None, [_vp]),
    "zvdb_search": (_i32, [_vp, _pf, _u32, _u32, _pu64, _pf, _pu32]),
    "zvdb_search_batch": (_i32, [_vp, _vp, _u64, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp]),
    "zvdb_search_batch_device": (_i32, [_vp, _vp, _u64, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _u64, _u64, _vp]),
    "zvdb_bruteforce_knn": (_i32, [_vp, _vp, _u64, _u32, _u32, _vp, _vp, _vp]),
    "zvdb_bruteforce_knn_device": (_i32, [_vp, _vp, _u64, _u32, _vp, _vp, _vp, _u64, _u64, _vp]),
    "zvdb_sync_device": (_i32, [_vp]),
    "zvdb_set_kernel_variant": (_i32, [_vp, _u32]),
    "zvdb_kernel_launches": (_u64, [_vp]),
    "zvdb_merge_topk_device": (_i32, [_vp, _vp, _vp, _u32, _u64, _u32, _vp, _vp, _vp, _vp]),
    "zvdb_shard_block_bytes": (_u64, [_u64, _u32]),
    "zvdb_search_batch_packed_device": (_i32, [_vp, _vp, _u64, _u32, _u32, _vp, _u64, _u64, _vp]),
    "zvdb_merge_topk_packed_device": (_i32, [_vp, _u32, _u64, _u32, _vp, _vp, _vp, _vp]),
    "zvdb_exchange_create": (_i32, [C.POINTER(_vp), _i32, _u32, _u32, _u64, _u32]),
    "zvdb_exchange_create_host": (_i32, [C.POINTER(_vp), _i32, _u32, _u32, _u64, _u32, _u32]),
    "zvdb_search_batch_exchange_host": (_i32, [_vp, _vp, _vp, _u64, _u32, _u32, _u32, _vp, _vp, _vp, _vp]),
    "zvdb_exchange_ipc_handle": (_i32, [_vp, _vp]),
    "zvdb_exchange_open_peers": (_i32, [_vp, _vp]),
    "zvdb_exchange_destroy": (None, [_vp]),
    "zvdb_search_batch_exchange": (_i32, [_vp, _vp, _vp, _u64, _u32, _u32, _vp, _vp, _vp, _vp]),
    "zvdb_last_error": (C.c_char_p, []),
    "zvdb_version": (C.c_char_p, []),
}


class ZvdbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"zvdb_b200 error {code}: {msg}")
        self.code = code


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing. Build it with `python -m zvdb_b200.build` (needs nvcc). "
                "zvdb_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)   # AttributeError here = header and library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != OK:
        raise ZvdbError(rc, lib().zvdb_last_error().decode("utf-8", "replace"))
