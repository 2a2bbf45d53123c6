"""ctypes binding of the C ABI declared in include/rass_b200.h.

The shared library is built in-tree by ``python -m rassengine_b200.build`` (``__graft_entry__.build()``).
There is no CPU fallback: a missing library is an ImportError-like failure at first use, and every compute
entry point fails with RASS_E_CUDA when no sm_100 device is present.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librass_b200.so")

RASS_OK = 0
RASS_E_INVALID, RASS_E_OOM, RASS_E_CUDA, RASS_E_NCCL, RASS_E_NOTFOUND, RASS_E_UNSUPPORTED, RASS_E_AGAIN = \
    -1, -2, -3, -4, -5, -6, -7
ERR_NAMES = {-1: "RASS_E_INVALID", -2: "RASS_E_OOM", -3: "RASS_E_CUDA", -4: "RASS_E_NCCL", -5: "RASS_E_NOTFOUND",
             -6: "RASS_E_UNSUPPORTED", -7: "RASS_E_AGAIN"}
METRIC_COSINE, METRIC_L2 = 0, 1
KEEP_FP32, BF16_ONLY, NO_INT8_SHADOW = 1, 2, 4
PATH_AUTO, PATH_STREAM, PATH_UMMA, PATH_EXACT, PATH_GEMM, PATH_UMMA8 = 0, 1, 2, 3, 4, 5
OPT_PATH, OPT_STREAM, OPT_KNN_PREFILTER, OPT_HYBRID_ORDERED, OPT_HYBRID_MAXSCORE, OPT_ASYNC_OVERLAP, \
    OPT_SCAN_RESERVE_SMS = 1, 2, 3, 4, 5, 6, 7
PATH_HYBRID_ORDER_FREE = 0x100


class RassStats(C.Structure):
    _fields_ = [("scan_ms", C.c_double), ("finish_ms", C.c_double), ("total_ms", C.c_double),
                ("rows_scanned", C.c_int64), ("bytes_streamed", C.c_int64), ("n_queries", C.c_int32),
                ("n_certified", C.c_int32), ("n_fallback", C.c_int32), ("path", C.c_int32), ("passes", C.c_int32),
                ("launches", C.c_int32), ("max_candidates", C.c_int32), ("n_retried", C.c_int32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class RassError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


_P = C.c_void_p
# name -> (restype, argtypes); every symbol include/rass_b200.h declares
PROTOTYPES = {
    "rass_version": (C.c_char_p, []),
    "rass_last_error": (C.c_char_p, [_P]),
    "rass_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int64, C.c_uint32, C.POINTER(_P)]),
    "rass_create_sharded": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int64, C.c_uint32,
                                      C.POINTER(_P)]),
    "rass_destroy": (C.c_int, [_P]),
    "rass_set_option": (C.c_int, [_P, C.c_int, C.c_int64]),
    "rass_set_row_base": (C.c_int, [_P, C.c_int64]),
    "rass_append": (C.c_int, [_P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "rass_append_dev": (C.c_int, [_P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "rass_overwrite": (C.c_int, [_P, C.c_int64, _P]),
    "rass_tombstone": (C.c_int, [_P, C.c_int64]),
    "rass_count": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "rass_rows": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "rass_store_info": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "rass_read_rows": (C.c_int, [_P, C.c_int64, C.c_int64, _P]),
    "rass_read_rows_list": (C.c_int, [_P, _P, C.c_int64, _P]),
    "rass_set_row_filter_rows": (C.c_int, [_P, _P, C.c_int64, C.c_int64]),
    "rass_search_knn": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P, C.POINTER(RassStats)]),
    "rass_search_knn_dev": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P, C.POINTER(RassStats)]),
    "rass_search_knn_dev_async": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P, C.c_int, _P]),
    "rass_search_knn_dev_wait": (C.c_int, [_P, C.c_int, C.POINTER(RassStats)]),
    "rass_async_join": (C.c_int, [_P, C.c_int, _P]),
    "rass_merge_topk_dev": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "rass_merge_scores_dev": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "rass_bm25_build": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, C.c_int64, C.c_int64, C.c_int64, _P]),
    "rass_search_hybrid": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_float, C.c_float, C.c_int, _P, _P,
                                     C.POINTER(RassStats)]),
    "rass_search_hybrid_weighted": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, C.c_float, C.c_int, _P, _P,
                                              C.POINTER(RassStats)]),
    "rass_bm25_build_fields": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, C.c_int]),
    "rass_text_add_rows": (C.c_int, [_P, C.c_int, _P, C.c_int64, _P, _P]),
    "rass_text_add_rows_dev": (C.c_int, [_P, C.c_int, _P, C.c_int64, _P, _P]),
    "rass_text_commit": (C.c_int, [_P, _P, C.c_int, C.c_int64]),
    "rass_text_omit_norms": (C.c_int, [_P, C.c_int, C.c_int]),
    "rass_text_size": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                 C.POINTER(C.c_int)]),
    "rass_text_export": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "rass_text_stats": (C.c_int, [_P, _P, _P, _P]),
    "rass_fuse_hybrid": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.c_float, _P, _P, C.c_float, C.c_int, _P, _P]),
    "rass_fuse_hybrid_dev": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.c_float, _P, _P, C.c_float, C.c_int, _P, _P, _P]),
    "rass_text_set_vocab": (C.c_int, [_P, C.c_char_p, _P, C.c_int64]),
    "rass_fuzzy_expand": (C.c_int, [_P, C.c_char_p, C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int64, _P, _P,
                                    C.POINTER(C.c_int64)]),
    "rass_set_row_filter": (C.c_int, [_P, _P, C.c_int64]),
    "rass_search_knn_filtered": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P, _P, _P]),
    "rass_search_hybrid_filtered": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, C.c_float, C.c_float, C.c_int, _P, _P,
                                              C.c_int, _P, _P, C.POINTER(RassStats)]),
    "rass_sync": (C.c_int, [_P]),
    "rass_last_stats": (C.c_int, [_P, C.POINTER(RassStats)]),
    "rass_save": (C.c_int, [_P, C.c_char_p]),
    "rass_load": (C.c_int, [_P, C.c_char_p]),
    "rass_debug_umma_scores": (C.c_int, [_P, _P, C.c_int, _P]),
    "rass_debug_gemm_scores": (C.c_int, [_P, _P, C.c_int, _P]),
    "rass_debug_umma8_scores": (C.c_int, [_P, _P, C.c_int, _P, _P, _P]),
}

_lib = None


def lib():
    """The loaded shared library (loads on first use; raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RassError(RASS_E_UNSUPPORTED, f"{LIB_PATH} is missing: run `python -m rassengine_b200.build` "
                            "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib
