"""ctypes binding of ``libmlvindex.so`` (C ABI in ``include/mlv_index.h``).

The library is built in-tree (``mlvectordb_b200/csrc/Makefile`` -> ``mlvectordb_b200/libmlvindex.so``)
for sm_100a.  There is no CPU fallback anywhere in this package: a missing library raises
``ImportError`` on first use and a missing GPU raises ``RuntimeError`` from
``mlv_index_create`` (status ``MLV_E_NO_DEVICE``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmlvindex.so")

MLV_OK = 0
MLV_E_INVALID, MLV_E_CUDA, MLV_E_NOMEM, MLV_E_UNSUPPORTED, MLV_E_NO_DEVICE = 1, 2, 3, 4, 5
MLV_MAX_K = 1024
METRIC_CODE = {"l2": 0, "ip": 1, "cosine": 2}
ABI_VERSION = 6


class IndexInfo(C.Structure):
    _fields_ = [
        ("rows", C.c_uint64),
        ("live", C.c_uint64),
        ("capacity", C.c_uint64),
        ("row_base", C.c_uint64),
        ("device_bytes", C.c_uint64),
        ("dim", C.c_uint32),
        ("ld", C.c_uint32),
        ("metric", C.c_int32),
        ("device", C.c_int32),
    ]


class GemmStats(C.Structure):
    _fields_ = [
        ("gemm_ms", C.c_double),
        ("gemm_launches_timed", C.c_uint64),
        ("searches", C.c_uint64),
        ("queries", C.c_uint64),
        ("fallback_queries", C.c_uint64),
        ("rounds", C.c_uint64),
        ("fast_queries", C.c_uint64),
        ("gathered_searches", C.c_uint64),
        ("half_queries", C.c_uint64),
        ("mispredicted_queries", C.c_uint64),
        ("half_scan_queries", C.c_uint64),
        ("half_scan_uncertified", C.c_uint64),
        ("q8_scan_queries", C.c_uint64),
        ("q8_scan_uncertified", C.c_uint64),
    ]


class HalfScanDebug(C.Structure):
    """``mlv_half_scan_debug_t``"""
    _fields_ = [
        ("delta_rel", C.c_float),
        ("scale", C.c_float),
        ("q_norm2", C.c_float),
        ("max_norm2", C.c_float),
        ("x_unscale", C.c_float),
        ("q_unscale", C.c_float),
        ("overflow", C.c_uint32),
        ("consumers", C.c_uint32),
    ]


class Q8ScanDebug(C.Structure):
    """``mlv_q8_scan_debug_t``"""
    _fields_ = [
        ("delta", C.c_float),
        ("q_norm2", C.c_float),
        ("q_scale", C.c_float),
        ("max_norm2", C.c_float),
        ("e_max", C.c_float),
        ("ld8", C.c_uint32),
    ]


class GemmRoundsCfg(C.Structure):
    """``mlv_gemm_rounds_cfg_t``"""
    _fields_ = [
        ("passes", C.c_uint32),
        ("bn", C.c_uint32),
        ("max_ctas", C.c_uint32),
        ("cap", C.c_uint32),
        ("kprime", C.c_uint32),
        ("n_rounds", C.c_uint32),
        ("round_end", C.POINTER(C.c_uint32)),
        ("round_jrank", C.POINTER(C.c_uint32)),
    ]


class Predicate(C.Structure):
    """``mlv_predicate_t``"""
    _fields_ = [("column", C.c_uint32), ("op", C.c_int32), ("a", C.c_int32), ("b", C.c_int32)]


MAX_COLUMNS, MAX_PREDICATES = 16, 8
MAX_GROUP_K = 32
COLUMN_MISSING = -(2 ** 31)
PRED_OPS = {"==": 0, "!=": 1, "<": 2, "<=": 3, ">": 4, ">=": 5, "between": 6}

_f32p = C.POINTER(C.c_float)
_i64p = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)
_h = C.c_void_p

# name -> (restype, argtypes): every symbol include/mlv_index.h declares
SIGNATURES = {
    "mlv_abi_version": (C.c_int, []),
    "mlv_device_count": (C.c_int, []),
    "mlv_status_string": (C.c_char_p, [C.c_int]),
    "mlv_last_error": (C.c_char_p, [_h]),
    "mlv_index_create": (C.c_int, [C.c_uint32, C.c_int, C.c_uint64, C.c_int, C.POINTER(_h)]),
    "mlv_index_destroy": (C.c_int, [_h]),
    "mlv_index_set_row_base": (C.c_int, [_h, C.c_uint64]),
    "mlv_index_add": (C.c_int, [_h, C.c_void_p, C.c_uint64, _u64p]),
    "mlv_index_add_device": (C.c_int, [_h, C.c_void_p, C.c_uint64, _u64p]),
    "mlv_index_add_synthetic": (C.c_int, [_h, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, _u64p]),
    "mlv_index_mark_deleted": (C.c_int, [_h, C.c_void_p, C.c_uint64, _u64p]),
    "mlv_index_compact": (C.c_int, [_h, C.c_void_p, _u64p]),
    "mlv_index_clear": (C.c_int, [_h]),
    "mlv_index_search": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mlv_index_search_device": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "mlv_index_range_search": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_float, C.c_void_p, C.c_uint64, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "mlv_index_range_search_device": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_float, C.c_void_p, C.c_uint64, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_void_p]),
    "mlv_index_order_pairs_device": (C.c_int, [_h, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mlv_index_get_rows": (C.c_int, [_h, C.c_void_p, C.c_uint64, C.c_void_p]),
    "mlv_index_info": (C.c_int, [_h, C.POINTER(IndexInfo)]),
    "mlv_merge_topk": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    "mlv_index_set_timing": (C.c_int, [_h, C.c_int]),
    "mlv_index_scan_time_ms": (C.c_int, [_h, C.POINTER(C.c_double), _u64p]),
    "mlv_index_set_tuning": (C.c_int, [_h, C.c_char_p, C.c_int]),
    "mlv_index_kernel_launches": (C.c_int, [_h, _u64p]),
    "mlv_index_debug_timeline": (C.c_int, [_h, _u64p, C.c_uint32, _u32p]),
    "mlv_filter_create": (C.c_int, [_h, C.c_void_p, C.c_uint64, C.POINTER(_h)]),
    "mlv_filter_passing": (C.c_int, [_h, _u64p]),
    "mlv_filter_destroy": (C.c_int, [_h]),
    "mlv_index_set_filter": (C.c_int, [_h, _h]),
    "mlv_filter_get_bitmap": (C.c_int, [_h, C.c_void_p, C.c_uint64]),
    "mlv_filter_create_where": (C.c_int, [_h, C.POINTER(Predicate), C.c_uint32, C.POINTER(_h)]),
    "mlv_index_set_column": (C.c_int, [_h, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint64]),
    "mlv_index_set_column_device": (C.c_int, [_h, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint64]),
    "mlv_index_get_column": (C.c_int, [_h, C.c_uint32, C.c_uint64, C.c_uint64, C.c_void_p]),
    "mlv_index_search_grouped": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p]),
    "mlv_index_search_grouped_device": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mlv_format_f32_json": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, _u64p]),
    "mlv_index_export_rows": (C.c_int, [_h, C.c_uint64, C.c_uint64, C.c_void_p]),
    "mlv_index_export_live": (C.c_int, [_h, C.c_void_p, C.c_uint64]),
    "mlv_index_import_rows": (C.c_int, [_h, C.c_void_p, C.c_uint64, C.c_void_p, _u64p]),
    "mlv_exchange_create": (C.c_int, [C.c_int, C.c_uint32, C.c_uint32, C.POINTER(_h), C.c_void_p]),
    "mlv_exchange_connect": (C.c_int, [_h, C.c_void_p]),
    "mlv_exchange_check": (C.c_int, [_h]),
    "mlv_exchange_set_timeout_ms": (C.c_int, [_h, C.c_uint32]),
    "mlv_exchange_destroy": (C.c_int, [_h]),
    "mlv_index_attach_exchange": (C.c_int, [_h, _h, C.c_void_p]),
    "mlv_index_exchange_supported": (C.c_int, [_h, C.c_uint32]),
    "mlv_index_search_exchange_device": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_void_p]),
    "mlv_index_search_exchange": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mlv_index_range_exchange_supported": (C.c_int, [_h]),
    "mlv_index_range_search_exchange_device": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                                         C.c_void_p, C.c_void_p]),
    "mlv_index_range_search_exchange": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_float, C.c_void_p, C.c_uint64, C.c_void_p,
                                                  C.c_void_p, C.c_void_p]),
    "mlv_index_submit": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, _u32p]),
    "mlv_index_collect": (C.c_int, [_h, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mlv_index_gemm_stats": (C.c_int, [_h, C.POINTER(GemmStats)]),
    "mlv_index_debug_gemm": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_void_p]),
    "mlv_index_debug_half_scan": (C.c_int, [_h, C.c_void_p, C.c_void_p, C.POINTER(HalfScanDebug)]),
    "mlv_index_debug_q8_scan": (C.c_int, [_h, C.c_void_p, C.c_void_p, C.POINTER(Q8ScanDebug)]),
    "mlv_index_debug_gemm_rounds": (C.c_int, [_h, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.POINTER(GemmRoundsCfg),
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _u64p]),
}

_lib = None


def lib() -> C.CDLL:
    """Load the C-ABI library; raise loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make -C mlvectordb_b200/csrc` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)       # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if L.mlv_abi_version() != ABI_VERSION:
            raise ImportError(f"libmlvindex.so ABI {L.mlv_abi_version()} != binding ABI {ABI_VERSION}; rebuild")
        _lib = L
    return _lib


def format_f32_json(values) -> bytes:
    """``mlv_format_f32_json``: fp32 values -> b"[v0,v1,...]" (shortest round-trip text), C speed."""
    import numpy as np
    v = np.ascontiguousarray(values, dtype=np.float32).reshape(-1)
    buf = C.create_string_buffer(16 * v.shape[0] + 2)
    n = C.c_uint64()
    check(lib().mlv_format_f32_json(v.ctypes.data, v.shape[0], buf, len(buf), C.byref(n)))
    return buf.raw[: n.value]


class MlvError(RuntimeError):
    """RuntimeError so that callers' ``except RuntimeError`` patterns (reference index.py:112) still apply."""

    def __init__(self, status: int, detail: str = ""):
        self.status = status
        text = lib().mlv_status_string(status).decode()
        super().__init__(f"mlv status {status} ({text})" + (f": {detail}" if detail else ""))


def check(status: int, handle=None) -> None:
    if status != MLV_OK:
        detail = ""
        if handle:
            detail = lib().mlv_last_error(handle).decode(errors="replace")
        raise MlvError(status, detail)
