"""ctypes binding of include/b200flat.h (the C-ABI boundary).  No torch types cross it.

The shared library is built in-tree by build.py (nvcc, sm_100a).  If it is missing this module
builds it; if that is impossible the import fails loudly -- there is no Python/CPU fallback.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200flat.so")
# diagnostics: B200FLAT_LIB=<path> loads another build of the library (same-box A/B runs of two kernel versions);
# entry points that build lacks are then skipped instead of failing the import
_LIB_OVERRIDE = os.environ.get("B200FLAT_LIB")
if _LIB_OVERRIDE:
    LIB_PATH = os.path.abspath(_LIB_OVERRIDE)

METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1
STORE_F32 = 0
STORE_BF16 = 1
MEM_HOST = 0
MEM_DEVICE = 1
ALGO_AUTO, ALGO_SCAN, ALGO_TENSOR = 0, 1, 2
POOL_CLS, POOL_MEAN = 0, 1

SEL_RANGE, SEL_BATCH, SEL_BITMAP = 1, 2, 3

OK, EINVAL, ENOGPU, ECUDA, EIO, EFORMAT, ENOMEM, ERANGE = 0, -1, -2, -3, -4, -5, -6, -7


class SearchParams(ctypes.Structure):
    _fields_ = [
        ("algo", ctypes.c_int32),
        ("scan_max_nq", ctypes.c_int32),
        ("slack", ctypes.c_int32),
        ("certify", ctypes.c_int32),
        ("id_offset", ctypes.c_int64),
        ("profile", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
    ]


class Selector(ctypes.Structure):
    """b2f_selector: a faiss ID selector as the filtered entry points take it."""
    _fields_ = [
        ("kind", ctypes.c_int32),
        ("negate", ctypes.c_int32),
        ("imin", ctypes.c_int64),
        ("imax", ctypes.c_int64),
        ("n", ctypes.c_int64),
        ("data", ctypes.c_void_p),
    ]


class Stats(ctypes.Structure):
    _fields_ = [
        ("launches", ctypes.c_int64),
        ("searches", ctypes.c_int64),
        ("fallback_queries", ctypes.c_int64),
        ("last_algo", ctypes.c_int32),
        ("last_kprime", ctypes.c_int32),
        ("last_main_ms", ctypes.c_float),
        ("last_total_ms", ctypes.c_float),
        ("last_main_launches", ctypes.c_int32),
        ("last_launches", ctypes.c_int32),
        ("bytes_rows", ctypes.c_int64),
        ("bytes_scan", ctypes.c_int64),
        ("overflow_queries", ctypes.c_int64),
        ("last_list_entries", ctypes.c_int64),
        ("prof_main_ms_sum", ctypes.c_double),
        ("prof_total_ms_sum", ctypes.c_double),
        ("prof_main_launches", ctypes.c_int64),
        ("prof_searches", ctypes.c_int64),
        ("rescued_queries", ctypes.c_int64),
        ("range_queries", ctypes.c_int64),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


_vp = ctypes.c_void_p
_i32 = ctypes.c_int32
_i64 = ctypes.c_int64
_u64 = ctypes.c_uint64

# name -> (restype, argtypes); mirrors include/b200flat.h one to one
PROTOTYPES = {
    "b2f_index_create": (ctypes.c_int, [_i32, _i32, _i32, _i32, ctypes.POINTER(_vp)]),
    "b2f_index_destroy": (ctypes.c_int, [_vp]),
    "b2f_index_reset": (ctypes.c_int, [_vp]),
    "b2f_index_reserve": (ctypes.c_int, [_vp, _i64]),
    "b2f_index_ntotal": (_i64, [_vp]),
    "b2f_index_d": (_i32, [_vp]),
    "b2f_index_metric": (_i32, [_vp]),
    "b2f_index_storage": (_i32, [_vp]),
    "b2f_index_device": (_i32, [_vp]),
    "b2f_index_add": (ctypes.c_int, [_vp, _i64, _vp, _i32, _vp]),
    "b2f_index_search": (ctypes.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _i32, _vp, ctypes.POINTER(SearchParams)]),
    "b2f_index_search_filtered": (ctypes.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _i32, _vp, ctypes.POINTER(SearchParams),
                                                 ctypes.POINTER(Selector)]),
    "b2f_index_range_search": (ctypes.c_int, [_vp, _i64, _vp, ctypes.c_float, _i32, _vp, ctypes.POINTER(SearchParams),
                                              ctypes.POINTER(_vp)]),
    "b2f_index_range_search_filtered": (ctypes.c_int, [_vp, _i64, _vp, ctypes.c_float, _i32, _vp, ctypes.POINTER(SearchParams),
                                                       ctypes.POINTER(Selector), ctypes.POINTER(_vp)]),
    "b2f_range_result_lims": (ctypes.c_int, [_vp, ctypes.POINTER(_i64)]),
    "b2f_range_result_fetch": (ctypes.c_int, [_vp, _vp, _vp, _i32, _vp]),
    "b2f_range_result_info": (ctypes.c_int, [_vp, ctypes.POINTER(_i64)]),
    "b2f_range_result_destroy": (ctypes.c_int, [_vp]),
    "b2f_index_remove_ids": (ctypes.c_int, [_vp, _i64, _vp, ctypes.POINTER(_i64)]),
    "b2f_index_remove_range": (ctypes.c_int, [_vp, _i64, _i64, ctypes.POINTER(_i64)]),
    "b2f_index_reconstruct":(ctypes.c_int, [_vp, _i64, _i64, _vp, _i32, _vp]),
    "b2f_index_write": (ctypes.c_int, [_vp, ctypes.c_char_p]),
    "b2f_index_read": (ctypes.c_int, [ctypes.c_char_p, _i32, _i32, ctypes.POINTER(_vp)]),
    "b2f_merge_topk_strided": (ctypes.c_int, [_i32, _i64, _i64, _i32, _vp, _vp, _i64, _vp, _vp, _i32, _vp]),
    "b2f_merge_range_strided": (ctypes.c_int, [_i64, _i32, _vp, _vp, _vp, _i64, _vp, _vp, _i32, _vp]),
    "b2f_exchange_create": (ctypes.c_int, [_i32, _i32, _i32, _i64, ctypes.POINTER(_vp), _vp]),
    "b2f_exchange_connect": (ctypes.c_int, [_vp, _vp]),
    "b2f_exchange_slot_bytes": (_i64, [_vp]),
    "b2f_exchange_merge": (ctypes.c_int, [_vp, _vp, _i64, _i32, _i64, _i64, _i64, _vp, _vp, _vp]),
    "b2f_exchange_search": (ctypes.c_int, [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, ctypes.POINTER(SearchParams)]),
    "b2f_exchange_destroy": (ctypes.c_int, [_vp]),
    "b2f_pool_normalize": (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _i32, _i32, _vp, _i32, _vp]),
    "b2f_index_add_pooled": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i64, _i32, _i32, _vp]),
    "b2f_index_search_pooled": (ctypes.c_int, [_vp, _vp, _vp, _i64, _i64, _i32, _i32, _i64, _vp, _vp, _vp, ctypes.POINTER(SearchParams)]),
    "b2f_synth_rows": (ctypes.c_int, [_u64, _i64, _i64, _i32, _i32, _vp, _i32, _vp]),
    "b2f_index_add_synth": (ctypes.c_int, [_vp, _u64, _i64, _i64, _i32]),
    "b2f_plan_describe": (ctypes.c_int, [_i64, _i64, _i32, _i64, _i32, ctypes.POINTER(_i32)]),
    "b2f_plan_unit_work": (ctypes.c_int, [_i32, _i32, _i32, _i64, _i32, _i32, ctypes.POINTER(_i32), ctypes.POINTER(_i64), _i64,
                                          ctypes.POINTER(_i32)]),
    "b2f_remove_plan": (ctypes.c_int, [_i64, _i64, _vp, _i64, _vp, ctypes.POINTER(_i64), _vp, _vp, _i64, ctypes.POINTER(_i64)]),
    "b2f_index_stats": (ctypes.c_int, [_vp, ctypes.POINTER(Stats)]),
    "b2f_last_error": (ctypes.c_char_p, []),
    "b2f_version": (ctypes.c_int, []),
    "b2f_device_count": (ctypes.c_int, []),
}

_lib = None


def load():
    """Load (building first if needed) libb200flat.so and attach prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build  # nvcc build; raises if nvcc is missing
        _build.build()
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover - loud failure, never a fallback
        raise ImportError(f"the CUDA extension {LIB_PATH} could not be loaded: {e}") from e
    for name, (res, args) in PROTOTYPES.items():
        if _LIB_OVERRIDE and not hasattr(lib, name):
            continue
        fn = getattr(lib, name)  # AttributeError = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    msg = load().b2f_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


class B200FlatError(RuntimeError):
    """A C-ABI call failed (surfaces like faiss's C++ exceptions: RuntimeError)."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"b200flat error {code}: {msg}")
        self.code = code


def check(rc: int):
    if rc != OK:
        raise B200FlatError(rc, last_error())
