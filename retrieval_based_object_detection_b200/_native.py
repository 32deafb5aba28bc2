"""ctypes binding of librbod.so -- the C ABI declared in include/rbod.h.

There is no CPU implementation behind this module: if the shared library is missing or a call
fails, an exception is raised.  Build it with ``python __graft_entry__.py build`` (or
``make -C retrieval_based_object_detection_b200/csrc``).
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RBOD_LIBRARY") or os.path.join(_HERE, "librbod.so")   # override: another build of the same ABI

RBOD_OK = 0
RBOD_E_IO = -5
RBOD_E_NOMEM = -12
RBOD_E_INVAL = -22
RBOD_E_RANGE = -34
RBOD_E_OVERFLOW = -75
RBOD_E_UNSUPPORTED = -95

RBOD_F32, RBOD_BF16, RBOD_F16 = 0, 1, 2
RBOD_COSINE, RBOD_DOT, RBOD_EUCLID, RBOD_MANHATTAN = 0, 1, 2, 3
RBOD_UPSERT_RAW = 1
DELEGATE_KINDS = {"average": 0, "centroid": 1, "weighted": 2, "medoid": 3}

DTYPES = {"f32": RBOD_F32, "fp32": RBOD_F32, "float32": RBOD_F32, "bf16": RBOD_BF16, "bfloat16": RBOD_BF16,
          "f16": RBOD_F16, "fp16": RBOD_F16, "float16": RBOD_F16}
METRICS = {"cosine": RBOD_COSINE, "dot": RBOD_DOT, "euclid": RBOD_EUCLID, "manhattan": RBOD_MANHATTAN}
# distances (smaller = closer): search scores ascend, out_scores64 carries the ordering key (-d^2 / -d)
DISTANCE_METRICS = ("euclid", "manhattan")


class GalleryInfo(ctypes.Structure):
    _fields_ = [("dim", ctypes.c_int32), ("dim_padded", ctypes.c_int32), ("dtype", ctypes.c_int32),
                ("metric", ctypes.c_int32), ("device", ctypes.c_int32), ("coop_refusals", ctypes.c_int32),
                ("rows", ctypes.c_int64), ("capacity", ctypes.c_int64), ("bytes_device", ctypes.c_int64),
                ("max_row_norm", ctypes.c_float), ("max_row_dev", ctypes.c_float)]


class SearchStats(ctypes.Structure):
    _fields_ = [("queries", ctypes.c_int64), ("fallback_queries", ctypes.c_int64), ("k3_launches", ctypes.c_int64),
                ("total_launches", ctypes.c_int64), ("candidates", ctypes.c_int32), ("slices", ctypes.c_int32),
                ("max_eps", ctypes.c_float), ("k3_ms", ctypes.c_float), ("sweep_queries", ctypes.c_int64),
                ("presample_retries", ctypes.c_int64)]


class RbodError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"librbod error {code}: {message}")
        self.code = code


_P = ctypes.c_void_p
_I64 = ctypes.c_int64
_I32 = ctypes.c_int32

# name -> (restype, argtypes); kept in one table so tests can check it against include/rbod.h
SIGNATURES = {
    "rbod_last_error": (ctypes.c_char_p, []),
    "rbod_abi_version": (ctypes.c_int, []),
    "rbod_create": (ctypes.c_int, [_I32, _I32, _I32, _I64, _I32, ctypes.POINTER(_P)]),
    "rbod_destroy": (ctypes.c_int, [_P]),
    "rbod_count": (_I64, [_P]),
    "rbod_info": (ctypes.c_int, [_P, ctypes.POINTER(GalleryInfo)]),
    "rbod_truncate": (ctypes.c_int, [_P, _I64]),
    "rbod_set_option": (ctypes.c_int, [_P, ctypes.c_char_p, _I64]),
    "rbod_upsert": (ctypes.c_int, [_P, _P, _I64, _P, _P, _I32, _P]),
    "rbod_get_rows": (ctypes.c_int, [_P, _P, _I64, _P, _P]),
    "rbod_l2norm_pack": (ctypes.c_int, [_P, _I64, _I32, _I32, _P, _I64, _P, _P]),
    "rbod_segment_mean": (ctypes.c_int, [_P, _P, _P, _I64, _P, _P]),
    "rbod_segment_sums": (ctypes.c_int, [_P, _P, _P, _I64, _P, _P]),
    "rbod_segment_finish": (ctypes.c_int, [_P, _P, _I64, _I32, _I32, _P, _P]),
    "rbod_segment_delegates": (ctypes.c_int, [_P, _I32, _P, _P, _I64, ctypes.c_double, _P, _P, _P]),
    "rbod_search": (ctypes.c_int, [_P, _P, _I64, _I32, _P, _P, _P, _P, ctypes.POINTER(SearchStats), _P]),
    "rbod_search_masks": (ctypes.c_int, [_P, _P, _I64, _I32, _P, _I32, _P, _P, _P, _P, ctypes.POINTER(SearchStats), _P]),
    "rbod_recommend": (ctypes.c_int, [_P, _P, _I64, _P, _P, _I64, _I32, _P, _I32, _P, _P, _P, _P,
                                      ctypes.POINTER(SearchStats), _P]),
    "rbod_discover": (ctypes.c_int, [_P, _P, _I64, _P, _P, _I64, _I32, _P, _I32, _P, _P, _P, _P,
                                     ctypes.POINTER(SearchStats), _P]),
    "rbod_search_mmr": (ctypes.c_int, [_P, _P, _I64, _I32, _I32, _P, _P, _P, _I32, _P, _P, _P, _P,
                                       ctypes.POINTER(SearchStats), _P]),
    "rbod_merge_topk": (ctypes.c_int, [_P, _P, _I32, _I64, _I32, _P, _P, _P, _P]),
    "rbod_merge_topk_packed": (ctypes.c_int, [_P, _P, _I32, _I64, _I32, _P, _P, _P, _P]),
    "rbod_search_begin": (ctypes.c_int, [_P, _P, _I64, _I32, _I32, _P, _P, ctypes.POINTER(SearchStats), _P]),
    "rbod_global_cut": (ctypes.c_int, [_P, _I32, _I64, _I32, _I32, _P, _P]),
    "rbod_search_end": (ctypes.c_int, [_P, _P, _I64, _I32, _P, _P, _P, ctypes.POINTER(SearchStats), _P]),
    "rbod_merge_topk_certified": (ctypes.c_int, [_P, _P, _I32, _I64, _I32, _P, _P, _P, _P, _P, _P]),
    "rbod_last_k3_ms": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_float)]),
    "rbod_debug_scores": (ctypes.c_int, [_P, _P, _I64, _P, _P]),
    "rbod_debug_profile": (ctypes.c_int, [_P, ctypes.POINTER(_I64)]),
    "rbod_debug_plan": (ctypes.c_int, [_I32, _I64, _I64, _I32, _I32, _I32, _I32, ctypes.POINTER(_I64)]),
}

_lib = None


def load():
    """Loads librbod.so (once).  Raises ImportError with build instructions if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run `python __graft_entry__.py build` "
            "(needs nvcc; targets sm_100a). There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = ABI mismatch, deliberately loud
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.rbod_abi_version() != 1:
        raise ImportError(f"librbod.so ABI version {lib.rbod_abi_version()} != 1")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != RBOD_OK:
        msg = load().rbod_last_error()
        raise RbodError(rc, msg.decode("utf-8", "replace") if msg else "")
