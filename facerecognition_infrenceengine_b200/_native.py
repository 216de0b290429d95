"""ctypes binding of libfrg.so (include/frg.h).  Thin by design: plain pointers and sizes.

The library is mandatory.  If it has not been built (``python -m
facerecognition_infrenceengine_b200.build``) importing this module raises; if it is built but no
CUDA device is present every compute call raises :class:`NativeError` - there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libfrg.so")

OK, ERR_INVALID, ERR_CUDA, ERR_NOMEM, ERR_UNSUPPORTED, ERR_STATE = range(6)
METRIC_COSINE, METRIC_EUCLIDEAN = 0, 1
VARIANT_AUTO, VARIANT_SCAN_F32, VARIANT_TC_EXACT, VARIANT_TC_BF16 = 0, 1, 2, 3
STORE_BF16_PLANE, STORE_RAW, STORE_BF16_ONLY = 1, 2, 4
ROWS_PRENORMALISED = 1
FIRST_STRICT, QUERY_PRENORMALISED = 1, 2
JOIN_SAME_TAG = 4
JOIN_SLAB_ROWS = 1024
CLUSTER_MAX_WINDOW = 16
XCHG_PUSH_ONLY, XCHG_MERGE_ONLY = 1, 2
MAX_K = 16

VARIANTS = {"auto": VARIANT_AUTO, "scan_f32": VARIANT_SCAN_F32, "tc_exact": VARIANT_TC_EXACT,
            "tc_bf16": VARIANT_TC_BF16}
METRICS = {"cosine": METRIC_COSINE, "euclidean": METRIC_EUCLIDEAN}


class NativeError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__("libfrg error %d: %s" % (code, message))
        self.code = code


class StoreStats(C.Structure):
    _fields_ = [("rows", C.c_int64), ("live", C.c_int64), ("capacity", C.c_int64),
                ("version", C.c_int64), ("bytes", C.c_int64), ("dim", C.c_int32),
                ("device", C.c_int32), ("flags", C.c_uint32), ("faults", C.c_uint32)]


class MatchParams(C.Structure):
    _fields_ = [("metric", C.c_int32), ("variant", C.c_int32), ("threshold", C.c_float),
                ("tenant", C.c_int32), ("row_offset", C.c_int64), ("flags", C.c_uint32),
                ("reserved", C.c_uint32)]


class Exchange(C.Structure):          # frg_exchange_t
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("peer_bufs", C.c_void_p),
                ("block_cap", C.c_int64), ("epoch", C.c_uint32), ("flags", C.c_uint32)]


class ExchangeStatus(C.Structure):    # frg_exchange_status_t
    _fields_ = [("code", C.c_int32), ("peer", C.c_int32), ("epoch", C.c_uint32), ("peer_epoch", C.c_uint32),
                ("nq", C.c_int32), ("k", C.c_int32), ("peer_nq", C.c_int32), ("peer_k", C.c_int32),
                ("slot", C.c_int32), ("reserved", C.c_int32)]


class ClusterRing(C.Structure):       # frg_cluster_ring_t
    _fields_ = [("members", C.c_void_p), ("len", C.c_void_p), ("head", C.c_void_p), ("capacity", C.c_int64),
                ("window", C.c_int32)]


# every symbol include/frg.h declares: (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    "frg_abi_version": (C.c_int, []),
    "frg_last_error": (C.c_char_p, []),
    "frg_device_count": (C.c_int, [C.POINTER(C.c_int32)]),
    "frg_store_create": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_uint32, C.POINTER(_P)]),
    "frg_store_destroy": (C.c_int, [_P]),
    "frg_store_reserve": (C.c_int, [_P, C.c_int64]),
    "frg_store_stats": (C.c_int, [_P, C.POINTER(StoreStats)]),
    "frg_store_upsert": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_uint32, _P]),
    "frg_store_upsert_host": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_uint32]),
    "frg_store_remove": (C.c_int, [_P, _P, C.c_int64, _P]),
    "frg_store_remove_host": (C.c_int, [_P, _P, C.c_int64]),
    "frg_store_compact": (C.c_int, [_P, _P]),
    "frg_store_read_host": (C.c_int, [_P, C.c_int64, C.c_int64, _P, _P]),
    "frg_store_fill_synthetic": (C.c_int, [_P, C.c_int64, C.c_int64, C.c_uint64, C.c_int32, _P]),
    "frg_match": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(MatchParams), _P, _P, _P, _P]),
    "frg_match_host": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(MatchParams), _P, _P, _P]),
    "frg_match_tenants": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(MatchParams), _P, _P, _P, _P, _P]),
    "frg_match_tenants_host": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(MatchParams), _P, _P, _P, _P]),
    "frg_first_match": (C.c_int, [_P, _P, C.c_int32, C.POINTER(MatchParams), _P, _P, _P]),
    "frg_first_match_host": (C.c_int, [_P, _P, C.c_int32, C.POINTER(MatchParams), _P, _P]),
    "frg_match_range": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(MatchParams), _P, _P, _P, _P]),
    "frg_match_range_host": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(MatchParams), _P, _P, _P]),
    "frg_match_range_tenants": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(MatchParams), _P, _P, _P, _P, _P]),
    "frg_match_range_tenants_host": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(MatchParams), _P, _P, _P,
                                               _P]),
    "frg_self_join": (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int32, C.POINTER(MatchParams), _P, _P, _P, _P]),
    "frg_self_join_host": (C.c_int, [_P, C.c_int64, C.c_int64, C.c_int32, C.POINTER(MatchParams), _P, _P, _P]),
    "frg_cluster_observe_host": (C.c_int, [_P, _P, C.c_int32, C.POINTER(MatchParams), C.POINTER(ClusterRing), _P,
                                           _P]),
    "frg_merge_topk": (C.c_int, [C.c_int32, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_float, _P, _P, _P, _P]),
    "frg_merge_topk_strided": (C.c_int, [C.c_int32, _P, C.c_int64, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_int32, C.c_float, _P, _P, _P, _P]),
    "frg_exchange_bytes": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "frg_match_exchange": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.POINTER(MatchParams), C.POINTER(Exchange),
                                     _P, _P, _P, _P, _P, _P]),
    "frg_exchange_merge_topk": (C.c_int, [C.c_int32, C.POINTER(Exchange), _P, _P, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_float, _P, _P, _P, _P]),
    "frg_exchange_status": (C.c_int, [C.c_int32, _P, C.c_int32, _P, C.POINTER(ExchangeStatus)]),
    "frg_last_launch_count": (C.c_int, []),
    "frg_last_variant": (C.c_char_p, []),
    "frg_profile_enable": (C.c_int, [C.c_int32]),
    "frg_profile_collect": (C.c_int, [C.POINTER(C.c_float), C.POINTER(C.c_int32)]),
    "frg_profile_stage_ms": (C.c_int, [C.c_int32, C.POINTER(C.c_float)]),
}


def _load() -> C.CDLL:
    # (re)build when the sources changed and a compiler is at hand; otherwise the library that
    # travelled with the tree is used as is.  A missing library is fatal: there is no CPU fallback.
    from . import build as _build
    try:
        _build.build()
    except Exception as e:  # no nvcc on this machine, or the compile failed
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libfrg.so is not built (%s missing) and could not be built here (%s). "
                "There is no CPU fallback." % (LIB_PATH, e))
        if not isinstance(e, _build.NoCompiler):
            raise
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header and library disagree
        fn.restype = res
        fn.argtypes = args
    if lib.frg_abi_version() != 1:
        raise ImportError("libfrg.so ABI version %d, expected 1" % lib.frg_abi_version())
    return lib


lib = _load()


def check(rc: int) -> None:
    if rc != OK:
        raise NativeError(rc, (lib.frg_last_error() or b"").decode("utf-8", "replace"))


def device_count() -> int:
    n = C.c_int32(0)
    check(lib.frg_device_count(C.byref(n)))
    return n.value


def last_launch_count() -> int:
    return int(lib.frg_last_launch_count())


def last_variant() -> str:
    return (lib.frg_last_variant() or b"").decode()


def profile_enable(on: bool) -> None:
    check(lib.frg_profile_enable(1 if on else 0))


def profile_collect():
    """(summed device ms of the dominant kernel launches since the last collect, launch count)."""
    ms, n = C.c_float(0), C.c_int32(0)
    check(lib.frg_profile_collect(C.byref(ms), C.byref(n)))
    return float(ms.value), int(n.value)


STAGE_NAMES = ["prep", "prepass", "floor", "dominant", "select", "fallback"]


def profile_stages():
    """Per-stage device ms accumulated by the last profile_collect()."""
    out = {}
    for i, name in enumerate(STAGE_NAMES):
        ms = C.c_float(0)
        check(lib.frg_profile_stage_ms(i, C.byref(ms)))
        out[name] = float(ms.value)
    return out
