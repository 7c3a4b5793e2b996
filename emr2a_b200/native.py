"""ctypes binding of libemr2a.so (the C-ABI declared in include/emr2a.h).

There is no CPU fallback: if the library is missing or no sm_100 device is
present, the product path raises.  ``symbols()`` lists every entry point the
header declares so the CPU test-suite can check the exports without a GPU.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libemr2a.so")

OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED, ERR_WORKSPACE = 0, 1, 2, 3, 4
F32, BF16 = 0, 1
NF_SEGNORM, NF_ROWNORM, NF_ZERO_GUARD, NF_STANDARDIZE = 1, 2, 4, 8
PREC_FP32, PREC_BF16X3, PREC_BF16X1, PREC_BF16_RESCORE = 0, 1, 2, 3
SCORE_NONE, SCORE_ZSCORE, SCORE_MINMAX = 0, 1, 2
ABI_VERSION = 13

_p = C.c_void_p
_i64 = C.c_int64
_int = C.c_int
_f = C.c_float
_sz = C.c_size_t

_SIGNATURES = {
    "emr2a_abi_version": (_int, []),
    "emr2a_last_error": (C.c_char_p, []),
    "emr2a_device_check": (_int, [C.POINTER(_int), C.POINTER(_int), C.POINTER(_int)]),
    "emr2a_normalize_fuse": (_int, [_p, _p, _i64, _int, _int, _i64, _i64, _f, _f, _int, _int,
                                    _p, _i64, _p, _p, _i64, _p, _p, _p, _p, _p]),
    "emr2a_scores": (_int, [_p, _p, _i64, _i64, _int, _i64, _i64, _p, _i64, _p]),
    "emr2a_euclid_workspace_bytes": (_sz, [_i64]),
    "emr2a_euclid_scores": (_int, [_p, _p, _i64, _int, _i64, _p, _p, _sz, _p]),
    "emr2a_late_fuse_scores": (_int, [_p, _p, _i64, _i64, _i64, _f, _f, _int, _p, _i64, _p]),
    "emr2a_topk_search_workspace_bytes": (_sz, [_i64, _i64, _int, _int, _int]),
    "emr2a_topk_search": (_int, [_p, _i64, _p, _p, _i64, _p, _i64, _p, _p, _i64, _i64, _i64, _int, _p, _p, _int,
                                 _i64, _int, _int, _p, _p, _p, _p, _p, _p, _sz, _p, _p]),
    "emr2a_topk_filter_workspace_bytes": (_sz, [_i64, _i64, _int, _int]),
    "emr2a_topk_filter": (_int, [_p, _i64, _p, _i64, _i64, _i64, _int, _p, _p, _int, _i64, _int, _p, _p, _p, _p, _sz, _p]),
    "emr2a_rescore_candidates": (_int, [_p, _p, _p, _p, _i64, _p, _i64, _i64, _i64, _int, _i64, _int, _p, _p, _p, _p, _p, _p]),
    "emr2a_verify_merged": (_int, [_p, _int, _i64, _p, _int, _i64, _p, _p, _p]),
    "emr2a_exact_rescan_workspace_bytes": (_sz, [_int, _int]),
    "emr2a_exact_rescan": (_int, [_p, _i64, _p, _i64, _i64, _int, _i64, _int, _p, _p, _p, _int, _p, _p, _sz, _p,
                                  _p, _i64, _p, _p, _p, _p]),
    "emr2a_range_search_workspace_bytes": (_sz, [_i64, _i64, _int]),
    "emr2a_range_search": (_int, [_p, _i64, _p, _i64, _p, _i64, _p, _i64, _i64, _i64, _int, _p, _p, _int, _i64, _f, _p, _p,
                                  _p, _i64, _p, _i64, _p, _p, _sz, _p, _p]),
    "emr2a_self_join_workspace_bytes": (_sz, [_i64, _int]),
    "emr2a_self_join": (_int, [_p, _i64, _p, _i64, _i64, _int, _i64, _i64, _p, _int, _f, _p, _p, _i64, _p, _i64, _p, _p,
                               _sz, _p]),
    "emr2a_topk_merge": (_int, [_p, _int, _i64, _int, _i64, _i64, _int, _p, _p]),
    "emr2a_keys_map_rows": (_int, [_p, _i64, _p, _i64, _i64, _p]),
    "emr2a_vote_metrics": (_int, [_p, _i64, _int, _p, _i64, _p, _p, _int, _int, C.POINTER(C.c_int32), _int, _int,
                                  _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "emr2a_topk_from_scores": (_int, [_p, _i64, _i64, _i64, _int, _p, _p]),
    "emr2a_column_moments_workspace_bytes": (_sz, [_i64, _int]),
    "emr2a_column_moments": (_int, [_p, _i64, _i64, _int, _p, _p, _p, _p, _sz, _p]),
    "emr2a_standardize": (_int, [_p, _i64, _i64, _int, _p, _p, _p, _i64, _p]),
    "emr2a_gram_f64_workspace_bytes": (_sz, [_i64, _int]),
    "emr2a_gram_f64": (_int, [_p, _i64, _i64, _int, _p, _p, _p, _p, _p, _sz, _p]),
    "emr2a_project": (_int, [_p, _i64, _i64, _int, _p, _p, _p, _i64, _int, _p, _p, _i64, _p]),
    "emr2a_scale_segments": (_int, [_p, _i64, _int, _int, _i64, _p, _p, _p]),
    "emr2a_keys_add_offset": (_int, [_p, _i64, _int, _p, _p]),
    "emr2a_segment_mean": (_int, [_p, _i64, _p, _i64, _int, _p, _i64, _p]),
    # diagnostics (not part of the reference-facing surface)
    "emr2a_debug_topk_search_dump": (_int, [_p, _p, _p, _p, _i64, _i64, _int, _i64, _i64, _p, _p, _i64, _int, _int,
                                            _p, _p, _sz, _p, _p]),
    "emr2a_debug_unit_clocks": (_int, [_p, _i64, _p]),
    "emr2a_debug_tc_timing": (_int, [_int]),
    "emr2a_debug_tc_elapsed": (_int, [_p, _int, _p]),
}


class LazyRows(C.Structure):
    """``emr2a_lazy_rows`` of include/emr2a.h: deferred fp32 rows (raw rows + the divisors K1 recorded)."""
    _fields_ = [("seg0", C.c_void_p), ("seg1", C.c_void_p), ("d0", C.c_int32), ("d1", C.c_int32),
                ("ld0", C.c_int64), ("ld1", C.c_int64), ("dtype", C.c_int32), ("w0", C.c_float), ("w1", C.c_float),
                ("flags", C.c_int32), ("row_div", C.c_void_p)]


def symbols():
    return sorted(_SIGNATURES)


class Emr2aError(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__(f"libemr2a error {code}: {text}")
        self.code = code


_lib: Optional[C.CDLL] = None


def load(check_device: bool = False) -> C.CDLL:
    """Load libemr2a.so (building is the job of ``__graft_entry__.build`` /
    ``python -m emr2a_b200.build``).  Raises if it is absent -- never falls back."""
    global _lib
    if _lib is None:
        if os.environ.get("EMR2A_NO_AUTOBUILD") != "1":
            try:            # rebuild when a CUDA source changed since the library was linked (no-op otherwise)
                from . import build as _build
                _build.build()
            except Exception as exc:  # pragma: no cover - nvcc missing: use what is there, or fail below
                if not os.path.exists(LIB_PATH):
                    raise ImportError(f"libemr2a.so is missing and could not be built: {exc}") from exc
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -m emr2a_b200.build` "
                "(the EMR2A B200 path has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if lib.emr2a_abi_version() != ABI_VERSION:
            raise ImportError(f"libemr2a ABI {lib.emr2a_abi_version()} != binding {ABI_VERSION}; rebuild")
        _lib = lib
    if check_device:
        device_check()
    return _lib


def last_error() -> str:
    return load().emr2a_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    if rc == OK:
        return
    text = last_error()
    if rc == ERR_INVALID:
        raise ValueError(text)
    raise Emr2aError(rc, text)


def device_check():
    sms, major, minor = _int(0), _int(0), _int(0)
    check(load().emr2a_device_check(C.byref(sms), C.byref(major), C.byref(minor)))
    return sms.value, major.value, minor.value


def ptr(t) -> Optional[int]:
    """Device pointer of a torch tensor (None passes NULL)."""
    if t is None:
        return None
    return t.data_ptr()
