"""ctypes binding of libstrkit_b200.so (the C ABI declared in include/strkit_b200.h).

There is no CPU fallback: if the shared library is missing, or there is no CUDA device, the
functions here raise -- loudly -- instead of computing anything on the host.
"""
from __future__ import annotations

import ctypes as C
import os

__all__ = ["lib", "StrkError", "check", "LIB_PATH", "build_hint"]

# STRKIT_B200_LIB: kernel-variant experiments only (an alternative build of the same C ABI)
LIB_PATH = os.environ.get("STRKIT_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                                             "libstrkit_b200.so")
build_hint = "build it with `python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a)"


class StrkError(RuntimeError):
    """A non-zero status from the native library (message from strk_last_error)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"strkit_b200 native error {code}: {message}")
        self.code = code


_vp = C.c_void_p
_i32, _i64, _u64 = C.c_int32, C.c_int64, C.c_uint64


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing; {build_hint}. strkit_b200 has no CPU fallback.")
    lib_ = C.CDLL(LIB_PATH)
    sig = {
        "strk_last_error": (C.c_char_p, []),
        "strk_version": (C.c_char_p, []),
        "strk_device_count": (C.c_int, []),
        "strk_init": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
        "strk_destroy": (C.c_int, [_vp]),
        "strk_sync": (C.c_int, [_vp]),
        "strk_host_register": (C.c_int, [_vp, _u64]),
        "strk_host_unregister": (C.c_int, [_vp]),
        "strk_batch_upload": (C.c_int, [_vp, _vp, _u64, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, C.POINTER(_vp)]),
        "strk_batch_create": (C.c_int, [_vp, C.POINTER(_vp)]),
        "strk_batch_fill": (C.c_int, [_vp, _vp, _vp, _u64, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64]),
        "strk_batch_fill_fmt": (C.c_int, [_vp, _vp, C.c_int, _vp, _u64, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64]),
        "strk_count_reads_fmt": (C.c_int, [_vp, C.c_int, _vp, _u64, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, C.c_int,
                                           C.c_int, C.c_int, C.c_int, _vp]),
        "strk_batch_run": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
        "strk_batch_download": (C.c_int, [_vp, _vp, _vp]),
        "strk_batch_free": (C.c_int, [_vp, _vp]),
        "strk_count_reads": (C.c_int, [_vp, _vp, _u64, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, C.c_int, C.c_int,
                                       C.c_int, C.c_int, _vp]),
        "strk_get_repeat_count": (C.c_int, [_vp, C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_int,
                                            C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
        "strk_score_tables": (C.c_int, [_vp, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _i64, _vp, C.c_int,
                                        _vp]),
        "strk_ref_boundary_tables": (C.c_int, [_vp, _vp, _u64, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, C.c_int,
                                               _vp]),
        "strk_ref_counts": (C.c_int, [_vp, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, C.c_int, C.c_int, _vp]),
        "strk_call_alleles": (C.c_int, [_vp, _vp, _vp, _vp, _i64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                                        C.c_int, C.c_int, _u64, _vp, _vp, _vp, _vp]),
        "strk_gmm_fit_counts": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_double, C.c_int, C.c_int, _vp]),
        "strk_call_alleles_ploidy": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.c_double, C.c_int, C.c_int, _u64, _vp, _vp, _vp, _vp]),
        "strk_gmm_fit_counts_ploidy": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, C.c_int, C.c_int, C.c_int, C.c_int,
                                                 C.c_double, C.c_int, C.c_int, _u64, _vp]),
        "strk_gmm_fit_counts_deep": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.c_double, C.c_int, C.c_int, _u64, _vp]),
        "strk_alleles_aggregate": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, C.c_int, C.c_int, _vp, _vp]),
        "strk_realign": (C.c_int, [_vp, _vp, _u64, _vp, _vp, _vp, _vp, _i64, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp, _vp,
                                   _vp]),
        "strk_get_stats": (C.c_int, [_vp, _vp]),
        "strk_measure_int_peak": (C.c_int, [_vp, _vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib_, name)  # AttributeError here = header and library out of sync
        fn.restype = res
        fn.argtypes = args
    return lib_


lib = _load()
EXPORTED = ("strk_last_error", "strk_version", "strk_device_count", "strk_init", "strk_destroy", "strk_sync", "strk_host_register",
            "strk_host_unregister", "strk_batch_upload", "strk_batch_create", "strk_batch_fill", "strk_batch_fill_fmt", "strk_count_reads_fmt", "strk_batch_run", "strk_batch_download", "strk_batch_free",
            "strk_count_reads", "strk_get_repeat_count", "strk_score_tables", "strk_ref_boundary_tables", "strk_ref_counts", "strk_call_alleles", "strk_gmm_fit_counts",
            "strk_call_alleles_ploidy", "strk_gmm_fit_counts_ploidy", "strk_gmm_fit_counts_deep", "strk_alleles_aggregate", "strk_realign", "strk_get_stats", "strk_measure_int_peak")


def check(rc: int) -> None:
    if rc != 0:
        raise StrkError(rc, lib.strk_last_error().decode("utf-8", "replace"))
