"""ctypes binding of include/psd_b200.h (libpsd_b200.so).  Mirrors, symbol for symbol, what the
Julia glue binds with ccall (julia/PeriodicSchurB200.jl)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libpsd_b200.so")
_lib = None

# every symbol include/psd_b200.h declares (checked by tests/test_capi_symbols.py)
EXPORTED_SYMBOLS = [
    "psd_version",
    "psd_device_count",
    "psd_last_error_string",
    "psd_create",
    "psd_destroy",
    "psd_handle_device_count",
    "psd_rpschur_batched",
    "psd_rpschur_batched_dev",
    "psd_rpschur_hessut_batched",
    "psd_rpschur_hessut_q_batched",
    "psd_rphess_batched",
    "psd_rphess_packed_batched",
    "psd_cpschur_batched",
    "psd_cpschur_hessut_batched",
    "psd_rgpschur_batched",
    "psd_rgpschur_hessut_batched",
    "psd_rphess_rowwise_batched",
    "psd_gphess_batched",
    "psd_dgemm_host",
    "psd_last_stats",
    "psd_set_profiling",
    "psd_kernel_times",
    "psd_large_stats",
    "psd_set_iters_output",
    "psd_host_alloc",
    "psd_host_free",
    "psd_rcheckpsd_batched",
    "psd_reigvecs_batched",
    "psd_ceigvecs_batched",
    "psd_fill_uniform_host",
    "psd_fill_uniform_dev",
]


class PsdError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"psd_b200 error {code}: {msg}")
        self.code = code
        self.msg = msg


def lib_path() -> str:
    return _LIB_PATH


def library_available() -> bool:
    return os.path.exists(_LIB_PATH)


def lib():
    """Load libpsd_b200.so; fails loudly (no fallback) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise PsdError(-2, f"{_LIB_PATH} not built: run __graft_entry__.build() "
                               "(there is no CPU fallback)")
        L = C.CDLL(_LIB_PATH)
        dp = C.POINTER(C.c_double)
        ip = C.POINTER(C.c_int32)
        vp = C.c_void_p
        L.psd_version.restype = C.c_int
        L.psd_device_count.restype = C.c_int
        L.psd_last_error_string.restype = C.c_char_p
        L.psd_create.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(C.c_int)]
        L.psd_destroy.argtypes = [vp]
        L.psd_handle_device_count.argtypes = [vp]
        L.psd_rpschur_batched.argtypes = [vp, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int,
                                          C.c_int, C.c_int, vp, vp, vp, vp]
        L.psd_rpschur_batched_dev.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int64,
                                              C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]
        L.psd_rpschur_hessut_batched.argtypes = [vp, C.c_int, C.c_int, C.c_int64, C.c_int,
                                                 C.c_int, C.c_int, vp, vp, vp, vp]
        L.psd_rpschur_hessut_q_batched.argtypes = [vp, C.c_int, C.c_int, C.c_int64, C.c_int,
                                                   C.c_int, vp, vp, vp, vp]
        L.psd_set_iters_output.argtypes = [vp, vp]
        L.psd_host_alloc.argtypes = [C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]
        L.psd_host_free.argtypes = [vp]
        L.psd_rphess_packed_batched.argtypes = [vp, C.c_int, C.c_int, C.c_int64, vp, vp]
        L.psd_rcheckpsd_batched.argtypes = [vp, C.c_int, C.c_int, C.c_int64, C.c_int, vp, vp, vp, vp, vp, vp]
        L.psd_reigvecs_batched.argtypes = [vp, C.c_int, C.c_int, C.c_int64, C.c_int, vp, vp, vp, vp, vp]
        L.psd_ceigvecs_batched.argtypes = L.psd_reigvecs_batched.argtypes
        L.psd_rphess_batched.argtypes = [vp, C.c_int, C.c_int, C.c_int64, C.c_int, vp, vp]
        L.psd_cpschur_batched.argtypes = [vp, C.c_int, C.c_int, C.c_int64, C.c_int, vp, C.c_int,
                                          C.c_int, C.c_int, vp, vp, vp, vp, vp, vp]
        L.psd_cpschur_hessut_batched.argtypes = [vp, C.c_int, C.c_int, C.c_int64, vp, C.c_int,
                                                 C.c_int, C.c_int, vp, vp, vp, vp, vp, vp]
        L.psd_rgpschur_batched.argtypes = L.psd_cpschur_batched.argtypes
        L.psd_rgpschur_hessut_batched.argtypes = L.psd_cpschur_hessut_batched.argtypes
        L.psd_rphess_rowwise_batched.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64,
                                                 vp, vp, vp]
        L.psd_dgemm_host.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                                     vp, C.c_int, vp, C.c_int, C.c_double, vp, C.c_int, C.c_int,
                                     C.POINTER(C.c_double)]
        L.psd_gphess_batched.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int64, vp, C.c_int, vp, vp]
        L.psd_last_stats.argtypes = [vp, C.POINTER(C.c_int64)]
        L.psd_set_profiling.argtypes = [vp, C.c_int]
        L.psd_kernel_times.argtypes = [vp, C.POINTER(C.c_double)]
        L.psd_large_stats.argtypes = [vp, C.POINTER(C.c_double)]
        L.psd_fill_uniform_host.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_int64, C.c_int64,
                                            C.c_int, vp]
        L.psd_fill_uniform_dev.argtypes = [vp, C.c_uint64, C.c_int, C.c_int, C.c_int64,
                                           C.c_int64, C.c_int, vp]
        for name in EXPORTED_SYMBOLS:
            if name not in ("psd_last_error_string",):
                getattr(L, name).restype = C.c_int if name != "psd_last_error_string" else C.c_char_p
        L.psd_last_error_string.restype = C.c_char_p
        _ = (dp, ip)
        _lib = L
    return _lib


def check(code: int):
    if code != 0:
        msg = lib().psd_last_error_string()
        raise PsdError(code, msg.decode() if msg else "")


def version() -> int:
    return int(lib().psd_version())


def device_count() -> int:
    return int(lib().psd_device_count())
