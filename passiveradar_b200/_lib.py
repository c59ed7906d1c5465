"""ctypes binding of libprcore.so (C ABI: include/prcore.h).

The library is the ONLY compute path of this package: if it is missing, cannot
be built, or finds no CUDA device, every operator raises -- there is no CPU
fallback (the numpy oracle under ``oracle/`` is test infrastructure and is never
imported from here).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PRC_LIBRARY") or os.path.join(_PKG, "libprcore.so")     # PRC_LIBRARY: A/B builds during development

PRC_OK = 0
PRC_E_INVALID = -1
PRC_E_CUDA = -2
PRC_E_SINGULAR = -3
PRC_E_NOMEM = -4
MEM_HOST = 0
MEM_DEVICE = 1
FLAG_ASYNC = 1
FLAG_WINDOW_F32 = 2
FLAG_ABS_C64 = 4
IQ_C64, IQ_I8, IQ_I16 = 0, 1, 2
MIX_NONE, MIX_C64, MIX_C128, MIX_F64, MIX_FS64 = 0, 1, 2, 3, 4
SIG_C64, SIG_I8, SIG_I16, SIG_F64, SIG_C128 = 0, 1, 2, 3, 4

# every symbol include/prcore.h declares: name -> (restype, argtypes)
_c64p = C.c_void_p
SIGNATURES = {
    "prc_version": (C.c_int, []),
    "prc_last_error": (C.c_char_p, []),
    "prc_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "prc_init": (C.c_int, [C.c_int]),
    "prc_shutdown": (None, []),
    "prc_sync": (C.c_int, [C.c_int, C.c_void_p]),
    "prc_launch_count": (C.c_uint64, []),
    "prc_profile_enable": (C.c_int, [C.c_int]),
    "prc_profile_collect": (C.c_int, []),
    "prc_profile_kernels": (C.c_int, []),
    "prc_profile_read": (C.c_int, [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "prc_profile_reset": (C.c_int, []),
    "prc_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_uint64]),
    "prc_host_free": (C.c_int, [C.c_void_p]),
    "prc_host_register": (C.c_int, [C.c_void_p, C.c_uint64]),
    "prc_host_unregister": (C.c_int, [C.c_void_p]),
    "prc_xambg_c64": (C.c_int, [_c64p, _c64p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                C.c_int64, _c64p, C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_ls_filter_c64": (C.c_int, [_c64p, _c64p, C.c_int64, C.c_int, C.c_int, C.c_float, _c64p, _c64p,
                                    C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_ls_toeplitz_c64": (C.c_int, [_c64p, _c64p, C.c_int64, C.c_int, C.c_int, _c64p, _c64p,
                                      C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_ls_multiple_c64": (C.c_int, [_c64p, _c64p, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_int,
                                      _c64p, _c64p, C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_ls_multiple_frames_c64": (C.c_int, [_c64p, _c64p, C.c_int64, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_void_p,
                                             C.c_int, _c64p, C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_nlms_c64": (C.c_int, [_c64p, _c64p, C.c_int64, C.c_int, C.c_int, C.c_float, C.c_int, _c64p,
                               _c64p, _c64p, C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_frame_c64": (C.c_int, [_c64p, _c64p, C.c_int64, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int,
                                C.c_void_p, _c64p, _c64p, _c64p, C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_frames_c64": (C.c_int, [_c64p, _c64p, C.c_int64, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int,
                                 C.c_void_p, _c64p, _c64p, _c64p, C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_nlms_frames_c64": (C.c_int, [_c64p, _c64p, C.c_int64, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_float, C.c_int,
                                      _c64p, _c64p, _c64p, C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_xambg_frames_c64": (C.c_int, [_c64p, _c64p, C.c_int64, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p, _c64p,
                                       C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_ls_status": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_int), C.c_int]),
    "prc_set_option": (C.c_int, [C.c_char_p, C.c_int]),
    "prc_get_option": (C.c_int, [C.c_char_p, C.POINTER(C.c_int)]),
    "prc_direct_xambg_c64": (C.c_int, [_c64p, _c64p, C.c_int64, C.c_int, C.c_int, C.c_double, _c64p,
                                       C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_iq_mix_c64": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_double, C.c_double, C.c_double,
                                 _c64p, C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_resample_out_len": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64)]),
    "prc_frontend_c64": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_double, C.c_double, C.c_double,
                                   C.c_int, C.c_int, C.c_void_p, C.c_int, _c64p, C.c_int64,
                                   C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_cfar2d_f32": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_xcorr_c64": (C.c_int, [_c64p, C.c_int64, _c64p, C.c_int64, C.c_int64, C.c_int64, _c64p,
                                C.c_int, C.c_int, C.c_void_p, C.c_uint]),
    "prc_channel_offset": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int64,
                                     C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_int, C.c_int, C.c_void_p, C.c_uint]),
}

_lib = None
_lock = threading.Lock()


class PrcoreError(RuntimeError):
    """A libprcore call returned a non-zero status."""

    def __init__(self, code, message):
        super().__init__(f"libprcore error {code}: {message}")
        self.code = code


def load(build_if_missing: bool = True):
    """Load (building first if the .so is absent and nvcc exists) and type the library."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if build_if_missing and not os.environ.get("PRC_LIBRARY"):
            # rebuild when the library is missing OR older than any source/header (a stale .so after an edit is
            # the worst kind of bug); a no-op when up to date.  Without nvcc an existing library is used as is
            # (the GPU box receives the library built here).
            from . import build as _build
            try:
                _build.build(force=False)
            except RuntimeError:
                if not os.path.exists(LIB_PATH):
                    raise
        if not os.path.exists(LIB_PATH):
            raise OSError(f"{LIB_PATH} not found")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(status: int):
    if status == PRC_OK:
        return
    msg = load().prc_last_error().decode("utf-8", "replace")
    if status == PRC_E_SINGULAR:
        raise np.linalg.LinAlgError(msg or "Singular matrix")
    if status == PRC_E_NOMEM:
        raise MemoryError(msg)
    raise PrcoreError(status, msg)


def set_option(name: str, value: int):
    """Run-time switch of the library (include/prcore.h: "fft", "fft_min_n")."""
    check(load().prc_set_option(name.encode(), int(value)))


def get_option(name: str) -> int:
    v = C.c_int(0)
    check(load().prc_get_option(name.encode(), C.byref(v)))
    return v.value


def device_count() -> int:
    n = C.c_int(0)
    st = load().prc_device_count(C.byref(n))
    return n.value if st == PRC_OK else 0


def launch_count() -> int:
    return int(load().prc_launch_count())


def profile(enable: bool):
    check(load().prc_profile_enable(1 if enable else 0))


def profile_reset():
    check(load().prc_profile_reset())


def profile_read():
    """{kernel name: (total_ms, launches)} accumulated since the last reset (synchronises)."""
    lib = load()
    check(lib.prc_profile_collect())
    out = {}
    for i in range(lib.prc_profile_kernels()):
        name = C.c_char_p()
        ms = C.c_double()
        cnt = C.c_uint64()
        check(lib.prc_profile_read(i, C.byref(name), C.byref(ms), C.byref(cnt)))
        out[name.value.decode()] = (ms.value, int(cnt.value))
    return out


def current_device() -> int:
    """Device used by the drop-in operators: PRC_DEVICE, else LOCAL_RANK (torchrun), else 0."""
    for key in ("PRC_DEVICE", "LOCAL_RANK"):
        v = os.environ.get(key)
        if v not in (None, ""):
            return int(v)
    return 0


def ptr(a) -> int:
    """Address of a numpy array (host) or of a torch CUDA tensor (device)."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()


def as_c64(x, name="input"):
    """1-D C-contiguous complex64 view/copy of an array-like (complex128 is rounded, as
    main.py:186-194 effectively does when it declares dtype=complex64)."""
    a = np.asarray(x)
    if a.ndim != 1:
        raise ValueError(f"{name} must be one-dimensional, got shape {a.shape}")
    return np.ascontiguousarray(a, dtype=np.complex64)
