"""ctypes binding of libgppd.so (include/gppd.h).  No fallback: if the shared
library is missing or no B200 is visible, calls raise."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# GPPD_LIBRARY: another build of the same library (kernel experiments, tools/); default in-tree
LIB_PATH = os.environ.get("GPPD_LIBRARY") or os.path.join(_HERE, "libgppd.so")
CSRC = os.path.join(_HERE, "csrc")

OK = 0
ONLYHIGH, FITOFFSETS, NO_RECENTER, KEEPRAW, BIG_ENDIAN, CENTER_EMPIRICAL, FP32 = 1, 2, 4, 8, 16, 32, 64
CENTER_ELLIPSE = 128
ELLIPSE_STRIDE = 6
METHOD_AUTO, METHOD_DIRECT, METHOD_HARMONIC = 0, 1, 2
INFO_STRIDE = 4
TRACE_MAX = 160


class Options(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("method", C.c_int32), ("maxfun", C.c_int32),
                ("has_xinit", C.c_int32), ("xinit", C.c_double * 2),
                ("rhobeg", C.c_double), ("rhoend", C.c_double),
                ("group_mask", C.c_uint32), ("reserved", C.c_uint32)]


SEG_COPY, SEG_BYTES, SEG_RECORDS = 0, 1, 2


class FileSegment(C.Structure):     # gppd_file_segment
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("offset", C.c_int64),
                ("length", C.c_int64), ("bytes", C.c_void_p)]


class GppdError(RuntimeError):
    def __init__(self, status, what, detail):
        super().__init__(f"libgppd: {what} (status {status}){': ' + detail if detail else ''}")
        self.status = status


_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_i8p = C.POINTER(C.c_int8)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_lib = None


def build(verbose: bool = False) -> str:
    """Compile libgppd.so for sm_100a with nvcc (make is incremental)."""
    subprocess.run(["make", "-C", CSRC] + ([] if verbose else ["-s"]), check=True)
    return LIB_PATH


def lib():
    """The loaded library; raises when libgppd.so has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GppdError(-1, "libgppd.so is not built", f"run `make -C {CSRC}` (needs nvcc); "
                        "there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    H = C.c_void_p
    L.gppd_version.restype = C.c_int
    L.gppd_strerror.restype = C.c_char_p
    L.gppd_strerror.argtypes = [C.c_int]
    L.gppd_last_error.restype = C.c_char_p
    L.gppd_create.argtypes = [C.c_int, C.POINTER(H)]
    L.gppd_destroy.argtypes = [H]
    L.gppd_alloc_pinned.argtypes = [H, C.c_uint64, C.POINTER(C.c_void_p)]
    L.gppd_free_pinned.argtypes = [H, C.c_void_p]
    L.gppd_idx.argtypes = [C.c_int] * 3
    L.gppd_phirange.argtypes = [_dp]
    L.gppd_buildstates.argtypes = [H, C.c_int64, _dp, _dp, C.c_int64, _dp, C.c_int64,
                                   C.c_int64, C.c_double, C.c_double, _i8p]
    L.gppd_num_windows.restype = C.c_int64
    L.gppd_num_windows.argtypes = [C.c_int64, C.c_int64]
    L.gppd_demodulate_f64.argtypes = [H, C.c_int64, C.c_int64, _dp, _dp, _i8p,
                                      C.POINTER(Options), _dp, _dp, _dp, _i32p, _dp]
    L.gppd_demodulate_f64_dev.argtypes = [H, C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.POINTER(Options), C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p]
    L.gppd_table_windows.argtypes = [C.c_int64, _i32p, C.c_double, C.c_double, _i64p, _i64p]
    tab = [C.c_int64, _i32p, C.c_double, _fp, _dp, _dp, C.c_int64, _dp, C.c_int64,
           C.c_double, C.POINTER(Options), _fp, _dp, _dp, _i32p, _i8p]
    L.gppd_process_table_f32.argtypes = [H] + tab
    L.gppd_submit_table_f32.argtypes = [H, C.c_int] + tab
    L.gppd_submit_fits_rows.argtypes = [
        H, C.c_int, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_double, _dp,
        _dp, C.c_int64, _dp, C.c_int64, C.c_double, C.POINTER(Options), C.c_void_p, _dp, _dp,
        _i32p, _i8p]
    L.gppd_file_submit.argtypes = [H, C.c_int, C.c_char_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                   C.c_int64, C.c_double, _dp, _dp, C.c_int64, _dp, C.c_int64, C.c_double,
                                   C.POINTER(Options)]
    L.gppd_file_wait.argtypes = [H, C.c_int, _dp, _dp, _i32p, _i8p]
    L.gppd_file_write.argtypes = [H, C.c_int, C.c_char_p, C.POINTER(FileSegment), C.c_int32, C.c_void_p,
                                  C.c_int64]
    L.gppd_file_drain.argtypes = [H]
    L.gppd_wait.argtypes = [H, C.c_int]
    L.gppd_centres.argtypes = [H, C.c_int, C.c_int64, _dp]
    L.gppd_ellipses.argtypes = [H, C.c_int, C.c_int64, _dp, _i32p]
    L.gppd_set_split_chains.argtypes = [H, C.c_int]
    L.gppd_debug_harmonics.argtypes = [H, C.c_int, _dp, C.c_int64]
    L.gppd_num_slots.argtypes = [H]
    L.gppd_process_table_f32_dev.argtypes = [
        H, C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_double, C.c_void_p,
        C.c_void_p, _dp, C.c_int64, _dp, C.c_int64, C.POINTER(Options), C.c_void_p,
        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    PP = C.POINTER(C.c_void_p)
    L.gppd_process_tables_f32_dev.argtypes = [
        H, C.c_int, C.c_void_p, C.c_int64, _i64p, _i64p, PP, _dp, PP, C.c_void_p,
        C.POINTER(_dp), _i64p, C.POINTER(_dp), _i64p, C.POINTER(Options), PP, PP, PP, PP, PP]
    L.gppd_debug_counters.argtypes = [H, C.POINTER(C.c_uint64), C.c_int]
    L.gppd_debug_counters.restype = C.c_int
    L.gppd_launch_count.restype = C.c_int64
    L.gppd_launch_count.argtypes = [H]
    L.gppd_enable_timing.argtypes = [H, C.c_int]
    L.gppd_pass_times.argtypes = [H, _dp, _i64p, C.c_int]
    L.gppd_measure_fp64_peak.argtypes = [H, _dp]
    for name in ("gppd_create", "gppd_destroy", "gppd_alloc_pinned", "gppd_free_pinned",
                 "gppd_idx", "gppd_phirange", "gppd_buildstates", "gppd_demodulate_f64",
                 "gppd_demodulate_f64_dev", "gppd_file_submit", "gppd_file_wait", "gppd_file_write",
                 "gppd_file_drain",
                 "gppd_table_windows", "gppd_process_table_f32", "gppd_submit_table_f32",
                 "gppd_submit_fits_rows", "gppd_centres", "gppd_ellipses", "gppd_debug_harmonics", "gppd_set_split_chains",
                 "gppd_wait", "gppd_num_slots", "gppd_process_table_f32_dev",
                 "gppd_process_tables_f32_dev", "gppd_enable_timing",
                 "gppd_pass_times", "gppd_measure_fp64_peak"):
        getattr(L, name).restype = C.c_int
    _lib = L
    return L


def check(status: int):
    if status != OK:
        L = lib()
        raise GppdError(status, L.gppd_strerror(status).decode(),
                        (L.gppd_last_error() or b"").decode())


def ptr(a, typ=_dp):
    return None if a is None else a.ctypes.data_as(typ)


class Handle:
    """Owns one gppd_handle (streams, scratch, pinned staging) on one GPU."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        check(lib().gppd_create(int(device), C.byref(self._h)))
        self.device = int(device)

    def close(self):
        if self._h:
            lib().gppd_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def raw(self):
        return self._h

    @property
    def launches(self) -> int:
        return int(lib().gppd_launch_count(self._h))

    @property
    def num_slots(self) -> int:
        return int(lib().gppd_num_slots(self._h))

    PASSES = ("segment", "basis", "stats", "fit", "demod", "export", "harmonics", "fallback")

    def fp64_peak_tflops(self) -> float:
        v = C.c_double(0)
        check(lib().gppd_measure_fp64_peak(self._h, C.byref(v)))
        return v.value

    def enable_timing(self, on: bool = True):
        check(lib().gppd_enable_timing(self._h, int(on)))

    def set_split_chains(self, on: bool = True):
        """FAINT and bright tables of a batch as two concurrent launch sequences (default on)."""
        check(lib().gppd_set_split_chains(self._h, int(on)))

    def pass_times(self, reset: bool = True):
        """{pass: (total ms, launches)} measured with CUDA events on the launching stream."""
        import numpy as np
        ms = np.zeros(8)
        cnt = np.zeros(8, dtype=np.int64)
        check(lib().gppd_pass_times(self._h, ptr(ms), ptr(cnt, _i64p), int(reset)))
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.PASSES)}


_default = {}


def default_handle() -> Handle:
    dev = int(os.environ.get("LOCAL_RANK", "0"))
    if dev not in _default:
        _default[dev] = Handle(dev)
    return _default[dev]
