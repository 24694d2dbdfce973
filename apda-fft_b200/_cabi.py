"""ctypes binding of libapda_b200.so (C ABI in include/apda_b200.h).

There is no CPU fallback: if the shared library is missing, or no sm_100 device is visible, every entry point
raises.  ``load()`` alone (no context) is enough to check that the library exports the ABI.
"""
from __future__ import annotations

import ctypes
import os
import statistics
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
# APDA_LIB: another build of the same library (same-box A/B measurements of kernel variants; see build.py APDA_LIB_OUT)
LIB_PATH = os.environ.get("APDA_LIB") or os.path.join(HERE, "libapda_b200.so")

OK = 0
ERR_INVALID, ERR_NO_DEVICE, ERR_CUDA, ERR_NOMEM, ERR_UNSUPPORTED, ERR_STATS_MEAN, ERR_STATS_STDEV = -1, -2, -3, -4, -5, -6, -7
CENTER_MEDIAN, CENTER_MEAN, CENTER_NONE = 0, 1, 2
MAX_REC_CAP = 64

_c = ctypes
_p, _i64, _int, _dbl, _u64 = _c.c_void_p, _c.c_int64, _c.c_int, _c.c_double, _c.c_uint64

# name -> (restype, argtypes): every symbol include/apda_b200.h declares
SIGNATURES = {
    "apda_ctx_create": (_int, [_int, _c.POINTER(_p)]),
    "apda_ctx_destroy": (_int, [_p]),
    "apda_ctx_set_stream": (_int, [_p, _p]),
    "apda_ctx_reset_stream": (_int, [_p]),
    "apda_ctx_set_generic_only": (_int, [_p, _int]),
    "apda_sync": (_int, [_p]),
    "apda_last_error": (_c.c_char_p, []),
    "apda_version": (_int, []),
    "apda_launch_count": (_i64, [_p]),
    "apda_fft_f64_dev": (_int, [_p, _p, _i64, _i64, _i64, _i64, _int, _p]),
    "apda_fft_f32_dev": (_int, [_p, _p, _i64, _i64, _i64, _i64, _int, _p]),
    "apda_fft_f64_host": (_int, [_p, _p, _i64, _i64, _i64, _i64, _int, _p]),
    "apda_fft_f32_host": (_int, [_p, _p, _i64, _i64, _i64, _i64, _int, _p]),
    "apda_fft_c2c_f64_host": (_int, [_p, _p, _i64, _i64, _p]),
    "apda_center_f64_host": (_int, [_p, _p, _i64, _p]),
    "apda_peaks_prominence_f64_dev": (_int, [_p, _p, _i64, _i64, _dbl, _p, _int, _int, _p]),
    "apda_peaks_prominence_f32_dev": (_int, [_p, _p, _i64, _i64, _dbl, _p, _int, _int, _p]),
    "apda_peaks_resolution_f64_dev": (_int, [_p, _p, _i64, _i64, _dbl, _p, _int, _int, _p]),
    "apda_peaks_resolution_f32_dev": (_int, [_p, _p, _i64, _i64, _dbl, _p, _int, _int, _p]),
    "apda_peaks_prominence_f64_host": (_int, [_p, _p, _i64, _i64, _dbl, _p, _int, _int, _p]),
    "apda_peaks_resolution_f64_host": (_int, [_p, _p, _i64, _i64, _dbl, _p, _int, _int, _p]),
    "apda_peaks_prominence_f32_host": (_int, [_p, _p, _i64, _i64, _dbl, _p, _int, _int, _p]),
    "apda_peaks_resolution_f32_host": (_int, [_p, _p, _i64, _i64, _dbl, _p, _int, _int, _p]),
    "apda_analyze_f64_dev": (_int, [_p, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p, _p]),
    "apda_analyze_f32_dev": (_int, [_p, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p, _p]),
    "apda_analyze_f64_host": (_int, [_p, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p]),
    "apda_analyze_f32_host": (_int, [_p, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p]),
    "apda_multi_analyze_f32_host": (_int, [_p, _int, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p]),
    "apda_multi_analyze_f64_host": (_int, [_p, _int, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p]),
    "apda_fft_ragged_f64_dev": (_int, [_p, _p, _p, _i64, _i64, _i64, _i64, _int, _p]),
    "apda_fft_ragged_f32_dev": (_int, [_p, _p, _p, _i64, _i64, _i64, _i64, _int, _p]),
    "apda_analyze_ragged_f64_dev": (_int, [_p, _p, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p, _p]),
    "apda_analyze_ragged_f32_dev": (_int, [_p, _p, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p, _p]),
    "apda_decode_wire16_f64_dev": (_int, [_p, _p, _i64, _i64, _i64, _p, _p, _i64, _p]),
    "apda_decode_wire16_f32_dev": (_int, [_p, _p, _i64, _i64, _i64, _p, _p, _i64, _p]),
    "apda_decode_wire16_f64_host": (_int, [_p, _p, _i64, _i64, _i64, _p, _p, _p]),
    "apda_analyze_wire16_f64_host": (_int, [_p, _p, _i64, _i64, _i64, _p, _i64, _int, _int, _dbl, _p, _int, _int, _p]),
    "apda_analyze_wire16_f32_host": (_int, [_p, _p, _i64, _i64, _i64, _p, _i64, _int, _int, _dbl, _p, _int, _int, _p]),
    "apda_parse_samples_f64_host": (_int, [_p, _p, _p, _i64, _i64, _p, _p, _p]),
    "apda_analyze_text_f64_host": (_int, [_p, _p, _p, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p, _p, _p]),
    "apda_analyze_text_f32_host": (_int, [_p, _p, _p, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p, _p, _p]),
    "apda_analyze_logs_f64_host": (_int, [_p, _p, _i64, _i64, _int, _int, _int, _int, _p, _p, _p, _p, _p]),
    "apda_analyze_logs_f32_host": (_int, [_p, _p, _i64, _i64, _int, _int, _int, _int, _p, _p, _p, _p, _p]),
    "apda_analyze_fused_f32_dev": (_int, [_p, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p]),
    "apda_analyze_fused_f32_host": (_int, [_p, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p]),
    "apda_resolve_fp32_ties_dev": (_int, [_p, _p, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p]),
    "apda_resolve_fp32_ties_host": (_int, [_p, _p, _p, _i64, _i64, _i64, _i64, _int, _int, _dbl, _p, _int, _int, _p]),
    "apda_present_dev": (_int, [_p, _p, _int, _i64, _i64, _dbl, _p, _int, _int, _p, _p, _p, _p, _p, _p]),
    "apda_present_host": (_int, [_p, _p, _int, _i64, _i64, _dbl, _p, _int, _int, _p, _p, _p, _p, _p, _p]),
    "apda_fleet_jsonl_dev": (_int, [_p, _p, _int, _i64, _i64, _dbl, _p, _int, _int, _i64, _p, _i64, _p]),
    "apda_fleet_jsonl_host": (_int, [_p, _p, _int, _i64, _i64, _dbl, _p, _int, _int, _i64, _p, _i64, _p]),
    "apda_prominence_f64_host":(_int, [_p, _p, _i64, _i64, _c.POINTER(_dbl)]),
    "apda_half_power_bins_f64_host": (_int, [_p, _p, _i64, _dbl, _i64, _c.POINTER(_i64)]),
    "apda_half_height_bins_f64_host": (_int, [_p, _p, _i64, _i64, _c.POINTER(_i64)]),
    "apda_synth_f64_dev": (_int, [_p, _i64, _i64, _i64, _u64, _int, _p]),
    "apda_synth_f32_dev": (_int, [_p, _i64, _i64, _i64, _u64, _int, _p]),
    "apda_peer_table_create": (_int, [_p, _i64, _c.POINTER(_p), _p]),
    "apda_peer_table_open": (_int, [_p, _p, _c.POINTER(_p)]),
    "apda_peer_table_close": (_int, [_p, _p]),
    "apda_peer_table_destroy": (_int, [_p, _p]),
    "apda_peer_signal": (_int, [_p, _p, _c.c_uint32]),
    "apda_peer_wait": (_int, [_p, _p, _int, _c.c_uint32, _dbl, _p]),
}


def max_peaks(n: int) -> int:
    """include/apda_b200.h APDA_MAX_PEAKS(n): most peaks one window of n bins can report."""
    return int(n) // 8 + 8


def jsonl_row_bytes(k: int) -> int:
    """include/apda_b200.h APDA_JSONL_ROW_BYTES(k): bound on the bytes of one fleet JSONL row with k peaks."""
    return 64 + 52 * int(k)


# record status bits (include/apda_b200.h)
STATUS_TRUNCATED, STATUS_OTHER_LENGTH, STATUS_EMPTY, STATUS_FP32_TIE = 1, 4, 8, 16

# apda_analyze_logs_*_host: header bytes per file and the per-file flag bits
LOG_HEAD_BYTES = 1024
LOG_SAMPLE_UNDECIDED, LOG_TOO_LONG, LOG_NO_SAMPLE_LINE, LOG_HEADER_UNDECIDED, LOG_UNREADABLE = 1, 2, 4, 8, 16


def check_record_status(recs) -> None:
    """The drop-in modules return reference-equivalent results or raise: a record whose status is not 0 (candidate
    list truncated, window transformed at another length, empty window) must never be handed out silently."""
    import numpy as np
    bad = np.flatnonzero(np.asarray(recs["status"]) != 0)
    if bad.size:
        raise ApdaError(ERR_UNSUPPORTED, f"record status {int(recs['status'][bad[0]])} on window {int(bad[0])} "
                                         f"({bad.size} of {len(recs)} windows): the result is not reference-equivalent")


class ApdaError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libapda_b200 error {code}: {message}")
        self.code = code
        self.message = message


_lib = None
_lock = threading.Lock()


def load() -> ctypes.CDLL:
    """dlopen the library and bind every declared symbol; raises if it is missing (no fallback path exists)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise ApdaError(ERR_NO_DEVICE, f"{LIB_PATH} is not built (python apda-fft_b200/build.py); "
                                               "there is no CPU fallback")
            lib = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(status: int) -> None:
    """Map a C status to the exception the reference raises for the same condition (SURVEY.md 8b)."""
    if status == OK:
        return
    msg = load().apda_last_error().decode("utf-8", "replace")
    if status in (ERR_STATS_MEAN, ERR_STATS_STDEV):
        raise statistics.StatisticsError(msg)
    if status == ERR_INVALID:
        raise ValueError(msg)
    if status == ERR_NOMEM:
        raise MemoryError(msg)
    raise ApdaError(status, msg)


class Context:
    """One apda_ctx (one host thread, one device)."""

    def __init__(self, device: int = 0):
        self._lib = load()
        handle = _p()
        check(self._lib.apda_ctx_create(int(device), ctypes.byref(handle)))
        self._h = handle
        self.device = int(device)

    @property
    def handle(self):
        return self._h

    def call(self, name: str, *args) -> None:
        check(getattr(self._lib, name)(self._h, *args))

    def set_stream(self, cuda_stream: int | None) -> None:
        """cuda_stream: raw cudaStream_t value (0 is the legacy default stream); None -> the context's own stream."""
        if cuda_stream is None:
            self.call("apda_ctx_reset_stream")
        else:
            self.call("apda_ctx_set_stream", _p(int(cuda_stream)))

    def set_generic_only(self, on: bool) -> None:
        self.call("apda_ctx_set_generic_only", int(bool(on)))

    def sync(self) -> None:
        self.call("apda_sync")

    def launch_count(self) -> int:
        return int(self._lib.apda_launch_count(self._h))

    def close(self) -> None:
        if self._h:
            self._lib.apda_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default: dict[tuple[int, int], Context] = {}


def default_context(device: int = 0) -> Context:
    """Per-(thread, device) context used by the drop-in modules."""
    key = (threading.get_ident(), device)
    ctx = _default.get(key)
    if ctx is None:
        ctx = _default[key] = Context(device)
    return ctx
