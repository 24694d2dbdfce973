"""Batched API over the C ABI: numpy host arrays (H2D/D2H inside the call) or raw device pointers (torch tensors).

    an = Analyzer(device=0)
    recs = an.analyze(samples_f32_or_f64[B, n_samples], fs=125.0, flexible=True)      # numpy structured records
    an.analyze_device(d_samples.data_ptr(), B, n_samples, N, "f32", d_rec.data_ptr()) # everything stays in HBM
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _cabi
from .records import record_dtype

_p = ctypes.c_void_p


def next_pow2(n: int) -> int:
    p = 1
    while p < n:
        p *= 2
    return p


def _suffix(dtype) -> str:
    dt = np.dtype(dtype)
    if dt == np.float64:
        return "f64"
    if dt == np.float32:
        return "f32"
    raise TypeError(f"unsupported dtype {dt}: the kernels compute in float32 or float64")


class Analyzer:
    def __init__(self, device: int = 0, ctx: _cabi.Context | None = None):
        self.ctx = ctx or _cabi.Context(device)

    # ---- host arrays -----------------------------------------------------------------------------------------
    def fft(self, samples: np.ndarray, n_fft: int | None = None, center: int = _cabi.CENTER_MEDIAN) -> np.ndarray:
        """[B, n_samples] real -> [B, N] complex (bin 0 == 0); start_fft of every row."""
        x = np.ascontiguousarray(np.atleast_2d(samples))
        sfx = _suffix(x.dtype)
        b, ns = x.shape
        n = next_pow2(ns) if n_fft is None else int(n_fft)
        out = np.empty((b, n), dtype=np.complex128 if sfx == "f64" else np.complex64)
        self.ctx.call(f"apda_fft_{sfx}_host", _p(x.ctypes.data), ns, ns, b, n, center, _p(out.ctypes.data))
        return out

    def fft_c2c(self, z: np.ndarray) -> np.ndarray:
        z = np.ascontiguousarray(np.atleast_2d(z), dtype=np.complex128)
        out = np.empty_like(z)
        self.ctx.call("apda_fft_c2c_f64_host", _p(z.ctypes.data), z.shape[0], z.shape[1], _p(out.ctypes.data))
        return out

    def peaks(self, spectra: np.ndarray, fs, flexible: bool = True, k: int | None = None,
              rec_cap: int | None = None) -> np.ndarray:
        """[B, n] complex spectra -> records[B]; complex64 input runs the fp32 kernels, anything else the fp64 ones."""
        z = np.atleast_2d(spectra)
        sfx = "f32" if z.dtype == np.complex64 else "f64"
        z = np.ascontiguousarray(z, dtype=np.complex64 if sfx == "f32" else np.complex128)
        b, n = z.shape
        k = (4 if flexible else 5) if k is None else int(k)
        cap = max(5, k) if rec_cap is None else int(rec_cap)
        recs = np.zeros(b, dtype=record_dtype(cap))
        fs_scalar, fs_arr = self._fs(fs, b)
        name = f"apda_peaks_prominence_{sfx}_host" if flexible else f"apda_peaks_resolution_{sfx}_host"
        self.ctx.call(name, _p(z.ctypes.data), n, b, fs_scalar, _p(fs_arr.ctypes.data if fs_arr is not None else 0),
                      k, cap, _p(recs.ctypes.data))
        return recs

    def analyze(self, samples: np.ndarray, fs, flexible: bool = True, k: int | None = None,
                n_fft: int | None = None, center: int = _cabi.CENTER_MEDIAN, rec_cap: int | None = None,
                resolve_ties: bool = True) -> np.ndarray:
        """[B, n_samples] real (float32 or float64) -> records[B]; spectra never leave the device.  float32 windows
        whose record status is APDA_STATUS_FP32_TIE get the float64 path's record (``resolve_ties``)."""
        x = np.ascontiguousarray(np.atleast_2d(samples))
        sfx = _suffix(x.dtype)
        b, ns = x.shape
        n = next_pow2(ns) if n_fft is None else int(n_fft)
        k = (4 if flexible else 5) if k is None else int(k)
        cap = max(5, k) if rec_cap is None else int(rec_cap)
        recs = np.zeros(b, dtype=record_dtype(cap))
        fs_scalar, fs_arr = self._fs(fs, b)
        self.ctx.call(f"apda_analyze_{sfx}_host", _p(x.ctypes.data), ns, ns, b, n, center, int(bool(flexible)),
                      fs_scalar, _p(fs_arr.ctypes.data if fs_arr is not None else 0), k, cap, _p(recs.ctypes.data))
        if sfx == "f32" and resolve_ties:
            self._resolve_fp32_ties(x, recs, fs, flexible, k, n, cap, center)
        return recs

    def _resolve_fp32_ties(self, x, recs, fs, flexible, k, n, cap, center) -> None:
        """Windows flagged APDA_STATUS_FP32_TIE (two equal fp32 magnitudes at a peak top: no strict local maximum, so
        the fp32 picker dropped a peak the fp64 reference reports) get the record the fp64 path computes from the same
        samples with the same centring (apda_resolve_fp32_ties_host).  About one window in 10^6 of the fleet generator."""
        b, ns = x.shape
        fs_scalar, fs_arr = self._fs(fs, b)
        self.ctx.call("apda_resolve_fp32_ties_host", _p(x.ctypes.data), _p(0), ns, ns, b, n, center, int(bool(flexible)),
                      fs_scalar, _p(fs_arr.ctypes.data if fs_arr is not None else 0), k, cap, _p(recs.ctypes.data))

    def analyze_fused(self, samples: np.ndarray, fs, flexible: bool = True, k: int | None = None,
                      center: int = _cabi.CENTER_MEDIAN, resolve_ties: bool = False) -> np.ndarray:
        """[B, N] float32, N in {1024, 2048, 4096, 8192} -> records[B] through the fused window->record kernel
        (``resolve_ties``: then the fp64 path's records for the windows flagged APDA_STATUS_FP32_TIE)."""
        x = np.ascontiguousarray(np.atleast_2d(samples), dtype=np.float32)
        b, ns = x.shape
        n = next_pow2(ns)
        k = (4 if flexible else 5) if k is None else int(k)
        recs = np.zeros(b, dtype=record_dtype(5))
        fs_scalar, fs_arr = self._fs(fs, b)
        self.ctx.call("apda_analyze_fused_f32_host", _p(x.ctypes.data), ns, ns, b, n, center, int(bool(flexible)), fs_scalar,
                      _p(fs_arr.ctypes.data if fs_arr is not None else 0), k, 5, _p(recs.ctypes.data))
        if resolve_ties:
            self._resolve_fp32_ties(x, recs, fs, flexible, k, n, 5, center)
        return recs

    def analyze_fused_device(self, d_samples: int, batch: int, n_samples: int, n_fft: int, fs: float, d_rec: int,
                             flexible: bool = True, k: int = 4, center: int = _cabi.CENTER_MEDIAN, d_fs: int = 0,
                             ld: int | None = None, resolve_ties: bool = False) -> None:
        self.ctx.call("apda_analyze_fused_f32_dev", _p(d_samples), n_samples, ld or n_samples, batch, n_fft, center,
                      int(bool(flexible)), float(fs), _p(d_fs), k, 5, _p(d_rec))
        if resolve_ties:
            self.resolve_fp32_ties_device(d_samples, batch, n_samples, n_fft, fs, d_rec, flexible, k, 5, center, d_fs,
                                          0, ld)

    # ---- wire-format ingest (16-bit samples, high byte first) ----------------------------------------------------------
    def decode_wire16(self, payload: np.ndarray, first_value) -> tuple[np.ndarray, np.ndarray]:
        """uint8[B, 2*n] payload rows + baseline per window -> (float64[B, n] compacted samples, int32[B] counts)."""
        pay = np.ascontiguousarray(np.atleast_2d(payload), dtype=np.uint8)
        b, nb = pay.shape
        n = nb // 2
        fv = np.ascontiguousarray(np.broadcast_to(np.asarray(first_value, dtype=np.float64), (b,)))
        out = np.zeros((b, n), dtype=np.float64)
        nv = np.zeros(b, dtype=np.int32)
        self.ctx.call("apda_decode_wire16_f64_host", _p(pay.ctypes.data), n, nb, b, _p(fv.ctypes.data), _p(out.ctypes.data),
                      _p(nv.ctypes.data))
        return out, nv

    def analyze_wire16(self, payload: np.ndarray, first_value, fs, n_fft: int | None = None, dtype: str = "f64",
                       flexible: bool = True, k: int | None = None, strict: bool = False) -> np.ndarray:
        """uint8[B, 2*n] payload rows -> records[B] (decode, drop non-finite, centre, FFT, pick; all on the device).
        Windows that lost samples keep their record but carry status bits (APDA_STATUS_OTHER_LENGTH: the reference
        would have transformed them at their own padded length; APDA_STATUS_EMPTY: its pickers raise): inspect
        ``recs["status"]``, or pass ``strict=True`` to raise when any window is not reference-equivalent."""
        pay = np.ascontiguousarray(np.atleast_2d(payload), dtype=np.uint8)
        b, nb = pay.shape
        n = nb // 2
        nfft = next_pow2(n) if n_fft is None else int(n_fft)
        fv = np.ascontiguousarray(np.broadcast_to(np.asarray(first_value, dtype=np.float64), (b,)))
        k = (4 if flexible else 5) if k is None else int(k)
        cap = max(5, k)
        recs = np.zeros(b, dtype=record_dtype(cap))
        fs_scalar, fs_arr = self._fs(fs, b)
        self.ctx.call(f"apda_analyze_wire16_{dtype}_host", _p(pay.ctypes.data), n, nb, b, _p(fv.ctypes.data), nfft,
                      _cabi.CENTER_MEDIAN, int(bool(flexible)), fs_scalar,
                      _p(fs_arr.ctypes.data if fs_arr is not None else 0), k, cap, _p(recs.ctypes.data))
        if strict:
            _cabi.check_record_status(recs)
        return recs

    # ---- whole sensor .log files ----------------------------------------------------------------------------------
    def analyze_logs(self, paths, n_fft: int, flexible: bool = True, k: int | None = None, dtype: str = "f64",
                     strict: bool = False) -> tuple[np.ndarray, list]:
        """Sensor ``.log`` paths -> (records[B], metas[B]): for every file what ``load_sensor`` followed by ``start_fft`` and
        the picker computes at length ``n_fft`` with the file's own sampling rate (apda_analyze_logs_*_host: the host
        only reads the files; headers, rates and samples are decoded on the device).  ``metas[b]`` is ``{"metadata",
        "summary"}`` as ``load_sensor`` returns them, or None where it returns None.  Files the device leaves undecided
        are re-read with ``load_sensor`` (so its exceptions, e.g. the ``OSError`` of ``open()``, propagate) and analysed
        with ``analyze`` at ``n_fft``.  As on every ragged path, a file whose samples pad to another length carries
        APDA_STATUS_OTHER_LENGTH, one without samples APDA_STATUS_EMPTY; with more than ``n_fft`` samples the record is
        empty with APDA_STATUS_OTHER_LENGTH, and without a fifth line (meta None) empty with APDA_STATUS_EMPTY.
        ``strict=True`` raises on any non-zero record status.  Use "f64" where the reference's samples matter (fp32
        records are not tie-resolved)."""
        import io
        import os
        from .utils import load_data
        if dtype not in ("f64", "f32"):
            raise ValueError(f"dtype must be 'f64' or 'f32', not {dtype!r}")
        paths = [os.fspath(p) for p in paths]
        b = len(paths)
        n = int(n_fft)
        k = (4 if flexible else 5) if k is None else int(k)
        cap = max(5, k)
        recs = np.zeros(b, dtype=record_dtype(cap))
        fs = np.zeros(b, dtype=np.float64)
        nv = np.zeros(b, dtype=np.int32)
        fl = np.zeros(b, dtype=np.int32)
        head = np.zeros((b, _cabi.LOG_HEAD_BYTES), dtype=np.uint8)
        c_paths = (ctypes.c_char_p * max(b, 1))(*[os.fsencode(p) for p in paths])
        self.ctx.call(f"apda_analyze_logs_{dtype}_host", ctypes.cast(c_paths, _p), b, n, _cabi.CENTER_MEDIAN,
                      int(bool(flexible)), k, cap, _p(recs.ctypes.data), _p(fs.ctypes.data), _p(nv.ctypes.data),
                      _p(fl.ctypes.data), _p(head.ctypes.data))
        metas: list = [None] * b
        redo = []
        for i in range(b):
            f = int(fl[i])
            if f & (_cabi.LOG_SAMPLE_UNDECIDED | _cabi.LOG_HEADER_UNDECIDED | _cabi.LOG_UNREADABLE):
                redo.append(i)
                continue
            if f & _cabi.LOG_NO_SAMPLE_LINE:
                continue
            text = head[i].tobytes().split(b"\0", 1)[0].decode("ascii")
            try:
                metadata, summary = load_data._parse_header(io.StringIO(text, newline=None).readlines())
            except (ValueError, IndexError):      # load_sensor raises the same: take its route below
                redo.append(i)
                continue
            metas[i] = {"metadata": metadata, "summary": summary}
        for i in redo:
            got = load_data.load_sensor(paths[i])
            if got is None:
                _empty_record(recs, i, _cabi.STATUS_EMPTY)
                continue
            metas[i] = {"metadata": got["metadata"], "summary": got["summary"]}
            x = np.asarray(got["samples"], dtype=np.float64 if dtype == "f64" else np.float32)
            if x.size > n:
                _empty_record(recs, i, _cabi.STATUS_OTHER_LENGTH)
            elif x.size == 0:
                _empty_record(recs, i, _cabi.STATUS_EMPTY)
            else:
                recs[i] = self.analyze(x[None, :], got["metadata"]["fs"], flexible=flexible, k=k, n_fft=n, rec_cap=cap,
                                       resolve_ties=False)[0]
                if next_pow2(x.size) != n:
                    recs["status"][i] |= _cabi.STATUS_OTHER_LENGTH
        if strict:
            _cabi.check_record_status(recs)
        return recs, metas

    def analyze_host_ptr(self, h_ptr: int, batch: int, n_samples: int, n_fft: int, dtype: str, fs: float,
                         h_rec_ptr: int, flexible: bool = True, k: int = 4, rec_cap: int = 5,
                         center: int = _cabi.CENTER_MEDIAN) -> None:
        """Same as analyze() on caller-owned (ideally pinned) host buffers given by address."""
        self.ctx.call(f"apda_analyze_{dtype}_host", _p(h_ptr), n_samples, n_samples, batch, n_fft, center,
                      int(bool(flexible)), float(fs), _p(0), k, rec_cap, _p(h_rec_ptr))

    # ---- device pointers (torch tensors: pass .data_ptr()) ---------------------------------------------------------
    def use_stream(self, cuda_stream: int | None) -> None:
        self.ctx.set_stream(cuda_stream)

    def fft_device(self, d_samples: int, batch: int, n_samples: int, n_fft: int, dtype: str, d_spec: int,
                   center: int = _cabi.CENTER_MEDIAN, ld: int | None = None) -> None:
        self.ctx.call(f"apda_fft_{dtype}_dev", _p(d_samples), n_samples, ld or n_samples, batch, n_fft, center, _p(d_spec))

    def peaks_device(self, d_spec: int, batch: int, n: int, dtype: str, fs: float, d_rec: int, flexible: bool = True,
                     k: int = 4, rec_cap: int = 5, d_fs: int = 0) -> None:
        kind = "prominence" if flexible else "resolution"
        self.ctx.call(f"apda_peaks_{kind}_{dtype}_dev", _p(d_spec), n, batch, float(fs), _p(d_fs), k, rec_cap, _p(d_rec))

    def analyze_device(self, d_samples: int, batch: int, n_samples: int, n_fft: int, dtype: str, fs: float, d_rec: int,
                       flexible: bool = True, k: int = 4, rec_cap: int = 5, center: int = _cabi.CENTER_MEDIAN,
                       d_spec_ws: int = 0, d_fs: int = 0, ld: int | None = None, resolve_ties: bool = False) -> None:
        """``resolve_ties`` (float32 only): then the fp64 path's records for the windows flagged APDA_STATUS_FP32_TIE,
        enqueued on the same stream (apda_resolve_fp32_ties_dev)."""
        self.ctx.call(f"apda_analyze_{dtype}_dev", _p(d_samples), n_samples, ld or n_samples, batch, n_fft, center,
                      int(bool(flexible)), float(fs), _p(d_fs), k, rec_cap, _p(d_spec_ws), _p(d_rec))
        if resolve_ties and dtype == "f32":
            self.resolve_fp32_ties_device(d_samples, batch, n_samples, n_fft, fs, d_rec, flexible, k, rec_cap, center,
                                          d_fs, 0, ld)

    def resolve_fp32_ties_device(self, d_samples: int, batch: int, n_samples: int, n_fft: int, fs: float, d_rec: int,
                                 flexible: bool = True, k: int = 4, rec_cap: int = 5, center: int = _cabi.CENTER_MEDIAN,
                                 d_fs: int = 0, d_n_valid: int = 0, ld: int | None = None) -> None:
        """Replace the records (written by any fp32 picker route for these float32 samples) whose status is exactly
        APDA_STATUS_FP32_TIE with the fp64 path's records of the widened samples; no host synchronisation."""
        self.ctx.call("apda_resolve_fp32_ties_dev", _p(d_samples), _p(d_n_valid), n_samples, ld or n_samples, batch, n_fft,
                      center, int(bool(flexible)), float(fs), _p(d_fs), k, rec_cap, _p(d_rec))

    # ---- record presentation (the reference's rounded fields, fleet JSONL rows) ----------------------------------------
    def present(self, recs: np.ndarray, fs, n: int, flexible: bool = True, k: int | None = None) -> dict:
        """records[B] -> dict of [B, k] numpy columns ``idx``, ``freq``, ``mag`` (plus ``prominence``, ``damping``,
        ``q_factor`` when ``flexible``): the fields of ``records.prominence_dicts`` / ``resolution_dicts`` computed on the
        device, bit-equal; slots past a window's count hold idx -1 and NaN.  ``k`` defaults to every slot of the record."""
        recs = np.ascontiguousarray(np.atleast_1d(recs))
        cap = recs.dtype["pk"].shape[0]
        k = cap if k is None else int(k)
        b = recs.shape[0]
        names = ["idx", "freq", "mag"] + (["prominence", "damping", "q_factor"] if flexible else [])
        out = {name: np.empty((b, k), dtype=np.int32 if name == "idx" else np.float64) for name in names}
        ptr = {name: _p(a.ctypes.data) for name, a in out.items()}
        fs_scalar, fs_arr = self._fs(fs, b)
        self.ctx.call("apda_present_host", _p(recs.ctypes.data), cap, b, int(n), fs_scalar,
                      _p(fs_arr.ctypes.data if fs_arr is not None else 0), int(bool(flexible)), k, ptr["idx"], ptr["freq"],
                      ptr["mag"], ptr.get("prominence", _p(0)), ptr.get("damping", _p(0)), ptr.get("q_factor", _p(0)))
        return out

    def present_device(self, d_rec: int, batch: int, rec_cap: int, n: int, fs: float, k: int, d_idx: int = 0,
                       d_freq: int = 0, d_mag: int = 0, d_prominence: int = 0, d_damping: int = 0, d_q: int = 0,
                       flexible: bool = True, d_fs: int = 0) -> None:
        """``present`` on device buffers ([batch, k] columns; 0 = not written); no host synchronisation."""
        self.ctx.call("apda_present_dev", _p(d_rec), rec_cap, batch, n, float(fs), _p(d_fs), int(bool(flexible)), k,
                      _p(d_idx), _p(d_freq), _p(d_mag), _p(d_prominence), _p(d_damping), _p(d_q))

    def fleet_jsonl(self, recs: np.ndarray, fs, n: int, flexible: bool = True, k: int = 4, first_window: int = 0,
                    path=None):
        """The text ``records.write_fleet_jsonl`` writes, byte for byte, made on the device: the bytes, or (``path``
        given) the number of rows written to that file."""
        recs = np.ascontiguousarray(np.atleast_1d(recs))
        cap = recs.dtype["pk"].shape[0]
        b = recs.shape[0]
        fs_scalar, fs_arr = self._fs(fs, b)
        text = np.empty(max(1, b * _cabi.jsonl_row_bytes(k)), dtype=np.uint8)
        offsets = np.empty(b + 1, dtype=np.int64)
        self.ctx.call("apda_fleet_jsonl_host", _p(recs.ctypes.data), cap, b, int(n), fs_scalar,
                      _p(fs_arr.ctypes.data if fs_arr is not None else 0), int(bool(flexible)), int(k), int(first_window),
                      _p(text.ctypes.data), text.size, _p(offsets.ctypes.data))
        rows = memoryview(text)[:int(offsets[b])]
        if path is None:
            return bytes(rows)
        with open(path, "wb") as fh:
            fh.write(rows)
        return b

    def fleet_jsonl_device(self, d_rec: int, batch: int, rec_cap: int, n: int, fs: float, d_text: int, text_cap: int,
                           d_offsets: int, flexible: bool = True, k: int = 4, first_window: int = 0,
                           d_fs: int = 0) -> None:
        """``fleet_jsonl`` into device buffers: ``text_cap >= batch * _cabi.jsonl_row_bytes(k)`` bytes of text and
        ``batch + 1`` int64 offsets (row w is text[offsets[w]:offsets[w + 1]]); no host synchronisation."""
        self.ctx.call("apda_fleet_jsonl_dev", _p(d_rec), rec_cap, batch, n, float(fs), _p(d_fs), int(bool(flexible)), k,
                      first_window, _p(d_text), text_cap, _p(d_offsets))

    def synth_device(self, first_window: int, count: int, n: int, dtype: str, d_out: int, seed: int = 42,
                     on_bin: bool = False) -> None:
        self.ctx.call(f"apda_synth_{dtype}_dev", first_window, count, n, seed, int(on_bin), _p(d_out))

    def sync(self) -> None:
        self.ctx.sync()

    def launch_count(self) -> int:
        return self.ctx.launch_count()

    @staticmethod
    def _fs(fs, batch: int):
        if np.isscalar(fs):
            return float(fs), None
        arr = np.ascontiguousarray(fs, dtype=np.float64)
        if arr.shape != (batch,):
            raise ValueError(f"fs must be a scalar or have shape ({batch},)")
        return float(arr[0]) if batch else 0.0, arr


def _empty_record(recs: np.ndarray, i: int, status: int) -> None:
    """The record the device writes for a window with no analysis result: count 0, every slot idx -1 and zeros."""
    recs["count"][i] = 0
    recs["status"][i] = status
    pk = recs["pk"]
    pk["idx"][i] = -1
    pk["width_bins"][i] = 0
    pk["mag"][i] = 0.0
    pk["prominence"][i] = 0.0


def multi_analyze(contexts, samples: np.ndarray, fs, flexible: bool = True, k: int | None = None,
                  n_fft: int | None = None, center: int = _cabi.CENTER_MEDIAN) -> np.ndarray:
    """One process, several GPUs: [B, n_samples] host windows sharded contiguously over ``contexts`` (``_cabi.Context``
    objects of different devices), every device writing its rows of the returned record table
    (apda_multi_analyze_*_host: one host thread per context, no collective)."""
    x = np.ascontiguousarray(np.atleast_2d(samples))
    sfx = _suffix(x.dtype)
    b, ns = x.shape
    n = next_pow2(ns) if n_fft is None else int(n_fft)
    k = (4 if flexible else 5) if k is None else int(k)
    cap = max(5, k)
    recs = np.zeros(b, dtype=record_dtype(cap))
    fs_scalar, fs_arr = Analyzer._fs(fs, b)
    handles = (ctypes.c_void_p * len(contexts))(*[c.handle for c in contexts])
    fn = getattr(_cabi.load(), f"apda_multi_analyze_{sfx}_host")
    _cabi.check(fn(handles, len(contexts), _p(x.ctypes.data), ns, ns, b, n, center, int(bool(flexible)), fs_scalar,
                   _p(fs_arr.ctypes.data if fs_arr is not None else 0), k, cap, _p(recs.ctypes.data)))
    return recs

