"""T2, second round: the parity holes the round-1 review listed (needs a B200: -m gpu).

  * multi-chunk host pipelines with pinned buffers where both pipeline streams use the device-side window lists
    (repair list of the fast pickers, ragged list of the ingest paths) at the same time,
  * record status bits on every ragged path, any k through the drop-ins, the fp32 tie flag,
  * fp32 K2 (N = 2^20 .. 2^24) against the C oracle,
  * result packing (SURVEY 8f rank 4) from a record table produced on the GPU.
"""
import ctypes
import json
import os
import sys

import numpy as np
import pytest

import cases
from oracle import c_oracle, ref_port

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_p = ctypes.c_void_p


@pytest.fixture(scope="module")
def an():
    import apda_fft_b200
    return apda_fft_b200.Analyzer(0)


def _dicts(rec, fs, n, flexible):
    from apda_fft_b200.records import prominence_dicts, resolution_dicts
    return prominence_dicts(rec, fs, n) if flexible else resolution_dicts(rec, fs, n)


# ---------------------------------------------------------------------------------------------------------------
# device-side window lists are per stream
# ---------------------------------------------------------------------------------------------------------------
def test_multichunk_pinned_noise_spectra_repair_list_per_stream(an):
    """More than three chunks of N = 8192 spectra in PINNED memory (so the two pipeline streams really overlap): noise
    plus 680 isolated spikes per window, i.e. 680 hot local maxima - more than the fast picker keeps on chip (160
    candidates for the flexible picker, 640 16-bit hot bins for the rigid one), so every window goes
    through the device-side repair list and the general kernel.  With one list per context, the next chunk's
    memset / appends on the other stream raced with this chunk's; now every record must equal, byte for byte, what the
    general kernel alone produces (apda_ctx_set_generic_only), and the oracle on a sample."""
    import torch
    from apda_fft_b200.records import record_dtype
    n, b = 8192, 3 * 1536 + 200
    rng = np.random.default_rng(77)
    z = torch.empty((b, n, 2), dtype=torch.float32).pin_memory()
    zn = z.numpy()
    zn[:] = rng.standard_normal((b, n, 2), dtype=np.float32)
    zn[:, 0, :] = 0
    for w in range(b):      # isolated spikes (even bins, distinct heights) well above mean + 2 sigma of the window
        at = 2 * rng.permutation(n // 4 - 2)[:680] + 2
        zn[w, at, 0] = 10.0 + 0.5 * rng.random(680, dtype=np.float32)
        zn[w, at, 1] = 0.0
    for flexible in (True, False):
        name = "apda_peaks_prominence_f32_host" if flexible else "apda_peaks_resolution_f32_host"
        k = 4 if flexible else 5
        fast = torch.zeros((b, 128), dtype=torch.uint8).pin_memory()
        slow = torch.zeros((b, 128), dtype=torch.uint8).pin_memory()
        an.ctx.call(name, _p(z.data_ptr()), n, b, 125.0, _p(0), k, 5, _p(fast.data_ptr()))
        an.ctx.set_generic_only(True)
        try:
            an.ctx.call(name, _p(z.data_ptr()), n, b, 125.0, _p(0), k, 5, _p(slow.data_ptr()))
        finally:
            an.ctx.set_generic_only(False)
        f, s = fast.numpy().view(record_dtype(5)).reshape(-1), slow.numpy().view(record_dtype(5)).reshape(-1)
        bad = np.flatnonzero((fast.numpy() != slow.numpy()).any(axis=1))
        assert bad.size == 0, (flexible, bad[:10], f[bad[:3]], s[bad[:3]])
        assert (f["status"] & 1 == 0).all()
        for w in (0, 1535, 1536, 1537, 3071, 3072, b - 1):
            zl = (zn[w, :, 0].astype(np.float64) + 1j * zn[w, :, 1].astype(np.float64)).tolist()
            want = ref_port.top_peaks_prominence(zl, 125.0) if flexible else ref_port.top_peaks_resolution(zl, 125.0)
            got = _dicts(f[w], 125.0, n, flexible)
            assert [p["idx"] for p in got] == [p["idx"] for p in want], (flexible, w)


def _wire_rows(rng, b, n, ragged_every):
    """uint8[b, 2n] wire payloads of finite random words; every `ragged_every`-th window loses samples to inf/nan words."""
    words = rng.integers(0, 1 << 16, size=(b, n), dtype=np.uint16) & np.uint16(0xBFFF)
    lost = np.zeros(b, dtype=np.int64)
    for w in range(0, b, ragged_every):
        kind = (w // ragged_every) % 4
        cnt = {0: 7, 1: n // 2 + 5, 2: n, 3: 1}[kind]          # a few, more than half (other padded length), all, one
        pos = rng.choice(n, size=cnt, replace=False)
        words[w, pos] = np.where(rng.random(cnt) < 0.5, 0x7C00, 0x7E01).astype(np.uint16)
        lost[w] = cnt
    pay = np.empty((b, 2 * n), dtype=np.uint8)
    pay[:, 0::2] = (words >> 8).astype(np.uint8)
    pay[:, 1::2] = (words & 0xFF).astype(np.uint8)
    return pay, lost


@pytest.mark.parametrize("dtype", ["f32", "f64"])
def test_multichunk_wire16_ragged_list_per_stream(dtype, an):
    """apda_analyze_wire16_*_host over several chunks (pinned payload) with ragged windows in every chunk: the records
    must equal those of the same call made slice by slice (each slice a single chunk on one stream), and the status
    bits must follow the per-window sample counts."""
    import torch
    from apda_fft_b200.records import record_dtype
    n = 4096
    chunk = (96 << 20) // (n * 2 * (4 if dtype == "f32" else 8))
    b = 2 * chunk + chunk // 2 + 37
    rng = np.random.default_rng(5)
    pay_np, lost = _wire_rows(rng, b, n, ragged_every=11)
    pay = torch.from_numpy(pay_np).pin_memory()
    fv = torch.from_numpy(rng.uniform(-1, 1, b)).pin_memory()
    whole = torch.zeros((b, 128), dtype=torch.uint8).pin_memory()
    parts = torch.zeros((b, 128), dtype=torch.uint8).pin_memory()

    def run(lo, hi, out):
        an.ctx.call(f"apda_analyze_wire16_{dtype}_host", _p(pay.data_ptr() + lo * 2 * n), n, 2 * n, hi - lo,
                    _p(fv.data_ptr() + 8 * lo), n, 0, 1, 125.0, _p(0), 4, 5, _p(out.data_ptr() + 128 * lo))

    run(0, b, whole)
    step = chunk // 3
    for lo in range(0, b, step):
        run(lo, min(b, lo + step), parts)
    bad = np.flatnonzero((whole.numpy() != parts.numpy()).any(axis=1))
    assert bad.size == 0, bad[:10]
    recs = whole.numpy().view(record_dtype(5)).reshape(-1)
    nv = n - lost
    assert ((recs["status"] & 8 != 0) == (nv == 0)).all()
    other = np.array([v > 0 and c_oracle.padded_len(int(v)) != n for v in nv])
    assert ((recs["status"] & 4 != 0) == other).all()
    assert (recs["status"][lost == 0] & ~16 == 0).all()


def test_ragged_status_bits_on_general_kernel_sizes(an):
    """Status bits 2 / 3 are written on every ragged path, not only where a specialised FFT kernel ran: N = 256 and
    N = 512 have none, and generic_only bypasses them at N = 4096."""
    import torch
    from apda_fft_b200.records import record_dtype
    dev = torch.device("cuda:0")
    an.use_stream(torch.cuda.current_stream(dev).cuda_stream)
    try:
        for n, generic in ((512, False), (256, False), (4096, True)):
            counts = [n, n // 2 - 3, 0, n - 1, n // 2 + 1, 1]
            x = torch.randn((len(counts), n), dtype=torch.float64, device=dev)
            d_nv = torch.tensor(counts, dtype=torch.int32, device=dev)
            d_rec = torch.zeros((len(counts), 128), dtype=torch.uint8, device=dev)
            an.ctx.set_generic_only(generic)
            try:
                an.ctx.call("apda_analyze_ragged_f64_dev", _p(x.data_ptr()), _p(d_nv.data_ptr()), n, n, len(counts), n, 0, 1,
                            125.0, _p(0), 4, 5, _p(0), _p(d_rec.data_ptr()))
                torch.cuda.synchronize()
            finally:
                an.ctx.set_generic_only(False)
            recs = d_rec.cpu().numpy().view(record_dtype(5)).reshape(-1)
            assert [int(s) & 12 for s in recs["status"]] == [0, 4, 8, 0, 0, 4], (n, recs["status"])
            assert recs["count"][2] == 0
    finally:
        an.use_stream(None)


# ---------------------------------------------------------------------------------------------------------------
# any k (reference: get_peak_prominence.py:149,223; get_peak_resolution.py:80,94)
# ---------------------------------------------------------------------------------------------------------------
def test_dropins_accept_any_k():
    sys.path.insert(0, os.path.join(ROOT, "apda-fft_b200"))
    from utils.get_peak_prominence import get_top_peaks_prominence
    from utils.get_peak_resolution import get_top_peaks_resolution
    rng = np.random.default_rng(11)
    for n in (256, 4096, 1 << 17):
        z = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).tolist()
        z[0] = 0
        for k in (65, 100, 5000, 10 ** 6):
            if n > 4096 and k > 100:
                continue
            got = get_top_peaks_prominence(z, 125.0, k)
            want = ref_port.top_peaks_prominence(z, 125.0, k)
            assert got == want, (n, k, len(got), len(want))
            got = get_top_peaks_resolution(z, 125.0, k)
            want = ref_port.top_peaks_resolution(z, 125.0, k)
            assert got == want, (n, k, len(got), len(want))
        if n == 4096:
            assert len(get_top_peaks_resolution(z, 125.0, 100)) > 5      # the wide records were really needed


# ---------------------------------------------------------------------------------------------------------------
# fp32 ties (two equal magnitudes at a peak top)
# ---------------------------------------------------------------------------------------------------------------
def test_fp32_tie_is_flagged_and_resolved_in_fp64(an):
    """A tone exactly half-way between two bins gives two magnitudes that differ only below fp32 resolution.  The fp32
    pickers (strict local maxima, like the reference) then see a plateau and report no peak there; the record carries
    APDA_STATUS_FP32_TIE and Analyzer.analyze re-runs such windows in fp64, which reports what the reference reports."""
    from apda_fft_b200 import _cabi
    n = 4096
    z = np.zeros((3, n), dtype=np.complex64)
    rng = np.random.default_rng(3)
    z[:, 1: n // 2] = (0.01 * (rng.standard_normal((3, n // 2 - 1)) + 1j * rng.standard_normal((3, n // 2 - 1)))).astype(np.complex64)
    for w in range(3):
        z[w, 300] = 40.0
        z[w, 900] = 25.0
    z[1, 500] = z[1, 501] = 30.0 + 0j          # exact tie, higher than the neighbours
    z[2, 500], z[2, 501] = 30.0, 29.0
    for flexible in (True, False):
        recs = an.peaks(z, 125.0, flexible=flexible)
        assert [int(s) for s in recs["status"]] == [0, _cabi.STATUS_FP32_TIE, 0], recs["status"]
        assert 500 not in list(recs[1]["pk"]["idx"]) and 501 not in list(recs[1]["pk"]["idx"])
        assert 500 in list(recs[2]["pk"]["idx"])
        an.ctx.set_generic_only(True)
        try:
            slow = an.peaks(z, 125.0, flexible=flexible)
        finally:
            an.ctx.set_generic_only(False)
        assert [int(s) for s in slow["status"]] == [0, _cabi.STATUS_FP32_TIE, 0]
    # through the sample path: a window whose fp32 spectrum ties is re-run in fp64 by Analyzer.analyze
    i = np.arange(n)
    x = (0.5 * np.sin(2 * np.pi * 200.5 * i / n) + 0.2 * np.sin(2 * np.pi * 611.0 * i / n + 1.0)).astype(np.float32)[None, :]
    raw = an.analyze(x, 125.0, flexible=True, resolve_ties=False)[0]
    fixed = an.analyze(x, 125.0, flexible=True)[0]
    want = c_oracle.peaks_prominence(c_oracle.start_fft_batch(x.astype(np.float64))[0], 125.0)
    if raw["status"] & _cabi.STATUS_FP32_TIE:       # whether fp32 ties here depends on rounding; if it does, it must be resolved
        assert fixed["status"] == 0
    assert [p["idx"] for p in _dicts(fixed, 125.0, n, True)] == [p["idx"] for p in want]


# ---------------------------------------------------------------------------------------------------------------
# K2 fp32 against the oracle at the cfg4 sizes
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("log2n", [20, 22, 24])
def test_cfg4_large_transform_f32_vs_oracle(log2n):
    """fp32 K2 (2-pass plan up to 2^22, 3-pass at 2^24 for fp32 tiles) against the bit-faithful C oracle run on the very
    same (fp32-quantised) samples: every bin within 1e-5 of the window's largest magnitude, peak magnitudes within
    rel 1e-5, peak index lists identical for both pickers."""
    import torch
    import apda_fft_b200
    from apda_fft_b200.records import record_dtype
    dev = torch.device("cuda:0")
    an = apda_fft_b200.Analyzer(0)
    an.use_stream(torch.cuda.current_stream(dev).cuda_stream)
    n = 1 << log2n
    i = np.arange(n, dtype=np.float64)
    x = np.round(0.5 * np.sin(2 * np.pi * 101.6 * i / n) + 0.3 * np.sin(2 * np.pi * 252.4 * i / n + 0.3)
                 + 0.2 * np.sin(2 * np.pi * 498.0 * i / n + 1.1) + 0.01 * np.cos(i * 0.37) + 0.125, 6).astype(np.float32)
    d_x = torch.from_numpy(x[None, :]).to(dev)
    d_spec = torch.empty((1, n, 2), dtype=torch.float32, device=dev)
    an.fft_device(d_x.data_ptr(), 1, n, n, "f32", d_spec.data_ptr())
    recs = {}
    for flexible in (True, False):
        d_rec = torch.zeros((1, 128), dtype=torch.uint8, device=dev)
        an.peaks_device(d_spec.data_ptr(), 1, n, "f32", 125.0, d_rec.data_ptr(), flexible=flexible, k=4 if flexible else 5)
        torch.cuda.synchronize()
        recs[flexible] = d_rec.cpu().numpy().view(record_dtype(5)).reshape(-1)[0]
    got = d_spec.cpu().numpy().view(np.complex64).reshape(n).astype(np.complex128)
    want = c_oracle.start_fft_batch(x.astype(np.float64)[None, :])[0]
    top = np.abs(want).max()
    assert np.abs(got - want).max() <= 1e-5 * top, np.abs(got - want).max() / top
    ref_p = ref_port.top_peaks_prominence(want.tolist(), 125.0)
    ref_r = ref_port.top_peaks_resolution(want.tolist(), 125.0)
    for flexible, ref in ((True, ref_p), (False, ref_r)):
        mine = _dicts(recs[flexible], 125.0, n, flexible)
        assert [p["idx"] for p in mine] == [p["idx"] for p in ref], (flexible, mine, ref)
        for g, r in zip(mine, ref):
            assert abs(g["mag"] - r["mag"]) <= 1e-4 + 1e-5 * r["mag"]
            if flexible:
                assert abs(g["prominence"] - r["prominence"]) <= 1e-5 * r["prominence"]
    assert [p["idx"] for p in ref_p] == [102, 252, 498]


# ---------------------------------------------------------------------------------------------------------------
# (f4) result packing from a table produced on the GPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flexible", [True, False])
def test_result_packing_from_gpu_record_table(flexible, tmp_path, an):
    """Records of a fleet batch computed on the GPU -> columnar Arrow table / JSONL / per-window gateway entries and
    uploader blocks, compared with what the reference's caller (GT_FFT_v5.py:644-659) and uploader
    (utils/fastapi_manager.py:37-47) build from the ORACLE's peaks of the same windows."""
    import apda_fft_b200.synth as synth
    from apda_fft_b200 import records
    b, n, fs, k = 96, 4096, 125.0, 4
    x = synth.fleet_windows(5_000, b, n)
    recs = an.analyze(x, fs, flexible=flexible, k=k)
    spectra = c_oracle.start_fft_batch(x)
    oracle_peaks = [(ref_port.top_peaks_prominence if flexible else ref_port.top_peaks_resolution)(spectra[w].tolist(), fs, k)
                    for w in range(b)]
    table = records.fleet_arrow(recs, fs, n, flexible=flexible, k=k, first_window=5_000)
    assert table.num_rows == b and table.column("window").to_pylist() == list(range(5_000, 5_000 + b))
    idx_col, freq_col, mag_col = (table.column(c).to_pylist() for c in ("idx", "freq", "mag"))
    path = tmp_path / "fleet.jsonl"
    assert records.write_fleet_jsonl(path, recs, fs, n, flexible=flexible, k=k, first_window=5_000) == b
    rows = [json.loads(line) for line in open(path)]
    summary = {"rms_x": 0.011, "rms_y": -0.0222, "rms_z": 0.9981, "temperature": 25.01, "humidity": 85.0}
    for w in range(b):
        want = oracle_peaks[w]
        assert idx_col[w] == [p["idx"] for p in want]
        assert freq_col[w] == [p["idx"] * (fs / n) for p in want]
        if flexible:
            assert [round(m, 4) for m in mag_col[w]] == [p["mag"] for p in want]
        else:
            assert mag_col[w] == [p["mag"] for p in want]
        # the reference caller's dict, built from the oracle's list vs from the GPU record
        ref_entry = {"peak_freq": -1, "max_mag": -1}
        if want:
            ref_entry["peak_freq"], ref_entry["max_mag"] = want[0]["freq"], want[0]["mag"]
            for i, pk in enumerate(want):
                ref_entry[f"peak_freq_{i + 1}"], ref_entry[f"max_mag_{i + 1}"] = pk["freq"], pk["mag"]
        entry = records.gateway_entry(_dicts(recs[w], fs, n, flexible))
        assert entry == ref_entry, w
        up = records.upload_metrics(summary, "Z", entry)
        assert up["fft_freqs"] == [ref_entry.get(f"peak_freq_{i}", 0.0) for i in range(1, 5)]
        assert up["fft_mags"] == [ref_entry.get(f"max_mag_{i}", 0.0) for i in range(1, 5)]
        assert rows[w]["window"] == 5_000 + w
        assert rows[w]["fft_freqs"] == ([p["freq"] for p in want] + [0.0] * k)[:k]
        assert rows[w]["fft_mags"] == ([p["mag"] for p in want] + [0.0] * k)[:k]


# ---------------------------------------------------------------------------------------------------------------
# one host process, several contexts / GPUs (C-ABI gather without a collective)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_multi_analyze_host_equals_single_context(dtype, an):
    """apda_multi_analyze_*_host shards the batch over several contexts (every visible GPU, and two contexts per GPU so
    that a one-GPU box exercises the sharding too): the table must equal the single-context call byte for byte, for a
    batch that does not divide evenly, per-window sampling rates included."""
    import torch
    import apda_fft_b200
    import apda_fft_b200.synth as synth
    from apda_fft_b200 import _cabi
    ndev = torch.cuda.device_count()
    ctxs = [_cabi.Context(d) for d in range(ndev) for _ in range(2)]
    b, n = 1003, 4096
    x = synth.fleet_windows(77, b, n).astype(dtype)
    x[5, :] = 0.25                                   # a constant window (no peaks) in the first shard
    fs = np.linspace(100.0, 200.0, b)
    for flexible in (True, False):
        want = an.analyze(x, fs, flexible=flexible, resolve_ties=False)
        got = apda_fft_b200.multi_analyze(ctxs, x, fs, flexible=flexible)
        assert got.tobytes() == want.tobytes(), flexible
    with pytest.raises(ValueError):
        apda_fft_b200.multi_analyze([ctxs[0], ctxs[0]], x, 125.0)
    for c in ctxs:
        c.close()


def test_half_spectrum_pipeline_equals_full_pipeline(an):
    """apda_analyze_f32_dev with the library's own workspace (K1 writes only bins [0, N/2)) gives the records of
    K1 (N bins) + K3, byte for byte; a caller-provided workspace still receives all N bins."""
    import torch
    dev = torch.device("cuda:0")
    an.use_stream(torch.cuda.current_stream(dev).cuda_stream)
    try:
        for n in (1024, 2048, 4096, 8192):
            b = 777
            x = torch.empty((b, n), dtype=torch.float32, device=dev)
            an.synth_device(123, b, n, "f32", x.data_ptr())
            spec = torch.zeros((b, n, 2), dtype=torch.float32, device=dev)
            ws = torch.zeros((b, n, 2), dtype=torch.float32, device=dev)
            rec_full = torch.zeros((b, 128), dtype=torch.uint8, device=dev)
            rec_half = torch.zeros((b, 128), dtype=torch.uint8, device=dev)
            rec_ws = torch.zeros((b, 128), dtype=torch.uint8, device=dev)
            for flexible in (True, False):
                k = 4 if flexible else 5
                an.fft_device(x.data_ptr(), b, n, n, "f32", spec.data_ptr())
                an.peaks_device(spec.data_ptr(), b, n, "f32", 125.0, rec_full.data_ptr(), flexible=flexible, k=k)
                an.analyze_device(x.data_ptr(), b, n, n, "f32", 125.0, rec_half.data_ptr(), flexible=flexible, k=k)
                an.analyze_device(x.data_ptr(), b, n, n, "f32", 125.0, rec_ws.data_ptr(), flexible=flexible, k=k,
                                  d_spec_ws=ws.data_ptr())
                torch.cuda.synchronize()
                assert torch.equal(rec_full, rec_half) and torch.equal(rec_full, rec_ws), (n, flexible)
                assert torch.equal(ws, spec), n          # all N bins in the caller's workspace
    finally:
        an.use_stream(None)


# ---------------------------------------------------------------------------------------------------------------
# text ingest across several chunks; peer-table flow control words
# ---------------------------------------------------------------------------------------------------------------
def test_multichunk_text_ingest_equals_per_log_calls(an):
    """apda_analyze_text_f32_host over more logs than one chunk holds (ragged: every 7th log is short, every 50th is
    empty or carries non-finite / unparsable pieces): records, sample counts and flags must equal those of the same logs
    sent in small batches (one chunk, one stream each)."""
    from apda_fft_b200.records import record_dtype
    n = 2048
    chunk = (96 << 20) // (n * 2 * 4)
    nlog = chunk + chunk // 3 + 11
    rng = np.random.default_rng(9)
    base_vals = np.round(np.sin(np.arange(n) * 0.21) * 1.3 + 0.2 * np.sin(np.arange(n) * 1.7), 6)
    base = ";".join("%8.6f" % v for v in base_vals) + ";\n"
    short = ";".join("%8.6f" % v for v in base_vals[: n // 2 - 9]) + ";\n"
    nasty = ";".join(["nan", "inf", "* MISSING PACKETS 3-4 *"] + ["%8.6f" % v for v in base_vals[:n - 3]]) + ";\n"
    texts = []
    for i in range(nlog):
        if i % 50 == 49:
            texts.append("" if i % 100 == 99 else nasty)
        elif i % 7 == 6:
            texts.append(short)
        else:
            texts.append(base if i % 2 else base.replace(" ", ""))
    blob = "".join(texts).encode()
    off = np.zeros(nlog + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(t.encode()) for t in texts])
    buf = np.frombuffer(blob, dtype=np.uint8)

    def run(lo, hi, recs, nv, fl):
        sub = off[lo:hi + 1] - off[lo]
        sub = np.ascontiguousarray(sub)
        an.ctx.call("apda_analyze_text_f32_host", _p(buf.ctypes.data + int(off[lo])), _p(sub.ctypes.data), hi - lo, n, n, 0, 1,
                    125.0, _p(0), 4, 5, _p(recs.ctypes.data + 128 * lo), _p(nv.ctypes.data + 4 * lo), _p(fl.ctypes.data + 4 * lo))

    whole = np.zeros(nlog, dtype=record_dtype(5)); nv_w = np.zeros(nlog, dtype=np.int32); fl_w = np.zeros(nlog, dtype=np.int32)
    parts = np.zeros(nlog, dtype=record_dtype(5)); nv_p = np.zeros(nlog, dtype=np.int32); fl_p = np.zeros(nlog, dtype=np.int32)
    run(0, nlog, whole, nv_w, fl_w)
    step = chunk // 4
    for lo in range(0, nlog, step):
        run(lo, min(nlog, lo + step), parts, nv_p, fl_p)
    assert np.array_equal(nv_w, nv_p) and np.array_equal(fl_w, fl_p)
    bad = np.flatnonzero(whole.view(np.uint8).reshape(nlog, 128) != parts.view(np.uint8).reshape(nlog, 128))
    assert bad.size == 0, bad[:10]
    assert (nv_w[[i for i in range(nlog) if i % 7 == 6 and i % 50 != 49]] == n // 2 - 9).all()
    assert (whole["status"][[i for i in range(nlog) if i % 100 == 99]] & 8 != 0).all()          # empty logs
    assert (whole["status"][[i for i in range(nlog) if i % 7 == 6 and i % 50 != 49]] & 4 != 0).all()   # other padded length
    assert (whole["status"][[i for i in range(0, nlog, 2) if i % 7 != 6 and i % 50 != 49]] == 0).all()


def test_peer_wait_times_out_and_resets():
    """apda_peer_wait gives up after its time-out instead of hanging the device (a peer died) and reports THAT wait: the
    word is 1 after a wait on counters that never arrive and 0 again after the next, satisfied wait."""
    import torch
    import apda_fft_b200
    from apda_fft_b200 import _cabi
    ctx = _cabi.Context(0)
    base = ctypes.c_void_p()
    handle = (ctypes.c_ubyte * 64)()
    ctx.call("apda_peer_table_create", ctypes.c_int64(4096), ctypes.byref(base), handle)
    try:
        flags, word = base.value, base.value + 128
        mem = torch.zeros(1)  # noqa: F841 - make sure torch has a CUDA context for the view below

        class _Mem:
            pass
        m = _Mem()
        m.__cuda_array_interface__ = {"shape": (1024,), "typestr": "<i4", "data": (base.value, False), "version": 3, "strides": None}
        view = torch.as_tensor(m, device="cuda:0")
        view.zero_()
        torch.cuda.synchronize()
        ctx.call("apda_peer_signal", _p(flags), 1)                      # rank 0 published step 1, rank 1 never does
        ctx.call("apda_peer_wait", _p(flags), 2, 1, 0.05, _p(word))
        ctx.sync()
        assert int(view[32]) == 1
        ctx.call("apda_peer_signal", _p(flags + 4), 1)
        ctx.call("apda_peer_wait", _p(flags), 2, 1, 0.05, _p(word))
        ctx.sync()
        assert int(view[32]) == 0
    finally:
        ctx.call("apda_peer_table_destroy", _p(base.value))
        ctx.close()


def test_large_window_median_unaligned_rows(an):
    """K2's bracket-select median reads the window with 128-bit loads: rows that start on every possible misalignment
    (batch of windows with an odd number of samples, fp64 rows 8-byte and fp32 rows 4-byte aligned only) must give the
    bit-exact spectrum (fp64) / the exactly median-centred transform (fp32), for short and long windows alike."""
    rng = np.random.default_rng(123)
    for n_samples, n in ((50_001, 1 << 16), (16_387, 1 << 15), (70_003, 1 << 17)):
        x = np.round(rng.standard_normal((5, n_samples)) * 0.3 + 0.77 + 0.2 * np.sin(np.arange(n_samples) * 0.01), 6)
        x[1] = np.round(x[1] * 0 + 0.5, 6)              # a constant window
        x[2, ::2] = 0.25                                 # half the samples equal
        got = an.fft(x, n_fft=n)
        want = c_oracle.start_fft_batch(x, n_fft=n)
        assert np.array_equal(got.view(np.float64), want.view(np.float64)), (n_samples, "fp64")
        x32 = x.astype(np.float32)
        got32 = an.fft(x32, n_fft=n)
        for w in range(x.shape[0]):
            centred = x32[w] - np.float32(np.median(x32[w]))
            ref = np.fft.fft(np.concatenate([centred.astype(np.float64), np.zeros(n - n_samples)]))
            ref[0] = 0
            scale = np.abs(ref).max() + 1e-30
            assert np.abs(got32[w] - ref).max() <= 2e-5 * scale + 1e-3, (n_samples, w)


# ---------------------------------------------------------------------------------------------------------------
# K3 large form: three-level prominence walks (bins / 1024-bin blocks / 32-block groups), grid-wide evaluation
# ---------------------------------------------------------------------------------------------------------------
def _hump_spectrum(log2n, seed):
    """Picker-only spectrum: a noise floor with wide triangular humps placed so that walks stop in the peak's own
    block, in another block of its own group, in another group, and at either end of the spectrum."""
    n = 1 << log2n
    half = n // 2
    rng = np.random.default_rng(seed)
    m = 0.5 + rng.uniform(0.0, 1.0, half)
    i = np.arange(half, dtype=np.float64)

    def hump(centre, height, radius):
        np.maximum(m, height * (1.0 - np.abs(i - centre) / radius), out=m)

    hump(700, 60.0, 300)                         # near the left end: the left walk runs off the spectrum
    hump(40_000, 80.0, 2_000)                    # same group as the next one (blocks 39 and 41)
    hump(42_500, 70.0, 1_500)
    hump(half // 2 + 1_025, 95.0, half // 64)    # the highest: both walks cross every group
    hump(half // 2 + 3 * (half // 8), 85.0, half // 96)
    hump(half - 900, 65.0, 500)                  # right end
    m[0] = 0.0
    z = np.zeros((1, n), dtype=np.complex128)
    z[0, :half] = m
    return z


@pytest.mark.parametrize("log2n", [20, 22])
def test_peaks_large_three_level_walks(log2n, an):
    n = 1 << log2n
    z = _hump_spectrum(log2n, log2n)
    for dt in (np.complex128, np.complex64):
        for flexible in (True, False):
            fast = an.peaks(z.astype(dt), 250.0, flexible=flexible)
            an.ctx.set_generic_only(True)
            try:
                slow = an.peaks(z.astype(dt), 250.0, flexible=flexible)
            finally:
                an.ctx.set_generic_only(False)
            assert fast.tobytes() == slow.tobytes(), (log2n, flexible, dt)
            assert int(fast[0]["count"]) >= 3 and int(fast[0]["status"]) == 0
    # any k, several windows per call (the scratch of the large form is reused window after window)
    z2 = np.concatenate([z, _hump_spectrum(log2n, 77)])
    for flexible in (True, False):
        fast = an.peaks(z2, 250.0, flexible=flexible, k=12)
        an.ctx.set_generic_only(True)
        try:
            slow = an.peaks(z2, 250.0, flexible=flexible, k=12)
        finally:
            an.ctx.set_generic_only(False)
        assert fast.tobytes() == slow.tobytes() and int(fast[1]["count"]) >= 4, (log2n, flexible)
        assert fast[0].tobytes() == an.peaks(z, 250.0, flexible=flexible, k=12)[0].tobytes()
    if log2n == 20:      # the reference-equivalent pure-Python picker is slow at these lengths: once is enough
        assert _dicts(an.peaks(z, 250.0, flexible=True)[0], 250.0, n, True) == c_oracle.peaks_prominence(z[0], 250.0)
        assert _dicts(an.peaks(z, 250.0, flexible=False)[0], 250.0, n, False) == c_oracle.peaks_resolution(z[0], 250.0)


def test_peaks_large_reports_fp32_tie(an):
    """The large form flags an fp32 plateau of two equal top bins like the windowed kernels do."""
    from apda_fft_b200 import _cabi
    n = 1 << 17
    z = _hump_spectrum(17, 5).astype(np.complex64)
    z[0, 30_000] = z[0, 30_001] = 200.0
    for flexible in (True, False):
        fast = an.peaks(z, 250.0, flexible=flexible)
        an.ctx.set_generic_only(True)
        try:
            slow = an.peaks(z, 250.0, flexible=flexible)
        finally:
            an.ctx.set_generic_only(False)
        assert int(fast[0]["status"]) & _cabi.STATUS_FP32_TIE and int(slow[0]["status"]) & _cabi.STATUS_FP32_TIE
        assert fast.tobytes() == slow.tobytes()


# ---------------------------------------------------------------------------------------------------------------
# windowed pickers on noise-like spectra: lazy evaluation in output order (flexible), packed hot list (rigid)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1024, 2048, 4096, 8192])
def test_noise_windows_fast_pickers_equal_general_kernel(n, an):
    """Pure-noise spectra have dozens of hot local maxima (about 2.3 % of the bins).  The fast flexible picker then visits
    the candidates in the reference's output order and evaluates prominence / width / damping only until k are accepted;
    the rigid one keeps bare 16-bit hot bins.  Both must give what the general kernel gives by evaluating everything:
    byte-equal records in fp64, equal index / width lists and magnitudes within fp32 rounding in fp32."""
    rng = np.random.default_rng(n)
    b = 96
    z = (rng.standard_normal((b, n)) + 1j * rng.standard_normal((b, n)))
    z[:, 0] = 0
    z[::7] *= np.linspace(1.0, 3.0, n)[None, :]          # coloured noise: candidates pile up at one end
    z[5::11, 300] = 40.0                                  # one dominant line on top of the noise
    for dt in (np.complex128, np.complex64):
        for flexible in (True, False):
            for k in ((1, 4, 5) if flexible else (2, 5)):
                fast = an.peaks(z.astype(dt), 125.0, flexible=flexible, k=k)
                an.ctx.set_generic_only(True)
                try:
                    slow = an.peaks(z.astype(dt), 125.0, flexible=flexible, k=k)
                finally:
                    an.ctx.set_generic_only(False)
                assert (fast["status"] == 0).all() and (slow["status"] == 0).all()
                if dt is np.complex128:
                    assert fast.tobytes() == slow.tobytes(), (n, flexible, k)
                else:
                    assert np.array_equal(fast["count"], slow["count"]), (n, flexible, k)
                    assert np.array_equal(fast["pk"]["idx"], slow["pk"]["idx"]), (n, flexible, k)
                    assert np.array_equal(fast["pk"]["width_bins"], slow["pk"]["width_bins"]), (n, flexible, k)
                    assert np.allclose(fast["pk"]["mag"], slow["pk"]["mag"], rtol=3e-7, atol=0)
                    assert np.allclose(fast["pk"]["prominence"], slow["pk"]["prominence"], rtol=1e-5, atol=1e-6)
            assert int(fast["count"].max()) >= 2
    # and against the reference-equivalent oracle on a few windows (fp64)
    rec = an.peaks(z[:6], 125.0, flexible=True)
    for w in range(6):
        assert _dicts(rec[w], 125.0, n, True) == c_oracle.peaks_prominence(z[w], 125.0), w


# ---------------------------------------------------------------------------------------------------------------
# exact median of quantised windows (an ADC's levels: the middle value is repeated hundreds of times)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_fft", [1024, 2048, 4096, 8192])
def test_quantised_windows_exact_median(n_fft, an):
    """Sensor words are 16-bit: a window holds a few dozen to a few hundred distinct values and the median value is
    repeated far more often than the selection's final ranking holds.  The in-register counting selection then cuts its
    bracket to the values inside it (plateau -> done).  fp64 spectra must stay bit-identical to the oracle, fp32 within
    the median test's bound; odd, even and padded lengths; plateaus that end exactly at the middle."""
    rng = np.random.default_rng(n_fft + 5)
    for n_samples in (n_fft, n_fft - 1, n_fft // 2 + 3, n_fft // 2 + 4):
        rows = []
        for lv in (50.0, 13.0, 5.0, 1.0, 0.3):                      # sigma in LSB; 1 LSB = 1/16384, offset 0.98 (gravity)
            rows.append(np.round(rng.standard_normal(n_samples) * lv) / 16384.0 + 0.98)
        rows.append((rng.random(n_samples) < 0.5) * 0.25)             # two levels
        rows.append(np.full(n_samples, 0.5))                          # constant
        r = np.full(n_samples, 1.25)                                  # 60 % plateau, outliers on both sides
        m = n_samples // 5
        r[:m] = 1.25 - rng.random(m)
        r[m:2 * m] = 1.25 + rng.random(m)
        rows.append(rng.permutation(r))
        h = np.empty(n_samples)                                       # lower half one value, upper half another
        h[: (n_samples + 1) // 2] = -0.375
        h[(n_samples + 1) // 2:] = 0.625
        rows.append(rng.permutation(h))
        t = np.concatenate([np.full(n_samples // 2 - 1, 2.0), [2.5, 3.0], np.full(n_samples - n_samples // 2 - 1, 4.0)])
        rows.append(rng.permutation(t))                               # single values at the middle between two plateaus
        x = np.stack(rows)
        want = c_oracle.start_fft_batch(x, n_fft=n_fft)
        got = an.fft(x, n_fft=n_fft)
        assert np.array_equal(got.view(np.float64), want.view(np.float64)), (n_fft, n_samples)
        x32 = x.astype(np.float32)
        want32 = c_oracle.start_fft_batch(x32.astype(np.float64), n_fft=n_fft)
        got32 = an.fft(x32, n_fft=n_fft)
        for q in range(x.shape[0]):
            scale = max(np.abs(want32[q]).max(), 1e-3)
            err = np.abs(got32[q].astype(np.complex128) - want32[q]).max()
            assert err <= 3e-6 * scale + n_samples * float(np.abs(x32[q]).max()) * 1.2e-7, (n_fft, n_samples, q, err, scale)


# ---------------------------------------------------------------------------------------------------------------
# batches of long windows: the median kernels of K2 and the large-form picker run many windows per launch set
# ---------------------------------------------------------------------------------------------------------------
def test_batches_of_long_windows_share_launch_sets(an):
    """N = 2^14 (fp64) and 2^15 ... 2^16 windows in batches larger than one launch set (256 windows for the median, 64 for
    the picker): every window's spectrum is bit-identical to the oracle's (fp64) and every record equals the one the same
    window gets when it is sent alone; different lengths, medians and peak positions per window."""
    rng = np.random.default_rng(99)
    for n, b, ns in ((1 << 14, 300, 16000), (1 << 15, 70, 1 << 15), (1 << 16, 70, 60001)):
        i = np.arange(ns, dtype=np.float64)
        x = np.empty((b, ns))
        for w in range(b):
            x[w] = np.round(0.5 * np.sin(2 * np.pi * (101.6 + 3 * w) * i / n) + 0.2 * np.sin(2 * np.pi * 1498.0 * i / n + 0.1 * w)
                            + 0.02 * rng.standard_normal(ns) + 0.01 * w, 6)
        got = an.fft(x, n_fft=n)
        want = c_oracle.start_fft_batch(x, n_fft=n)
        assert np.array_equal(got.view(np.float64), want.view(np.float64)), n
        got32 = an.fft(x.astype(np.float32), n_fft=n)
        scale = np.abs(want).max(axis=1, keepdims=True)
        assert (np.abs(got32.astype(np.complex128) - want) <= 2e-5 * scale).all(), n
        for flexible in (True, False):
            recs = an.analyze(x, 250.0, flexible=flexible, n_fft=n)
            assert (recs["status"] == 0).all()
            for w in (0, 1, 63, 64, 65, b - 1):
                alone = an.analyze(x[w:w + 1], 250.0, flexible=flexible, n_fft=n)
                assert recs[w].tobytes() == alone[0].tobytes(), (n, flexible, w)
            top = recs["pk"]["idx"][:, 0]
            assert np.array_equal(top, np.round(101.6 + 3 * np.arange(b)).astype(top.dtype)), (n, flexible)


# ---------------------------------------------------------------------------------------------------------------
# windowed pickers: peaks, plateaus and hot runs at every structural boundary of the warp-per-window kernels
# ---------------------------------------------------------------------------------------------------------------
def _edge_spectra(n, dtype):
    """Real-valued spectra (magnitude m -> bin m + 0j) whose hot bins sit where the fast pickers change code path:
    bin 0 / 1, the last candidate bin HALF-2 and the non-candidate HALF-1, both sides of quad (4-bin) and lane-chunk
    (HALF/32-bin) boundaries, equal adjacent hot bins (fp32 tie flag) inside a quad, across quads, across chunks and at
    the end of the half spectrum, descending / ascending hot runs (only one local maximum) and a hot quad holding two
    local maxima."""
    half, c = n // 2, (n // 2) // 32
    rng = np.random.default_rng(n)
    layouts = [
        {1: 9.0, 40: 7.0, 500: 5.0},
        {0: 50.0, 2: 8.0, 3: 7.5, 4: 9.5, 300: 6.0},
        {half - 2: 9.0, half - 1: 4.0, 100: 7.0},
        {half - 1: 9.0, half - 3: 6.0, 17: 7.0},
        {c - 1: 9.0, c + 1: 8.0, 2 * c: 7.0, 3 * c - 1: 6.0, 3 * c + 2: 5.5},
        {7: 8.0, 8: 8.0, 200: 6.0},                      # equal pair across a quad boundary
        {c - 1: 8.5, c: 8.5, 300: 6.0},                  # equal pair across a chunk boundary
        {101: 8.0, 102: 8.0, 103: 2.0, 400: 6.0},        # equal pair inside a quad
        {half - 2: 7.0, half - 1: 7.0, 60: 9.0},         # equal pair at the end (no right outer neighbour)
        {200: 10.0, 201: 9.0, 202: 8.0, 199: 8.5, 198: 7.0},   # hot run around one maximum
        {320: 6.0, 322: 9.0, 321: 1.0, 323: 5.0},        # two local maxima in one quad
        {4 * 77: 9.0, 4 * 77 + 3: 8.0, 4 * 78: 8.5},     # maxima at both ends of a quad and the start of the next
        {5: 6.0, 6: 6.0, 7: 6.0, 900 % half: 9.0},       # three equal bins: no plateau top with a strict outer neighbour pair
    ]
    z = np.zeros((len(layouts), n), dtype=np.complex64 if dtype == np.float32 else np.complex128)
    for w, lay in enumerate(layouts):
        mag = (0.01 + 0.01 * rng.random(half)).astype(dtype)
        for b_, m in lay.items():
            mag[b_ % half] = dtype(m)
        z[w, :half] = mag
        z[w, half:] = mag[::-1]
    return z


@pytest.mark.parametrize("n", [1024, 4096, 8192])
def test_fast_pickers_at_quad_chunk_and_end_boundaries(n, an):
    """The specialised pickers (fp32 and fp64) against the general kernel (byte-equal records, tie status included) and the
    oracle (index lists) on spectra whose hot bins sit on every quad / chunk / end-of-spectrum boundary."""
    for dtype in (np.float32, np.float64):
        z = _edge_spectra(n, dtype)
        for flexible in (True, False):
            fast = an.peaks(z, 250.0, flexible=flexible)
            an.ctx.set_generic_only(True)
            try:
                slow = an.peaks(z, 250.0, flexible=flexible)
            finally:
                an.ctx.set_generic_only(False)
            for w in range(z.shape[0]):
                assert fast[w].tobytes() == slow[w].tobytes(), (n, dtype.__name__, flexible, w, fast[w], slow[w])
                zl = z[w].astype(np.complex128).tolist()
                want = ref_port.top_peaks_prominence(zl, 250.0) if flexible else ref_port.top_peaks_resolution(zl, 250.0)
                got = _dicts(fast[w], 250.0, n, flexible)
                assert [p["idx"] for p in got] == [p["idx"] for p in want], (n, dtype.__name__, flexible, w)
            assert ((fast["status"] & ~16) == 0).all()
