"""apda_resolve_fp32_ties_{dev,host}: records flagged APDA_STATUS_FP32_TIE (status exactly 16) get the fp64 path's
record of the widened samples; every other byte stays as it was.

Tie-rich windows: two equal-amplitude on-bin tones at adjacent bins j, j+1 plus a third tone.  In exact arithmetic
|X[j]| == |X[j+1]|; the fp64 reference sees the rounding of the fp32 samples and reports one of the two bins, while the
fp32 magnitudes are often exactly equal, so the fp32 pickers find no strict local maximum there and flag the window.
For a padded window (n_samples = N - 1) every tone is phased to be exactly 0 at the dropped sample i = N - 1, and so
that the median's leakage (|med| at every bin, phase 2*pi*j/N) is orthogonal to both tone bins: the tie survives the
padding and the centring.

Every resolved record is held byte for byte to apda_analyze_f64_dev (apda_analyze_ragged_f64_dev) on the widened
samples, and its index list to the C oracle where the reference's median centring applies.
"""
import contextlib
import ctypes

import numpy as np
import pytest

from oracle import c_oracle

_p = ctypes.c_void_p
SENT = 0xA5
GUARD = 4096
CENTER_MEDIAN, CENTER_MEAN, CENTER_NONE = 0, 1, 2
TIE, OTHER_LENGTH, EMPTY = 16, 4, 8
SIZES = [64, 256, 512, 1024, 2048, 4096, 8192]


def rec_dtype(cap):
    peak = np.dtype([("idx", "<i4"), ("width_bins", "<i4"), ("mag", "<f8"), ("prominence", "<f8")])
    return np.dtype([("count", "<i4"), ("status", "<i4"), ("pk", peak, (cap,))])


def tie_windows(b, n, n_samples=None, seed=0, zero_tail=None):
    """float32[b, n_samples] tie-rich windows (see the module docstring) and their tone bins j.  zero_tail (default:
    padded windows) fixes the phases so that every tone is 0 at i = n - 1; otherwise the phases are random."""
    ns = n if n_samples is None else n_samples
    zero_tail = ns < n if zero_tail is None else zero_tail
    rng = np.random.default_rng(seed)
    half = n // 2
    lo, hi = 16, min(400, half - 5)
    j = rng.integers(lo, hi + 1, size=b)
    m = rng.integers(8, half - 3, size=b)
    clash = np.abs(m - j) < 4
    m[clash] = np.where(j[clash] + 6 < half - 3, j[clash] + 6, j[clash] - 6)
    a = rng.uniform(0.5, 2.0, size=b)
    c = a * rng.uniform(0.3, 0.9, size=b)
    i = np.arange(ns, dtype=np.float64)[None, :]
    if not zero_tail:
        ph1, ph2, ph3 = (rng.uniform(0, 2 * np.pi, size=b) for _ in range(3))
    else:  # each tone 0 at i = n - 1, median leakage orthogonal to bins j and j+1
        ph1 = 2 * np.pi * j / n + np.pi / 2
        ph2 = ph1 + np.pi + 2 * np.pi / n
        ph3 = 2 * np.pi * m / n + np.pi / 2
    w = 2 * np.pi / n
    x = (a[:, None] * np.cos(w * j[:, None] * i + ph1[:, None]) + a[:, None] * np.cos(w * (j + 1)[:, None] * i + ph2[:, None])
         + c[:, None] * np.cos(w * m[:, None] * i + ph3[:, None]))
    return x.astype(np.float32), j


def test_tie_generator_premise():
    """No GPU: numpy's fp32 FFT of the generator's windows has equal magnitudes at j, j+1 on a large share of windows,
    and the fp64 FFT of the same (widened) samples on none."""
    x, j = tie_windows(2000, 4096)
    r = np.arange(len(j))
    m32 = np.abs(np.fft.fft(x, axis=1).astype(np.complex64))
    m64 = np.abs(np.fft.fft(x.astype(np.float64), axis=1))
    assert (m32[r, j] == m32[r, j + 1]).mean() >= 0.2
    assert (m64[r, j] == m64[r, j + 1]).mean() <= 0.01
    xp, jp = tie_windows(64, 4096, 4095, seed=3)
    full, _ = tie_windows(64, 4096, 4096, seed=3, zero_tail=True)
    assert np.abs(full[:, -1]).max() < 1e-6          # the dropped sample is (up to rounding) zero
    assert np.array_equal(xp, full[:, :4095])


# ---------------------------------------------------------------------------------------------------------------
# device helpers
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def an():
    import torch
    import apda_fft_b200
    a = apda_fft_b200.Analyzer(0)
    a.use_stream(torch.cuda.current_stream(torch.device("cuda:0")).cuda_stream)
    yield a
    a.use_stream(None)


@contextlib.contextmanager
def generic(an, on):
    an.ctx.set_generic_only(on)
    try:
        yield
    finally:
        an.ctx.set_generic_only(False)


class Guarded:
    """Device buffer of `nbytes` between GUARD sentinel bytes; optional initial content."""

    def __init__(self, nbytes, init=None):
        import torch
        self.n = int(nbytes)
        self.buf = torch.full((2 * GUARD + self.n,), SENT, dtype=torch.uint8, device="cuda:0")
        if init is not None:
            self.buf[GUARD:GUARD + self.n] = torch.from_numpy(np.ascontiguousarray(init).view(np.uint8).reshape(-1)).cuda()
        self.ptr = self.buf.data_ptr() + GUARD

    def bytes(self):
        import torch
        torch.cuda.synchronize()
        h = self.buf.cpu().numpy()
        assert (h[:GUARD] == SENT).all(), "bytes before the buffer were written"
        assert (h[GUARD + self.n:] == SENT).all(), "bytes after the buffer were written"
        return h[GUARD:GUARD + self.n].copy()


def rows_on_device(x, ld=None, off=0):
    """x[b, ns] at row pitch ld from element `off` of a NaN-filled float32 device buffer -> (buffer, row-0 address)."""
    import torch
    b, ns = x.shape
    ld = ns if ld is None else ld
    buf = torch.full((off + b * ld + 67,), float("nan"), dtype=torch.float32, device="cuda:0")
    buf[off:off + b * ld].view(b, ld)[:, :ns] = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return buf, buf.data_ptr() + off * 4


def k_default(flexible):
    return 4 if flexible else 5


def fp32_records(an, route, ptr, ns, ld, b, n, flexible, k, cap, fs=125.0, d_fs=0, flags=CENTER_MEDIAN, d_nv=None):
    """Records of one fp32 route as a sentinel-guarded device buffer (plus the caller's spectrum workspace, if any)."""
    import torch
    rec = Guarded(b * rec_dtype(cap).itemsize)
    rec.rows = b
    ws = None
    if route in ("split", "split_generic"):
        spec = torch.empty((b, n, 2), dtype=torch.float32, device="cuda:0")
        with generic(an, route == "split_generic"):
            an.ctx.call("apda_fft_f32_dev", _p(ptr), ns, ld, b, n, flags, _p(spec.data_ptr()))
            kind = "prominence" if flexible else "resolution"
            an.ctx.call(f"apda_peaks_{kind}_f32_dev", _p(spec.data_ptr()), n, b, fs, _p(d_fs), k, cap, _p(rec.ptr))
    elif route in ("analyze", "analyze_ws"):
        if route == "analyze_ws":
            ws = Guarded(b * n * 8)
        an.ctx.call("apda_analyze_f32_dev", _p(ptr), ns, ld, b, n, flags, int(flexible), fs, _p(d_fs), k, cap,
                    _p(ws.ptr if ws else 0), _p(rec.ptr))
    elif route == "fused":
        an.ctx.call("apda_analyze_fused_f32_dev", _p(ptr), ns, ld, b, n, flags, int(flexible), fs, _p(d_fs), k, cap,
                    _p(rec.ptr))
    elif route == "ragged":
        if d_nv is None:
            d_nv = torch.full((b,), ns, dtype=torch.int32, device="cuda:0")
        an.ctx.call("apda_analyze_ragged_f32_dev", _p(ptr), _p(d_nv.data_ptr()), ns, ld, b, n, flags, int(flexible), fs,
                    _p(d_fs), k, cap, _p(0), _p(rec.ptr))
    else:
        raise ValueError(route)
    return rec, ws


def set_status(rec, rows, value):
    """Overwrite the status word of some records in a Guarded device table."""
    import torch
    h = rec.bytes()
    rb = h.size // rec.rows
    for w in rows:
        h[w * rb + 4: w * rb + 8] = np.array([value], dtype="<i4").view(np.uint8)
    rec.buf[GUARD:GUARD + rec.n] = torch.from_numpy(h).cuda()


def resolve_dev(an, ptr, ns, ld, b, n, flexible, k, cap, rec, fs=125.0, d_fs=0, flags=CENTER_MEDIAN, d_nv=0):
    an.ctx.call("apda_resolve_fp32_ties_dev", _p(ptr), _p(d_nv), ns, ld, b, n, flags, int(flexible), fs, _p(d_fs), k, cap,
                _p(rec.ptr))


def f64_records(an, x, n, flexible, k, cap, fs=125.0, fs_arr=None, flags=CENTER_MEDIAN, nv=None):
    """apda_analyze_f64_dev (apda_analyze_ragged_f64_dev with nv) on the widened samples, as bytes [b, rec]."""
    import torch
    b, ns = x.shape
    d_x = torch.from_numpy(x.astype(np.float64)).cuda()
    d_fs = torch.from_numpy(fs_arr).cuda() if fs_arr is not None else None
    rec = Guarded(b * rec_dtype(cap).itemsize)
    if nv is None:
        an.ctx.call("apda_analyze_f64_dev", _p(d_x.data_ptr()), ns, ns, b, n, flags, int(flexible), fs,
                    _p(d_fs.data_ptr() if d_fs is not None else 0), k, cap, _p(0), _p(rec.ptr))
    else:
        d_nv = torch.from_numpy(nv).cuda()
        an.ctx.call("apda_analyze_ragged_f64_dev", _p(d_x.data_ptr()), _p(d_nv.data_ptr()), ns, ns, b, n, flags,
                    int(flexible), fs, _p(d_fs.data_ptr() if d_fs is not None else 0), k, cap, _p(0), _p(rec.ptr))
    return rec.bytes().reshape(b, -1)


def oracle_idx(x_row64, n, flexible, k, fs):
    spec = c_oracle.start_fft_batch(x_row64[None, :], n)[0]
    out = c_oracle.peaks_prominence(spec, fs, k) if flexible else c_oracle.peaks_resolution(spec, fs, k)
    return [p["idx"] for p in out]


def check_resolved(before, after, want64, cap, x=None, n=None, flexible=True, k=4, fs=None, oracle_max=12):
    """before/after: fp32 record bytes [b, rec] around the resolver; want64: the fp64 path's bytes for every window.
    Returns the indices of the windows that were resolved."""
    dt = rec_dtype(cap)
    rb, ra = before.view(dt).reshape(-1), after.view(dt).reshape(-1)
    tied = np.flatnonzero(rb["status"] == TIE)
    keep = np.flatnonzero(rb["status"] != TIE)
    assert np.array_equal(after[keep], before[keep]), "a record without status 16 changed"
    assert np.array_equal(after[tied], want64[tied]), "a resolved record differs from the fp64 path's"
    assert (ra["status"][tied] == 0).all()
    if x is not None:
        for w in tied[:oracle_max]:
            f = 125.0 if fs is None else float(fs[w])
            got = [int(v) for v in ra["pk"]["idx"][w][: ra["count"][w]]]
            assert got == oracle_idx(x[w].astype(np.float64), n, flexible, k, f), w
    return tied


# ---------------------------------------------------------------------------------------------------------------
# 1. every route, every size
# ---------------------------------------------------------------------------------------------------------------
ROUTES = ["split", "split_generic", "analyze", "analyze_ws", "fused", "ragged"]


@pytest.mark.gpu
@pytest.mark.parametrize("flexible", [True, False], ids=["prom", "res"])
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("route", ROUTES)
def test_every_route_every_size(an, route, n, flexible):
    if route == "fused" and n < 1024:
        pytest.skip("the fused kernel serves N = 1024 ... 8192")
    b = 192
    k = k_default(flexible)
    x, _ = tie_windows(b, n, seed=n + 7 * flexible)
    buf, ptr = rows_on_device(x)
    samples_before = buf.cpu().numpy().copy()
    rec, ws = fp32_records(an, route, ptr, n, n, b, n, flexible, k, 5)
    before = rec.bytes().reshape(b, -1)
    ws_before = ws.bytes() if ws else None
    resolve_dev(an, ptr, n, n, b, n, flexible, k, 5, rec)
    after = rec.bytes().reshape(b, -1)
    want = f64_records(an, x, n, flexible, k, 5)
    tied = check_resolved(before, after, want, 5, x, n, flexible, k)
    assert len(tied) >= 0.2 * b, f"only {len(tied)} of {b} windows flagged"
    dt = rec_dtype(5)
    rb, ra = before.view(dt).reshape(-1), after.view(dt).reshape(-1)
    assert any(list(rb["pk"]["idx"][w]) != list(ra["pk"]["idx"][w]) for w in tied), "no resolved list differs"
    assert np.array_equal(buf.cpu().numpy(), samples_before, equal_nan=True), "samples were written"
    if ws is not None:
        assert np.array_equal(ws.bytes(), ws_before), "the caller's spectrum workspace was written"


# ---------------------------------------------------------------------------------------------------------------
# 2. inputs: centrings, strided / misaligned rows, k, rec_cap, per-window fs
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("flexible", [True, False], ids=["prom", "res"])
@pytest.mark.parametrize("flags,padded", [(CENTER_MEDIAN, False), (CENTER_MEDIAN, True), (CENTER_NONE, False),
                                          (CENTER_NONE, True), (CENTER_MEAN, False)],
                         ids=["median", "median-padded", "none", "none-padded", "mean"])
@pytest.mark.parametrize("n", [1024, 4096])
def test_centrings(an, n, flags, padded, flexible):
    """Candidates from a device-side search: the fp32 analysis without resolution, keeping what it flags (plus as many
    unflagged windows).  CENTER_MEAN is resolved with the reference's median."""
    k = k_default(flexible)
    ns = n - 1 if padded else n
    cand, _ = tie_windows(1024, n, ns, seed=11 + n)
    _, cptr = rows_on_device(cand)
    crec, _ = fp32_records(an, "analyze", cptr, ns, ns, len(cand), n, flexible, k, 5, flags=flags)
    st = crec.bytes().view(rec_dtype(5))["status"]
    flagged = np.flatnonzero(st == TIE)
    assert flagged.size >= 8, f"the search found {flagged.size} flagged windows"
    pick = np.sort(np.concatenate([flagged[:96], np.flatnonzero(st == 0)[:96]]))
    x = cand[pick]
    b = len(x)
    _, ptr = rows_on_device(x)
    rec, _ = fp32_records(an, "analyze", ptr, ns, ns, b, n, flexible, k, 5, flags=flags)
    before = rec.bytes().reshape(b, -1)
    resolve_dev(an, ptr, ns, ns, b, n, flexible, k, 5, rec, flags=flags)
    after = rec.bytes().reshape(b, -1)
    want = f64_records(an, x, n, flexible, k, 5, flags=CENTER_MEDIAN if flags == CENTER_MEAN else flags)
    ref = x if flags != CENTER_NONE else None          # the oracle centres with the median
    tied = check_resolved(before, after, want, 5, ref, n, flexible, k)
    assert tied.size >= 8


@pytest.mark.gpu
@pytest.mark.parametrize("ld_extra,off", [(1, 1), (3, 3), (64, 1)])
@pytest.mark.parametrize("route", ["analyze", "ragged", "fused"])
def test_strided_misaligned_rows(an, route, ld_extra, off):
    """Rows at pitch ld > n_samples from element offsets 1 and 3, NaN in the gaps: the resolved records equal those of
    contiguous rows (reading at n_samples instead of ld would pull NaN into the transform)."""
    n, b, k = 2048, 160, 4
    x, _ = tie_windows(b, n, seed=5)
    _, ptr = rows_on_device(x, n + ld_extra, off)
    rec, _ = fp32_records(an, route, ptr, n, n + ld_extra, b, n, True, k, 5)
    before = rec.bytes().reshape(b, -1)
    resolve_dev(an, ptr, n, n + ld_extra, b, n, True, k, 5, rec)
    after = rec.bytes().reshape(b, -1)
    tied = check_resolved(before, after, f64_records(an, x, n, True, k, 5), 5, x, n, True, k)
    assert tied.size >= 0.2 * b


@pytest.mark.gpu
@pytest.mark.parametrize("flexible", [True, False], ids=["prom", "res"])
@pytest.mark.parametrize("k,cap", [(1, 5), (2, 5), (3, 5), (5, 5), (4, 16), (5, 64), (16, 16), (5, "max")])
def test_k_rec_cap_and_fs(an, k, cap, flexible):
    """k = 1..5 and wider records, with a pseudo-random sampling rate per window through d_fs.  The pickers' decisions
    depend on fs only through rounding, except at fs = 0 (flexible picker: every half-power width is 0 Hz, so the
    reference reports no peak): every fifth window gets that rate, so a window judged at another window's rate shows."""
    import torch
    n, b = 4096, 160
    cap = int(n // 8 + 8) if cap == "max" else cap
    x, _ = tie_windows(b, n, seed=k * 100 + cap)
    fs = np.random.default_rng(k + cap).uniform(50.0, 3000.0, size=b)
    if flexible:
        fs[::5] = 0.0
    d_fs = torch.from_numpy(fs).cuda()
    _, ptr = rows_on_device(x)
    rec, _ = fp32_records(an, "analyze", ptr, n, n, b, n, flexible, k, cap, fs=1.0, d_fs=d_fs.data_ptr())
    before = rec.bytes().reshape(b, -1)
    resolve_dev(an, ptr, n, n, b, n, flexible, k, cap, rec, fs=1.0, d_fs=d_fs.data_ptr())
    after = rec.bytes().reshape(b, -1)
    want = f64_records(an, x, n, flexible, k, cap, fs=1.0, fs_arr=fs)
    tied = check_resolved(before, after, want, cap, x, n, flexible, k, fs=fs)
    assert tied.size >= 0.2 * b


# ---------------------------------------------------------------------------------------------------------------
# 3. ragged batches
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("flexible", [True, False], ids=["prom", "res"])
@pytest.mark.parametrize("n", [1024, 4096, 8192])
def test_ragged_counts(an, n, flexible):
    """Counts: full, one short (same padded length), another padded length, empty.  Only status exactly 16 changes;
    16 | OTHER_LENGTH records keep every byte."""
    import torch
    k = k_default(flexible)
    b = 256
    full, _ = tie_windows(b, n, seed=n + 1)
    short, _ = tie_windows(b, n, n - 1, seed=n + 2)
    x = full.copy()
    kind = np.arange(b) % 4
    x[kind == 1, : n - 1] = short[kind == 1]
    nv = np.where(kind == 0, n, np.where(kind == 1, n - 1, np.where(kind == 2, n // 2 - 1, 0))).astype(np.int32)
    x[kind == 2, n // 2 - 1:] = 0.0
    d_nv = torch.from_numpy(nv).cuda()
    _, ptr = rows_on_device(x)
    rec, _ = fp32_records(an, "ragged", ptr, n, n, b, n, flexible, k, 5, d_nv=d_nv)
    set_status(rec, np.flatnonzero(kind == 2)[::3], TIE | OTHER_LENGTH)  # a tie in a window of another padded length
    before = rec.bytes().reshape(b, -1)
    resolve_dev(an, ptr, n, n, b, n, flexible, k, 5, rec, d_nv=d_nv.data_ptr())
    after = rec.bytes().reshape(b, -1)
    want = f64_records(an, x, n, flexible, k, 5, nv=nv)
    tied = check_resolved(before, after, want, 5)
    st = before.view(rec_dtype(5))["status"]
    assert set(kind[tied]) <= {0, 1} and (kind[tied] == 0).any() and (kind[tied] == 1).any()
    assert (st == TIE | OTHER_LENGTH).any() and (st == OTHER_LENGTH).any() and (st == EMPTY).any()
    for w in tied[:8]:
        got = after[w].view(rec_dtype(5))[0]
        assert [int(v) for v in got["pk"]["idx"][: got["count"]]] == oracle_idx(x[w, : nv[w]].astype(np.float64), n,
                                                                                 flexible, k, 125.0)


# ---------------------------------------------------------------------------------------------------------------
# 4. host twin and the Analyzer
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("ragged", [False, True], ids=["full", "ragged"])
@pytest.mark.parametrize("n", [256, 4096, 8192])
def test_host_equals_dev(an, n, ragged):
    import torch
    b, k, cap = 300, 4, 5
    x, _ = tie_windows(b, n, seed=n + 31)
    fs = np.random.default_rng(n).uniform(60.0, 900.0, size=b)
    fs[::5] = 0.0                                   # see test_k_rec_cap_and_fs
    nv = np.where(np.arange(b) % 3 == 2, n - 1, n).astype(np.int32) if ragged else None
    d_fs = torch.from_numpy(fs).cuda()
    d_nv = torch.from_numpy(nv).cuda() if ragged else None
    _, ptr = rows_on_device(x)
    rec, _ = fp32_records(an, "ragged" if ragged else "analyze", ptr, n, n, b, n, True, k, cap, fs=1.0,
                          d_fs=d_fs.data_ptr(), d_nv=d_nv)
    before = rec.bytes().reshape(b, -1)
    h = before.copy()
    an.ctx.call("apda_resolve_fp32_ties_host", _p(x.ctypes.data), _p(nv.ctypes.data if ragged else 0), n, n, b, n,
                CENTER_MEDIAN, 1, 1.0, _p(fs.ctypes.data), k, cap, _p(h.ctypes.data))
    resolve_dev(an, ptr, n, n, b, n, True, k, cap, rec, fs=1.0, d_fs=d_fs.data_ptr(),
                d_nv=d_nv.data_ptr() if ragged else 0)
    after = rec.bytes().reshape(b, -1)
    assert (before.view(rec_dtype(cap))["status"] == TIE).sum() >= 0.2 * b
    assert np.array_equal(h, after)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [16384, 65536])
def test_host_large_n(an, n):
    """Beyond one CTA in fp64: the fp64 analysis pipeline on the gathered windows.  Windows are marked status 16 in the
    host table (the resolver re-runs exactly those), one with 16 | 4 must stay as it is."""
    b, k, cap = 12, 4, 5
    x, _ = tie_windows(b, n, seed=n)
    xs = np.full((b, n + 5), np.nan, dtype=np.float32)
    xs[:, :n] = x
    recs = np.zeros(b, dtype=rec_dtype(cap))
    an.ctx.call("apda_analyze_f32_host", _p(xs.ctypes.data), n, n + 5, b, n, CENTER_MEDIAN, 1, 125.0, _p(0), k, cap,
                _p(recs.ctypes.data))
    recs["status"][[1, 4, 7, 8]] = TIE
    recs["status"][10] = TIE | OTHER_LENGTH
    before = recs.copy()
    mark = np.flatnonzero(recs["status"] == TIE)
    an.ctx.call("apda_resolve_fp32_ties_host", _p(xs.ctypes.data), _p(0), n, n + 5, b, n, CENTER_MEDIAN, 1, 125.0, _p(0),
                k, cap, _p(recs.ctypes.data))
    want = np.zeros(len(mark), dtype=rec_dtype(cap))
    xw = np.ascontiguousarray(x[mark].astype(np.float64))
    an.ctx.call("apda_analyze_f64_host", _p(xw.ctypes.data), n, n, len(mark), n, CENTER_MEDIAN, 1, 125.0, _p(0), k, cap,
                _p(want.ctypes.data))
    assert recs[mark].tobytes() == want.tobytes()
    rest = np.setdiff1d(np.arange(b), mark)
    assert recs[rest].tobytes() == before[rest].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("flexible", [True, False], ids=["prom", "res"])
def test_analyzer_median_matches_python_rerun(an, flexible):
    """Analyzer.analyze with CENTER_MEDIAN: byte-equal to the fp64 re-run in Python the library used before."""
    n, b = 4096, 200
    x, _ = tie_windows(b, n, seed=77)
    fs = np.random.default_rng(1).uniform(80.0, 500.0, size=b)
    got = an.analyze(x, fs, flexible=flexible)
    old = an.analyze(x, fs, flexible=flexible, resolve_ties=False)
    tied = np.flatnonzero(old["status"] & TIE)
    assert tied.size >= 0.2 * b
    old[tied] = an.analyze(x[tied].astype(np.float64), fs[tied], flexible=flexible, n_fft=n)
    assert got.tobytes() == old.tobytes()


@pytest.mark.gpu
def test_analyzer_center_none_padded(an):
    """Analyzer.analyze with CENTER_NONE on padded windows: the resolved records are the fp64 analysis with CENTER_NONE
    (the old Python re-run centred them with the median)."""
    n = 4096
    cand, _ = tie_windows(1024, n, n - 1, seed=99)
    raw = an.analyze(cand, 125.0, n_fft=n, center=CENTER_NONE, resolve_ties=False)
    x = cand[np.flatnonzero(raw["status"] == TIE)[:64]]
    assert len(x) >= 8
    got = an.analyze(x, 125.0, n_fft=n, center=CENTER_NONE)
    want = an.analyze(x.astype(np.float64), 125.0, n_fft=n, center=CENTER_NONE)
    assert (got["status"] == 0).all()
    assert got.tobytes() == want.tobytes()


# ---------------------------------------------------------------------------------------------------------------
# 5. the fleet
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cfg5_fleet_split_pipeline(an):
    """1M x 4096 fp32 (generator seed 42) through K1 + K3, then the resolver: every status 0, and every formerly tied
    window equals the oracle's dicts."""
    import torch
    from apda_fft_b200.records import prominence_dicts
    b, n = 1_000_000, 4096
    need = b * n * 4 + b * n * 8 + b * 128
    free, _ = torch.cuda.mem_get_info()
    if free < need + (1 << 30):
        pytest.skip(f"needs {need + (1 << 30)} bytes of device memory, {free} free")
    d_x = torch.empty((b, n), dtype=torch.float32, device="cuda:0")
    an.synth_device(0, b, n, "f32", d_x.data_ptr(), seed=42)
    d_spec = torch.empty((b, n, 2), dtype=torch.float32, device="cuda:0")
    d_rec = torch.zeros((b, 128), dtype=torch.uint8, device="cuda:0")
    an.fft_device(d_x.data_ptr(), b, n, n, "f32", d_spec.data_ptr())
    an.peaks_device(d_spec.data_ptr(), b, n, "f32", 125.0, d_rec.data_ptr(), flexible=True, k=4)
    torch.cuda.synchronize()
    before = d_rec.cpu().numpy().view(rec_dtype(5)).reshape(-1)
    an.resolve_fp32_ties_device(d_x.data_ptr(), b, n, n, 125.0, d_rec.data_ptr(), flexible=True, k=4)
    torch.cuda.synchronize()
    after = d_rec.cpu().numpy().view(rec_dtype(5)).reshape(-1)
    tied = np.flatnonzero(before["status"] == TIE)
    assert (after["status"] == 0).all()
    keep = np.flatnonzero(before["status"] != TIE)
    assert after[keep].tobytes() == before[keep].tobytes()
    if tied.size:
        xs = d_x[torch.as_tensor(tied, device="cuda:0")].cpu().numpy().astype(np.float64)
        want = c_oracle.start_fft_batch(xs)
        for i, w in enumerate(tied):
            assert prominence_dicts(after[w], 125.0, n) == c_oracle.peaks_prominence(want[i], 125.0), w


# ---------------------------------------------------------------------------------------------------------------
# 6. behaviour
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_permuted_batch_gives_permuted_records(an):
    n, b = 2048, 400
    x, _ = tie_windows(b, n, seed=123)
    perm = np.random.default_rng(4).permutation(b)
    out = []
    for xx in (x, x[perm]):
        _, ptr = rows_on_device(xx)
        rec, _ = fp32_records(an, "split", ptr, n, n, b, n, True, 4, 5)
        resolve_dev(an, ptr, n, n, b, n, True, 4, 5, rec)
        out.append(rec.bytes().reshape(b, -1))
    assert np.array_equal(out[0][perm], out[1])


@pytest.mark.gpu
def test_launch_count_fixed(an):
    n, b = 1024, 256
    counts = []
    for seed, tie_rich in ((1, True), (2, False)):
        x, _ = tie_windows(b, n, seed=seed)
        if not tie_rich:
            x = np.random.default_rng(seed).standard_normal((b, n)).astype(np.float32)
        _, ptr = rows_on_device(x)
        rec, _ = fp32_records(an, "analyze", ptr, n, n, b, n, True, 4, 5)
        ties = int((rec.bytes().view(rec_dtype(5))["status"] == TIE).sum())
        c0 = an.launch_count()
        resolve_dev(an, ptr, n, n, b, n, True, 4, 5, rec)
        counts.append((an.launch_count() - c0, ties))
    assert counts[0][1] > 0 and counts[1][1] == 0
    assert counts[0][0] == counts[1][0] == 2


@pytest.mark.gpu
def test_dev_does_not_wait_for_the_stream(an):
    import time
    import torch
    n, b = 1024, 64
    x, _ = tie_windows(b, n, seed=9)
    _, ptr = rows_on_device(x)
    rec, _ = fp32_records(an, "analyze", ptr, n, n, b, n, True, 4, 5)
    resolve_dev(an, ptr, n, n, b, n, True, 4, 5, rec)     # workspace and list grown outside the timed call
    torch.cuda.synchronize()
    done = torch.cuda.Event()
    torch.cuda._sleep(2_000_000_000)                     # about a second of GPU time queued on the stream
    t0 = time.perf_counter()
    resolve_dev(an, ptr, n, n, b, n, True, 4, 5, rec)
    dt = time.perf_counter() - t0
    done.record()
    assert not done.query() and dt < 0.2, dt
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_errors_and_empty_batch(an):
    import torch
    n, b = 1024, 4
    d_x = torch.zeros((b, n), dtype=torch.float32, device="cuda:0")
    rec = Guarded(b * 128)
    x, r = d_x.data_ptr(), rec.ptr
    call = lambda *a: an.ctx.call("apda_resolve_fp32_ties_dev", *a)  # noqa: E731
    ok = [_p(x), _p(0), n, n, b, n, CENTER_MEDIAN, 1, 125.0, _p(0), 4, 5, _p(r)]

    def bad(i, v, exc=ValueError):
        a = list(ok)
        a[i] = v
        with pytest.raises(exc):
            call(*a)
    from apda_fft_b200._cabi import ApdaError
    bad(0, _p(0))                                       # samples NULL
    bad(12, _p(0))                                      # records NULL
    big = torch.zeros(16384, dtype=torch.float32, device="cuda:0")
    a = list(ok)
    a[0], a[2], a[3], a[4], a[5] = _p(big.data_ptr()), 16384, 16384, 1, 16384
    with pytest.raises(ApdaError) as e:                 # N > 8192 on _dev
        call(*a)
    assert e.value.code == -5
    a = list(ok)
    a[2], a[6] = n - 1, CENTER_MEAN                     # CENTER_MEAN with padding
    with pytest.raises(ValueError):
        call(*a)
    bad(10, 0)                                          # k < 1
    bad(11, 3)                                          # rec_cap < k
    bad(11, 10_000)                                     # rec_cap beyond APDA_MAX_PEAKS
    bad(6, 7)                                           # unknown flags
    a = list(ok)
    a[4] = 0
    c0 = an.launch_count()
    call(*a)                                            # batch 0: nothing happens
    assert an.launch_count() == c0
    assert (rec.bytes() == SENT).all()
    h = np.zeros(b, dtype=rec_dtype(5))
    with pytest.raises(ValueError):
        an.ctx.call("apda_resolve_fp32_ties_host", _p(0), _p(0), n, n, b, n, CENTER_MEDIAN, 1, 125.0, _p(0), 4, 5,
                    _p(h.ctypes.data))
