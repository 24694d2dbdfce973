"""The C ABI beyond the benchmark's inputs (include/apda_b200.h, DESIGN.md section 3), on every kernel route:

  1. rows at a pitch ``ld > n_samples`` and from a misaligned base (the FFT kernels' predicated variants, K2's masked
     128-bit median loads, the host pipeline's pitched copy), with NaN in the gaps and after the last row;
  2. ``APDA_CENTER_NONE`` (and ``APDA_CENTER_MEAN``) against the oracle's uncentred transform;
  3. per-window sampling rates that change the peak list (flexible: the hump exclusion through round(j*fs/n, 4);
     rigid: the zeroing radius round(0.02*f/df)), drawn pseudo-randomly per window;
  4. every k and record width, with sentinel-filled record buffers: every byte of every record is written, the slots
     after ``count`` hold idx -1 and zeros, and nothing past the last record is touched.

fp64 results are held bit for bit to the C oracle; fp32 spectra to the oracle run on the fp32-quantised samples within
the bounds the rest of the suite uses (K1: 3e-6*scale + n_samples*max|x|*1.2e-7, K2: 2e-5*scale), fp32 records by their
index lists.  A strided or misaligned call must give exactly the bytes of the same call on contiguous rows.
"""
import contextlib
import ctypes
import struct

import numpy as np
import pytest

from oracle import c_oracle

_p = ctypes.c_void_p
SENT = 0xA5          # byte every output buffer starts as
GUARD = 4096         # sentinel bytes on both sides of every device output buffer
CENTER_MEDIAN, CENTER_MEAN, CENTER_NONE = 0, 1, 2
EMPTY_SLOT = np.frombuffer(struct.pack("<iidd", -1, 0, 0.0, 0.0), dtype=np.uint8)


def max_peaks(n):
    return n // 8 + 8


def rec_dtype(cap):
    peak = np.dtype([("idx", "<i4"), ("width_bins", "<i4"), ("mag", "<f8"), ("prominence", "<f8")])
    return np.dtype([("count", "<i4"), ("status", "<i4"), ("pk", peak, (cap,))])


def _sfx(dt):
    return "f32" if np.dtype(dt) == np.float32 else "f64"


def _cdt(dt):
    return np.complex64 if np.dtype(dt) == np.float32 else np.complex128


# ---------------------------------------------------------------------------------------------------------------
# fixtures and device helpers
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
    """Device output buffer of `nbytes`, every byte SENT, with GUARD sentinel bytes before and after it."""

    def __init__(self, nbytes):
        import torch
        self.n = int(nbytes)
        self.buf = torch.full((2 * GUARD + self.n,), SENT, dtype=torch.uint8, device="cuda:0")
        self.ptr = self.buf.data_ptr() + GUARD

    def bytes(self):
        import torch
        torch.cuda.synchronize()
        h = self.buf.cpu().numpy()
        assert (h[:GUARD] == SENT).all(), "bytes before the output buffer were written"
        assert (h[GUARD + self.n:] == SENT).all(), "bytes after the output buffer were written"
        return h[GUARD:GUARD + self.n].copy()


def rows_on_device(x, ld, off):
    """x[b, ns] placed at row pitch `ld` from element `off` of a NaN-filled device buffer (NaN in the gaps between rows
    and in a tail after the last one).  Returns (buffer, address of row 0)."""
    import torch
    b, ns = x.shape
    t = torch.from_numpy(np.ascontiguousarray(x))
    buf = torch.full((off + b * ld + 67,), float("nan"), dtype=t.dtype, device="cuda:0")
    buf[off:off + b * ld].view(b, ld)[:, :ns] = t.to("cuda:0")
    return buf, buf.data_ptr() + off * buf.element_size()


def to_dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def fft_dev(an, ptr, ns, ld, b, n, dt, flags=CENTER_MEDIAN):
    out = Guarded(b * n * 2 * np.dtype(dt).itemsize)
    an.ctx.call(f"apda_fft_{_sfx(dt)}_dev", _p(ptr), ns, ld, b, n, flags, _p(out.ptr))
    return out.bytes().view(_cdt(dt)).reshape(b, n)


def fft_ragged_dev(an, ptr, d_nv, n_max, ld, b, n, dt, flags=CENTER_MEDIAN):
    out = Guarded(b * n * 2 * np.dtype(dt).itemsize)
    an.ctx.call(f"apda_fft_ragged_{_sfx(dt)}_dev", _p(ptr), _p(d_nv.data_ptr()), n_max, ld, b, n, flags, _p(out.ptr))
    return out.bytes().view(_cdt(dt)).reshape(b, n)


def analyze_dev(an, ptr, ns, ld, b, n, dt, flexible, fs=125.0, d_fs=None, k=None, cap=5, ws=False, flags=CENTER_MEDIAN):
    """apda_analyze_*_dev -> (records bytes [b, rec], full spectra from the caller's workspace or None)."""
    k = (4 if flexible else 5) if k is None else k
    rec = Guarded(b * rec_dtype(cap).itemsize)
    spec = Guarded(b * n * 2 * np.dtype(dt).itemsize) if ws else None
    an.ctx.call(f"apda_analyze_{_sfx(dt)}_dev", _p(ptr), ns, ld, b, n, flags, int(flexible), fs,
                _p(0 if d_fs is None else d_fs.data_ptr()), k, cap, _p(spec.ptr if ws else 0), _p(rec.ptr))
    r = rec.bytes().reshape(b, -1)
    return r, (spec.bytes().view(_cdt(dt)).reshape(b, n) if ws else None)


def analyze_ragged_dev(an, ptr, d_nv, n_max, ld, b, n, dt, flexible, fs=125.0, d_fs=None, k=None, cap=5, ws=False):
    k = (4 if flexible else 5) if k is None else k
    rec = Guarded(b * rec_dtype(cap).itemsize)
    spec = Guarded(b * n * 2 * np.dtype(dt).itemsize) if ws else None
    an.ctx.call(f"apda_analyze_ragged_{_sfx(dt)}_dev", _p(ptr), _p(d_nv.data_ptr()), n_max, ld, b, n, CENTER_MEDIAN,
                int(flexible), fs, _p(0 if d_fs is None else d_fs.data_ptr()), k, cap, _p(spec.ptr if ws else 0),
                _p(rec.ptr))
    r = rec.bytes().reshape(b, -1)
    return r, (spec.bytes().view(_cdt(dt)).reshape(b, n) if ws else None)


def fused_dev(an, ptr, ns, ld, b, n, flexible, fs=125.0, d_fs=None, k=None, flags=CENTER_MEDIAN):
    k = (4 if flexible else 5) if k is None else k
    rec = Guarded(b * 128)
    an.ctx.call("apda_analyze_fused_f32_dev", _p(ptr), ns, ld, b, n, flags, int(flexible), fs,
                _p(0 if d_fs is None else d_fs.data_ptr()), k, 5, _p(rec.ptr))
    return rec.bytes().reshape(b, 128)


def peaks_dev(an, z, flexible, fs=125.0, fs_w=None, k=None, cap=5):
    """Device picker on complex spectra z[b, n] (complex64 -> fp32 kernels)."""
    b, n = z.shape
    dt = np.float32 if z.dtype == np.complex64 else np.float64
    k = (4 if flexible else 5) if k is None else k
    d_z = to_dev(z.view(dt))
    d_fs = None if fs_w is None else to_dev(np.asarray(fs_w, dtype=np.float64))
    rec = Guarded(b * rec_dtype(cap).itemsize)
    kind = "prominence" if flexible else "resolution"
    an.ctx.call(f"apda_peaks_{kind}_{_sfx(dt)}_dev", _p(d_z.data_ptr()), n, b, fs,
                _p(0 if d_fs is None else d_fs.data_ptr()), k, cap, _p(rec.ptr))
    return rec.bytes().reshape(b, -1)


# ---------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------
def k1_bound(want, x32):
    """fp32 K1 / general-kernel bound of the suite (test_quantised_windows_exact_median)."""
    scale = max(float(np.abs(want).max()), 1e-3)
    return 3e-6 * scale + x32.shape[-1] * float(np.abs(x32).max()) * 1.2e-7


def k2_bound(want):
    return 2e-5 * float(np.abs(want).max())


def fp32_bound(n, want, x32):
    return k2_bound(want) if n > 8192 else k1_bound(want, x32)


def uncentred_oracle(row, n):
    """start_fft without the median: the reference fft of the zero-padded row, bin 0 := 0."""
    z = np.zeros(n, dtype=np.complex128)
    z[:row.shape[0]] = np.asarray(row, dtype=np.float64)
    out = c_oracle.fft_c2c(z)
    out[0] = 0
    return out


def median_in(x, dt):
    """statistics.median of each row, computed in the compute dtype: the middle value, or (a + b) / 2 of the two
    middle values (for fp32: the fp32 sum halved, as the kernels form it)."""
    s = np.sort(np.asarray(x, dtype=dt), axis=1)
    n = s.shape[1]
    if n % 2:
        return s[:, n // 2]
    return ((s[:, n // 2 - 1] + s[:, n // 2]) * dt(0.5)).astype(dt)


_ORACLE = {}


def oracle_list(key, spec_row, fs, flexible, k):
    """Reference peak list (list of dicts) of one spectrum row at `fs`, cached per (key, fs, picker).  The reference
    stops at k accepted peaks, so the list for any k is a prefix of the list for the largest k."""
    n = spec_row.shape[0]
    ck = (key, float(fs), bool(flexible))
    if ck not in _ORACLE:
        row = np.asarray(spec_row, dtype=np.complex128)
        pick = c_oracle.peaks_prominence if flexible else c_oracle.peaks_resolution
        _ORACLE[ck] = pick(row, float(fs), max_peaks(n))
    return _ORACLE[ck][:k]


def _dicts(rec, fs, n, flexible):
    from apda_fft_b200.records import prominence_dicts, resolution_dicts
    return prominence_dicts(rec, fs, n) if flexible else resolution_dicts(rec, fs, n)


def check_records(raw, cap, k, n, flexible, fs_w, want, exact, status=(0, 16)):
    """raw: uint8[b, 8 + 24*cap] records that started as SENT bytes.  Every byte must have been written: count <= k,
    a known status, the peaks of `want(w)` (the reference list of window w: dicts equal in fp64, indices in fp32) and
    idx -1 / width 0 / mag 0 / prominence 0 in every slot after count."""
    b = raw.shape[0]
    recs = raw.view(rec_dtype(cap)).reshape(b)
    slots = raw[:, 8:].reshape(b, cap, 24)
    for w in range(b):
        cnt, st = int(recs["count"][w]), int(recs["status"][w])
        assert 0 <= cnt <= k and st in status, (w, cnt, st)
        assert (slots[w, cnt:] == EMPTY_SLOT).all(), (w, cnt, slots[w, cnt:cnt + 2])
        fs = float(fs_w[w])
        ref = want(w)
        got = _dicts(recs[w], fs, n, flexible)
        if exact:
            assert got == ref, (w, fs, got, ref)
        else:
            assert [p["idx"] for p in got] == [p["idx"] for p in ref], (w, fs, got, ref)
    return recs


# ---------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------
def skewed_windows(b, ns, seed, dc=0.77):
    """Tones + skewed (exponential) noise + a DC offset: median, mean and 0 are three different centres."""
    rng = np.random.default_rng(seed)
    i = np.arange(ns, dtype=np.float64)
    x = np.empty((b, ns))
    for w in range(b):
        x[w] = (0.5 * np.sin(2 * np.pi * (31.3 + 0.71 * w) * i / ns) + 0.2 * np.sin(2 * np.pi * 201.0 * i / ns + 0.1 * w)
                + 0.3 * rng.exponential(1.0, ns) + dc + 0.01 * w)
    return np.round(x, 6)


def designed_mags(n, flexible, big=1.0, spikes=0, seed=0):
    """Half spectrum (n // 2 magnitudes, all exact in fp32) whose reference peak list depends on fs.
    flexible: a peak at p0, a shelf up to a 5 % bump at p1 = 1.05 * p0 (prominence / magnitude < 0.10, so a hump of p0
    exactly when round(p1*df, 4) lies within 5 % of round(p0*df, 4)), and a peak at p2.
    rigid: spikes at 125 (10), 128 (8), 122 (7.5) and p3 (5); the zeroing radius round(0.02 * 125 +- ulp) is 2 or 3
    depending on fs, which keeps or removes 122 and 128.
    spikes: that many isolated spikes of 10 .. 10.5 (times 1) on even bins away from the designed peaks (big scales
    the designed part above them), so that the fast pickers hand the window to the general kernel."""
    half = n // 2
    rng = np.random.default_rng(seed)
    m = rng.uniform(0.01, 0.02, half)
    j = np.arange(half, dtype=np.float64)
    if flexible:
        if half >= 1024:
            p0, p1, p2, s = 200, 210, 600, 7
            m = np.maximum(m, 10.0 * np.exp(-((j - p0) / 3.0) ** 2))
            m[p1 - s:p1] = np.linspace(3.93, 3.99, s)
            m[p1 + 1:p1 + 1 + s] = np.linspace(3.99, 3.93, s)
            m[p1] = 4.3
            m[p2], m[p2 - 1], m[p2 + 1] = 6.0, 3.0, 3.0
        else:
            p0, p1, p2, s = 100, 105, 180, 2
            m[100:108] = [5.0, 4.6, 4.3, 3.98, 3.99, 4.4, 3.99, 3.98]
            m[p2], m[p2 - 1], m[p2 + 1] = 3.0, 1.5, 1.5
        keep = [(p0 - 20, p1 + s + 20), (p2 - 5, p2 + 5)]
    else:
        p3 = 700 if half > 720 else half * 3 // 4
        m[125], m[128], m[122], m[p3] = 10.0, 8.0, 7.5, 5.0
        keep = [(110, 140), (p3 - 10, p3 + 10)]
    m = (m * big).astype(np.float32).astype(np.float64)
    if spikes:
        ok = np.ones(half // 2, dtype=bool)
        ok[0] = False
        for lo, hi in keep:
            ok[max(0, lo // 2):hi // 2 + 1] = False
        at = 2 * rng.permutation(np.flatnonzero(ok))[:spikes]
        m[at] = (10.0 + 0.5 * rng.random(spikes)).astype(np.float32)
    m[0] = 0.0
    return m


def designed_spectra(b, n, flexible, dt, **kw):
    """b copies of the designed picker-only spectrum (magnitude in the real part, imaginary part 0)."""
    z = np.zeros((b, n), dtype=_cdt(dt))
    z[:, :n // 2] = designed_mags(n, flexible, **kw)
    return z


def designed_samples(n, flexible):
    """Time-domain window whose start_fft is the designed spectrum: the inverse DFT of its Hermitian extension."""
    m = designed_mags(n, flexible)
    z = np.zeros(n, dtype=np.complex128)
    z[1:n // 2] = m[1:]
    z[n // 2 + 1:] = m[1:][::-1]
    return np.fft.ifft(z).real + 0.25


_FS_CAND = np.round(np.random.default_rng(2024).uniform(50.0, 1000.0, 400), 3)


def fs_classes(key, spec_row, flexible, k, per_class=4):
    """Sampling rates of _FS_CAND grouped by the reference's peak list on spec_row: {index tuple: [fs, ...]}, scanned
    until two outcomes have `per_class` rates each."""
    out = {}
    for fs in _FS_CAND:
        out.setdefault(tuple(p["idx"] for p in oracle_list(key, spec_row, fs, flexible, k)), []).append(float(fs))
        full = [v for v in out.values() if len(v) >= per_class]
        if len(full) >= 2:
            break
    return {o: v[:per_class] for o, v in out.items() if len(v) >= 2}


def fs_per_window(classes, b, seed):
    """A pseudo-random (not periodic) rate per window: each window picks an outcome, then one of its rates."""
    rng = np.random.default_rng(seed)
    groups = list(classes.values())
    return np.array([groups[g][rng.integers(len(groups[g]))] for g in rng.integers(len(groups), size=b)])


# ---------------------------------------------------------------------------------------------------------------
# without a GPU: the fs-dependent inputs really are fs-dependent
# ---------------------------------------------------------------------------------------------------------------
def test_designed_inputs_are_fs_sensitive():
    """Both outcomes occur among the chosen rates for every designed input the GPU tests use, so a kernel that read
    another window's fs would get another peak list for about half of the windows."""
    for n in (512, 1024, 4096, 8192, 1 << 16):
        for flexible in (True, False):
            k = 4 if flexible else 5
            variants = [{}]
            if n == 8192:
                variants.append({"big": 4.0, "spikes": 200 if flexible else 680})
            for kw in variants:
                z = designed_spectra(1, n, flexible, np.float64, **kw)[0]
                cls = fs_classes(("cpu-design", n, tuple(kw.items())), z, flexible, k)
                assert len(cls) >= 2 and all(len(v) >= 2 for v in cls.values()), (n, flexible, kw, cls)
    for n in (4096, 16384):
        for flexible in (True, False):
            x = designed_samples(n, flexible)
            for dt in (np.float64, np.float32):
                spec = c_oracle.start_fft_batch(x.astype(dt).astype(np.float64)[None, :])[0]
                cls = fs_classes(("cpu-samples", n, dt), spec, flexible, 4 if flexible else 5)
                assert len(cls) >= 2, (n, flexible, dt, cls)


# ---------------------------------------------------------------------------------------------------------------
# 1. strided and misaligned rows
# ---------------------------------------------------------------------------------------------------------------
# (name, N, generic_only, batch): K1 fast kernels, the shared-memory general kernel (N <= 512, and 1024..8192 under
# generic_only), K2 (N >= 16384; 301 windows at 2^14 cross the median's 256-window launch sets)
FFT_ROUTES = [("k1", 1024, False, 37), ("k1", 4096, False, 37), ("k1", 8192, False, 5), ("smem", 512, False, 37),
              ("smem_generic", 4096, True, 37), ("k2", 16384, False, 301)]


def _layouts(ns):
    return [(ns, 0), (ns + 1, 0), (ns + 3, 1), (ns + 64, 3)]


def _lengths(n):
    return (n, n - 3, 3 * n // 4 + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("route,n,gen,b", FFT_ROUTES, ids=[f"{r[0]}-{r[1]}" for r in FFT_ROUTES])
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_strided_misaligned_rows(route, n, gen, b, dt, an):
    """apda_fft / apda_analyze (own workspace = half-spectrum K1, and a caller workspace) / the fused kernel on rows at
    pitch ld from a misaligned base: no NaN from the gaps, nothing written around the outputs, fp64 spectra bit-equal
    to the oracle, and every strided result bit-equal to the contiguous one (the FULL and predicated variants compute
    the same exact median and the same butterflies)."""
    lengths = _lengths(n) if b < 100 else (n - 3,)
    with generic(an, gen):
        for ns in lengths:
            x = skewed_windows(b, ns, seed=ns).astype(dt)
            base = None
            for ld, off in _layouts(ns):
                buf, ptr = rows_on_device(x, ld, off)
                res = {"spec": fft_dev(an, ptr, ns, ld, b, n, dt)}
                for flexible in (True, False):
                    res[("own", flexible)] = analyze_dev(an, ptr, ns, ld, b, n, dt, flexible)[0]
                    res[("ws", flexible)], res[("wsspec", flexible)] = analyze_dev(an, ptr, ns, ld, b, n, dt, flexible, ws=True)
                    if dt == np.float32 and 1024 <= n <= 8192 and not gen:
                        res[("fused", flexible)] = fused_dev(an, ptr, ns, ld, b, n, flexible)
                del buf
                assert np.isfinite(res["spec"].view(dt)).all(), (ld, off)
                for key, v in res.items():
                    if key[0] in ("own", "ws", "fused"):
                        recs = v.view(rec_dtype(5)).reshape(b)
                        assert np.isfinite(recs["pk"]["mag"]).all() and np.isfinite(recs["pk"]["prominence"]).all()
                        assert (recs["count"] >= 1).all() and ((recs["status"] & ~16) == 0).all(), (key, ld, off)
                if base is None:
                    base = res
                    want = c_oracle.start_fft_batch(x.astype(np.float64), n_fft=n)
                    if dt == np.float64:
                        assert np.array_equal(res["spec"].view(np.float64), want.view(np.float64)), (ns, "fp64 vs oracle")
                    else:
                        for w in range(b):
                            err = np.abs(res["spec"][w].astype(np.complex128) - want[w]).max()
                            assert err <= fp32_bound(n, want[w], x[w]), (ns, w, err)
                    for flexible in (True, False):
                        assert np.array_equal(res[("wsspec", flexible)], res["spec"]), (ns, flexible)
                    continue
                for key in base:
                    assert np.array_equal(np.asarray(base[key]).view(np.uint8), np.asarray(res[key]).view(np.uint8)), \
                        (route, ns, ld, off, key)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [512, 4096])
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_strided_misaligned_rows_ragged(n, dt, an):
    """apda_fft_ragged / apda_analyze_ragged at pitch ld from a misaligned base: windows of the common length on the
    fast kernels (N = 4096) or the general kernel (N = 512), shorter ones through the general kernel's list; fp64
    spectra bit-equal to the oracle at each window's own sample count, everything bit-equal to the contiguous call."""
    import torch
    b = 41
    rng = np.random.default_rng(n + 1)
    nv = np.where(rng.random(b) < 0.6, n, rng.integers(1, n, size=b)).astype(np.int32)
    nv[[3, 17]] = (n - 3, 3 * n // 4 + 1)
    d_nv = torch.from_numpy(nv).to("cuda:0")
    x = skewed_windows(b, n, seed=n + 2).astype(dt)
    for w in range(b):
        x[w, nv[w]:] = np.nan                       # samples past n_valid must never be read
    base = None
    for ld, off in _layouts(n):
        buf, ptr = rows_on_device(x, ld, off)
        res = {"spec": fft_ragged_dev(an, ptr, d_nv, n, ld, b, n, dt)}
        for flexible in (True, False):
            res[flexible] = analyze_ragged_dev(an, ptr, d_nv, n, ld, b, n, dt, flexible)[0]
        del buf
        assert np.isfinite(res["spec"].view(dt)).all(), (ld, off)
        if base is None:
            base = res
            for w in range(b):
                want = c_oracle.start_fft_batch(x[w:w + 1, :nv[w]].astype(np.float64), n_fft=n)[0]
                if dt == np.float64:
                    assert np.array_equal(res["spec"][w].view(np.float64), want.view(np.float64)), (w, nv[w])
                else:
                    err = np.abs(res["spec"][w].astype(np.complex128) - want).max()
                    assert err <= k1_bound(want, x[w, :nv[w]]), (w, nv[w], err)
            for flexible in (True, False):
                recs = res[flexible].view(rec_dtype(5)).reshape(b)
                other = np.array([c_oracle.padded_len(int(v)) != n for v in nv])
                assert ((recs["status"] & 4 != 0) == other).all() and ((recs["status"] & ~(4 | 16)) == 0).all()
            continue
        for key in base:
            assert np.array_equal(base[key].view(np.uint8), res[key].view(np.uint8)), (n, ld, off, key)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_host_entry_points_pitched_rows(dt, an):
    """The _host entry points with ld > n_samples (pitched copy) over more than two pipeline chunks, NaN in the host
    gaps and per-window rates: results bit-equal to the contiguous call."""
    n, ns = 1024, 1021
    ld = ns + 5
    chunk = (96 << 20) // (n * 2 * np.dtype(dt).itemsize)
    b = 2 * chunk + 77
    sfx = _sfx(dt)
    rng = np.random.default_rng(3)
    one = skewed_windows(61, ns, seed=4).astype(dt)
    x = one[rng.integers(61, size=b)] + (rng.integers(-8, 8, size=(b, 1)) * 0.125).astype(dt)
    pitched = np.full((b, ld), np.nan, dtype=dt)
    pitched[:, :ns] = x
    x = np.ascontiguousarray(x)
    fs_w = np.round(rng.uniform(50.0, 1000.0, b), 3)

    def fft(src, stride):
        out = np.empty((b, n), dtype=_cdt(dt))
        an.ctx.call(f"apda_fft_{sfx}_host", _p(src.ctypes.data), ns, stride, b, n, CENTER_MEDIAN, _p(out.ctypes.data))
        return out

    def analyze(src, stride, flexible, name):
        recs = np.zeros(b, dtype=rec_dtype(5))
        an.ctx.call(name, _p(src.ctypes.data), ns, stride, b, n, CENTER_MEDIAN, int(flexible), 125.0,
                    _p(fs_w.ctypes.data), 4 if flexible else 5, 5, _p(recs.ctypes.data))
        return recs

    a, c = fft(pitched, ld), fft(x, ns)
    assert np.isfinite(a.view(dt)).all() and np.array_equal(a.view(dt), c.view(dt))
    names = [f"apda_analyze_{sfx}_host"] + (["apda_analyze_fused_f32_host"] if dt == np.float32 else [])
    for name in names:
        for flexible in (True, False):
            ra, rc = analyze(pitched, ld, flexible, name), analyze(x, ns, flexible, name)
            assert ra.tobytes() == rc.tobytes(), (name, flexible)
            assert np.isfinite(ra["pk"]["mag"]).all() and (ra["count"] >= 1).all()
    # the fused kernel's chunks are sized by samples, not spectra: make its pipeline run more than two chunks too
    if dt == np.float32:
        fchunk = (96 << 20) // (ns * 4)
        bf = 2 * fchunk + 33
        xf = np.ascontiguousarray(one[rng.integers(61, size=bf)])
        pf = np.full((bf, ld), np.nan, dtype=dt)
        pf[:, :ns] = xf
        fsf = np.round(rng.uniform(50.0, 1000.0, bf), 3)
        out = []
        for src, stride in ((pf, ld), (xf, ns)):
            recs = np.zeros(bf, dtype=rec_dtype(5))
            an.ctx.call("apda_analyze_fused_f32_host", _p(src.ctypes.data), ns, stride, bf, n, CENTER_MEDIAN, 1, 125.0,
                        _p(fsf.ctypes.data), 4, 5, _p(recs.ctypes.data))
            out.append(recs)
        assert out[0].tobytes() == out[1].tobytes()


# ---------------------------------------------------------------------------------------------------------------
# 2. APDA_CENTER_NONE / APDA_CENTER_MEAN
# ---------------------------------------------------------------------------------------------------------------
CENTER_ROUTES = [("k1", 1024, False, 9), ("k1", 4096, False, 9), ("smem", 512, False, 9),
                 ("smem_generic", 4096, True, 9), ("k2", 16384, False, 5)]


def _run_fft(an, route, x, n, dt, flags, nv=None):
    b, ns = x.shape
    if route == "ragged":
        import torch
        buf, ptr = rows_on_device(x, ns, 0)
        return fft_ragged_dev(an, ptr, torch.from_numpy(nv).to("cuda:0"), ns, ns, b, n, dt, flags)
    buf, ptr = rows_on_device(x, ns, 0)
    return fft_dev(an, ptr, ns, ns, b, n, dt, flags)


@pytest.mark.gpu
@pytest.mark.parametrize("route,n,gen,b", CENTER_ROUTES + [("ragged", 4096, False, 9), ("ragged", 512, False, 9)],
                         ids=[f"{r[0]}-{r[1]}" for r in CENTER_ROUTES] + ["ragged-4096", "ragged-512"])
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_center_none(route, n, gen, b, dt, an):
    """CENTER_NONE transforms the samples as given: the reference fft of the zero-padded row with bin 0 := 0 (bit for
    bit in fp64, within the K1 / K2 bound in fp32).  Padded windows then differ from CENTER_MEDIAN (at full length
    centring only moves the zeroed bin 0).  Pre-centred windows y = x - median(x) (computed in the compute dtype) give
    exactly CENTER_MEDIAN(x): every route centres with one subtraction of the exact median, fp32 included."""
    with generic(an, gen):
        for ns in _lengths(n):
            x = skewed_windows(b, ns, seed=ns + 11, dc=37.5).astype(dt)
            nv = None
            if route == "ragged":
                nv = np.full(b, ns, dtype=np.int32)
                nv[1], nv[4] = ns - 5, ns // 2 + 1
            got = _run_fft(an, route, x, n, dt, CENTER_NONE, nv)
            med = _run_fft(an, route, x, n, dt, CENTER_MEDIAN, nv)
            for w in range(b):
                cnt = ns if nv is None else int(nv[w])
                want = uncentred_oracle(x[w, :cnt], n)
                if dt == np.float64:
                    assert np.array_equal(got[w].view(np.float64), want.view(np.float64)), (ns, w)
                else:
                    err = np.abs(got[w].astype(np.complex128) - want).max()
                    assert err <= fp32_bound(n, want, x[w, :cnt]), (ns, w, err)
                if cnt < n:
                    assert not np.array_equal(got[w], med[w]), (ns, w, "CENTER_NONE centred a padded window")
            y = np.empty_like(x)
            for w in range(b):
                cnt = ns if nv is None else int(nv[w])
                y[w, :cnt] = x[w, :cnt] - median_in(x[w:w + 1, :cnt], dt)[0]
                y[w, cnt:] = x[w, cnt:]
            pre = _run_fft(an, route, y, n, dt, CENTER_NONE, nv)
            assert np.array_equal(pre.view(dt), med.view(dt)), (route, ns, "pre-centred CENTER_NONE != CENTER_MEDIAN")


@pytest.mark.gpu
@pytest.mark.parametrize("route,n,gen,b", CENTER_ROUTES, ids=[f"{r[0]}-{r[1]}" for r in CENTER_ROUTES])
def test_center_mean(route, n, gen, b, an):
    """CENTER_MEAN (fp32, full-length windows only) leaves bins >= 1 as the median-centred reference has them (within
    the K1 / K2 bound) and bin 0 exactly 0; fp64 and padded windows reject it, the fused kernel rejects CENTER_NONE."""
    x = skewed_windows(b, n, seed=n + 5, dc=3.0).astype(np.float32)
    with generic(an, gen):
        got = _run_fft(an, route, x, n, np.float32, CENTER_MEAN)
        want = c_oracle.start_fft_batch(x.astype(np.float64), n_fft=n)
        assert (got[:, 0] == 0).all()
        for w in range(b):
            err = np.abs(got[w, 1:].astype(np.complex128) - want[w, 1:]).max()
            assert err <= fp32_bound(n, want[w], x[w]), (w, err)
        with pytest.raises(ValueError):
            _run_fft(an, route, x.astype(np.float64), n, np.float64, CENTER_MEAN)
        with pytest.raises(ValueError):
            _run_fft(an, route, np.ascontiguousarray(x[:, :n - 3]), n, np.float32, CENTER_MEAN)
    if n <= 8192 and route == "k1":
        buf, ptr = rows_on_device(x, n, 0)
        from apda_fft_b200 import _cabi
        with pytest.raises(_cabi.ApdaError) as err:
            fused_dev(an, ptr, n, n, b, n, True, flags=CENTER_NONE)
        assert err.value.code == _cabi.ERR_UNSUPPORTED


# ---------------------------------------------------------------------------------------------------------------
# 3. per-window sampling rates that change the peak list
# ---------------------------------------------------------------------------------------------------------------
# (name, n, generic_only, batch, design keywords): fast pickers, their repair list (hot maxima beyond what they keep
# on chip), the general kernel in shared memory (n = 512; 4096 under generic_only; fp32 32768) and in the global
# workspace (fp64 32768; 2^16 under generic_only), the large form (2^16, more than one 64-window launch set)
PICK_ROUTES = [("fast", 1024, False, 37, {}), ("fast", 4096, False, 37, {}), ("fast", 8192, False, 37, {}),
               ("repair", 8192, False, 37, "spikes"), ("general", 512, False, 37, {}),
               ("general_generic", 4096, True, 37, {}), ("general_32k", 32768, False, 9, {}),
               ("general_global_generic", 1 << 16, True, 5, {}), ("large", 1 << 16, False, 131, {})]


def _design_kw(kw, flexible):
    if kw == "spikes":
        return {"big": 4.0, "spikes": 200 if flexible else 680}
    return kw


@pytest.mark.gpu
@pytest.mark.parametrize("route,n,gen,b,kw", PICK_ROUTES, ids=[f"{r[0]}-{r[1]}" for r in PICK_ROUTES])
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_per_window_fs_pickers_dev(route, n, gen, b, kw, dt, an):
    """apda_peaks_*_dev with d_fs: every window at its own (pseudo-random) rate gets the reference's list at that
    rate; both outcomes occur in the batch."""
    for flexible in (True, False):
        k = 4 if flexible else 5
        dkw = _design_kw(kw, flexible)
        z = designed_spectra(b, n, flexible, dt, **dkw)
        key = ("design", n, tuple(dkw.items()))
        cls = fs_classes(key, z[0], flexible, k)
        fs_w = fs_per_window(cls, b, seed=n + b)
        with generic(an, gen):
            raw = peaks_dev(an, z, flexible, fs=fs_w[0] + 1.0, fs_w=fs_w, k=k)
        recs = check_records(raw, 5, k, n, flexible, fs_w, lambda w: oracle_list(key, z[0], fs_w[w], flexible, k),
                             exact=dt == np.float64)
        outcomes = {tuple(r["pk"]["idx"][:r["count"]]) for r in recs}
        assert len(outcomes) >= 2, (route, flexible, outcomes)
        if route == "repair":       # the designed peaks still lead the list of a window handed to the general kernel
            assert (recs["pk"]["idx"][:, 0] == (200 if flexible else 125)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_per_window_fs_pickers_host(dt, an):
    """apda_peaks_*_host with h_fs over more than two pipeline chunks: the per-chunk copy of the rates."""
    n = 1024
    chunk = (96 << 20) // (n * 2 * np.dtype(dt).itemsize)
    b = 2 * chunk + 101
    sfx = _sfx(dt)
    for flexible in (True, False):
        k = 4 if flexible else 5
        z = designed_spectra(b, n, flexible, dt)
        key = ("design", n, ())
        fs_w = fs_per_window(fs_classes(key, z[0], flexible, k), b, seed=b)
        recs = np.full(b, 0, dtype=rec_dtype(5))
        recs.view(np.uint8)[:] = SENT
        kind = "prominence" if flexible else "resolution"
        an.ctx.call(f"apda_peaks_{kind}_{sfx}_host", _p(z.ctypes.data), n, b, 125.0, _p(fs_w.ctypes.data), k, 5,
                    _p(recs.ctypes.data))
        raw = recs.view(np.uint8).reshape(b, 128)
        # windows of one rate share one reference list: check one per rate in full, all of them by their bytes
        for fs in np.unique(fs_w):
            sel = np.flatnonzero(fs_w == fs)
            check_records(raw[sel[:1]], 5, k, n, flexible, fs_w[sel[:1]],
                          lambda w: oracle_list(key, z[0], fs, flexible, k), exact=dt == np.float64)
            assert (raw[sel] == raw[sel[0]]).all(), (flexible, fs)
        assert len({raw[i].tobytes() for i in range(0, b, 97)}) >= 2


@pytest.mark.gpu
@pytest.mark.parametrize("n,gen", [(4096, False), (4096, True), (16384, False)], ids=["k1-4096", "generic-4096", "k2-16384"])
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_per_window_fs_analyze_and_fused(n, gen, dt, an):
    """apda_analyze_*_dev (and the fused kernel) with d_fs on time-domain windows whose spectrum is the designed one;
    the reference lists come from the oracle's transform of the same (fp32-quantised) samples."""
    import torch
    b = 37
    for flexible in (True, False):
        k = 4 if flexible else 5
        x1 = designed_samples(n, flexible).astype(dt)
        spec = c_oracle.start_fft_batch(x1.astype(np.float64)[None, :])[0]
        key = ("samples", n, np.dtype(dt).name)
        fs_w = fs_per_window(fs_classes(key, spec, flexible, k), b, seed=n + 7)
        x = np.repeat(x1[None, :], b, axis=0)
        buf, ptr = rows_on_device(x, n, 0)
        d_fs = torch.from_numpy(fs_w).to("cuda:0")
        want = lambda w: oracle_list(key, spec, fs_w[w], flexible, k)      # noqa: E731
        with generic(an, gen):
            for ws in (False, True):
                raw, _ = analyze_dev(an, ptr, n, n, b, n, dt, flexible, fs=fs_w[0] + 1.0, d_fs=d_fs, k=k, ws=ws)
                recs = check_records(raw, 5, k, n, flexible, fs_w, want, exact=dt == np.float64)
                assert len({tuple(r["pk"]["idx"][:r["count"]]) for r in recs}) >= 2
            if dt == np.float32 and 1024 <= n <= 8192 and not gen:
                raw = fused_dev(an, ptr, n, n, b, n, flexible, fs=fs_w[0] + 1.0, d_fs=d_fs, k=k)
                check_records(raw, 5, k, n, flexible, fs_w, want, exact=False)


# ---------------------------------------------------------------------------------------------------------------
# 4. k and record width
# ---------------------------------------------------------------------------------------------------------------
def noise_spectra(b, n, dt, seed):
    """Noise-like magnitudes (Rayleigh, on a 2^-16 grid: exact in fp32, so both precisions decide alike) with a few
    lines: dozens of candidates per window.  Other sizes get a quiet floor with up to 90 isolated lines below bin 400
    instead: the reference keeps most of them (its damping window drops single-bin lines far up the spectrum, and it
    keeps few noise maxima of a short spectrum), and its picker stays fast at 2^16 bins."""
    rng = np.random.default_rng(seed)
    half = n // 2
    if 2048 <= n <= 8192:
        m = np.round(rng.rayleigh(1.0, (b, half)) * 65536.0) / 65536.0
    else:
        m = np.round(rng.uniform(0.01, 0.02, (b, half)) * 65536.0) / 65536.0
        spots = np.arange(12, min(half - 2, 400), 3)
        cnt = min(90, 3 * spots.size // 4)
        for w in range(b):
            at = rng.choice(spots, size=cnt, replace=False)
            m[w, at] = np.round(rng.uniform(1.0, 9.0, cnt) * 65536.0) / 65536.0
    m[:, 0] = 0.0
    m[:, 300 % (half - 1)] = 12.0
    m[::3, (7 * half) // 10] = 9.5
    z = np.zeros((b, n), dtype=_cdt(dt))
    z[:, :half] = m
    return z


def _caps(n):
    mp = max_peaks(n)
    out = [(5, k) for k in range(1, 6)]
    for cap in (6, 16, 64, mp):
        out += [(cap, cap), (cap, max(1, cap // 3))]
    return out


K_ROUTES = [("fast", 1024, False, 7, None), ("fast", 4096, False, 7, None), ("fast", 8192, False, 7, None),
            ("repair", 8192, False, 5, "spikes"), ("general", 512, False, 7, None), ("general_generic", 4096, True, 7, None),
            ("general_32k", 32768, False, 3, None), ("general_global_generic", 1 << 16, True, 3, None),
            ("large", 1 << 16, False, 3, None)]


@pytest.mark.gpu
@pytest.mark.parametrize("route,n,gen,b,kind", K_ROUTES, ids=[f"{r[0]}-{r[1]}" for r in K_ROUTES])
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_k_and_record_width(route, n, gen, b, kind, dt, an):
    """k = 1..5 in 128-byte records and rec_cap in {6, 16, 64, APDA_MAX_PEAKS(n)} with k = rec_cap and k < rec_cap,
    records starting as 0xA5 bytes: everything written, empty slots as the general kernel writes them, lists equal to
    the reference (dicts in fp64, indices in fp32), nothing written past the last record."""
    rng = np.random.default_rng(n + b)
    for flexible in (True, False):
        if kind == "spikes":
            z = designed_spectra(b, n, flexible, dt, **_design_kw("spikes", flexible))
        else:
            z = noise_spectra(b, n, dt, seed=n)
        fs_w = np.round(rng.uniform(50.0, 1000.0, b), 3)
        with generic(an, gen):
            for cap, k in _caps(n):
                raw = peaks_dev(an, z, flexible, fs=125.0, fs_w=fs_w, k=k, cap=cap)
                key = ("k", kind, n, b)     # the same magnitudes in both precisions and on every route of this n
                recs = check_records(raw, cap, k, n, flexible, fs_w,
                                     lambda w: oracle_list(key + (w,), z[w], fs_w[w], flexible, k),
                                     exact=dt == np.float64)
                if cap == 64 and k == 64 and kind is None:     # the wide records were really needed
                    assert recs["count"].max() >= (17 if flexible else 6), (flexible, recs["count"])


@pytest.mark.gpu
def test_k_fused_tail(an):
    """The fused kernel's tail for k = 1..5 (fp32, 128-byte records that start as 0xA5 bytes)."""
    import torch
    b, n = 9, 4096
    rng = np.random.default_rng(5)
    x = np.round(rng.standard_normal((b, n)) * 0.3 + 0.5 * np.sin(np.arange(n) * 0.3) + 1.0, 6).astype(np.float32)
    spec = c_oracle.start_fft_batch(x.astype(np.float64))
    fs_w = np.round(rng.uniform(50.0, 1000.0, b), 3)
    buf, ptr = rows_on_device(x, n, 0)
    d_fs = torch.from_numpy(fs_w).to("cuda:0")
    for flexible in (True, False):
        for k in range(1, 6):
            raw = fused_dev(an, ptr, n, n, b, n, flexible, d_fs=d_fs, k=k)
            check_records(raw, 5, k, n, flexible, fs_w, lambda w: oracle_list(("fused", w), spec[w], fs_w[w], flexible, k),
                          exact=False)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [512, 4096])
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_k_and_record_width_ragged(n, dt, an):
    """apda_analyze_ragged_* with wide records: the status kernel rewrites headers at APDA_REC_BYTES(rec_cap) strides
    (bit 4: other padded length, bit 8: empty window), every other byte is the picker's."""
    import torch
    b = 11
    nv = np.array([n, n // 2 - 3, 0, n, n - 1, n // 2 + 1, 1, n, n, 3 * n // 4, n], dtype=np.int32)
    x = skewed_windows(b, n, seed=n + 9).astype(dt)
    for w in range(b):
        x[w, nv[w]:] = np.nan
    buf, ptr = rows_on_device(x, n, 0)
    d_nv = torch.from_numpy(nv).to("cuda:0")
    fs_w = np.round(np.random.default_rng(n).uniform(50.0, 1000.0, b), 3)
    d_fs = torch.from_numpy(fs_w).to("cuda:0")
    want_status = [8 if v == 0 else (4 if c_oracle.padded_len(int(v)) != n else 0) for v in nv]
    for flexible in (True, False):
        for cap, k in _caps(n):
            raw, spec = analyze_ragged_dev(an, ptr, d_nv, n, n, b, n, dt, flexible, d_fs=d_fs, k=k, cap=cap, ws=True)
            recs = raw.view(rec_dtype(cap)).reshape(b)
            assert [int(s) & ~16 for s in recs["status"]] == want_status, (cap, k, recs["status"])
            assert recs["count"][2] == 0
            slots = raw[:, 8:].reshape(b, cap, 24)
            for w in range(b):
                assert (slots[w, recs["count"][w]:] == EMPTY_SLOT).all(), (cap, k, w)
            full = np.flatnonzero(nv == n)
            check_records(raw[full], cap, k, n, flexible, fs_w[full],
                          lambda i: oracle_list(("ragged", n, np.dtype(dt).name, int(full[i])),
                                                c_oracle.start_fft_batch(x[full[i]:full[i] + 1].astype(np.float64))[0],
                                                fs_w[full[i]], flexible, k),
                          exact=dt == np.float64)
