"""The length axis (include/apda_b200.h, DESIGN.md K1 / K2 / K3): every transform length N = 2^1 ... 2^30 and batches past
K2's launch limits, on every route that length selects.

  1. N = 2^1 ... 2^25 against the C oracle, full (n_samples = N) and odd padded (N/2 + 1) windows, batches that cross
     each route's unit (a tail block of K1 / K3 windows; K2's median launch sets of min(256, 256 MB / row) windows;
     K3-large's launch sets of at most 64), through apda_fft / apda_analyze (own and caller workspace) / apda_peaks on the
     oracle's spectrum / the _host entry points / apda_fft_c2c_f64_host; N <= 2^16 again under generic_only.  Pickers
     are held to the reference up to 2^24, the spectrum alone above.
  2. The host pipeline at 2^21 ... 2^24 (three-pass plans) with three different windows: chunks of several windows and
     chunks that alternate between the pipeline's two streams.
  3. N = 2^26 ... 2^30 on periodic windows, whose spectrum is known exactly, checked on the device.
  4. 65537 windows at N = 2^14 (more than gridDim.y holds) and the ragged entry points at the shared-memory limit.

Windows of one batch are one designed window shifted by multiples of 1/8 (exact in fp32 too): every route centres with
one subtraction of the exact median, so every window's spectrum and record must be bit-equal to window 0's, and a
window centred with another window's median (or never centred) differs from it in every bin of a padded window.
fp64 is held bit for bit to the C oracle; fp32 spectra to the oracle within the suite's K1 (N <= 8192) / K2 bounds,
fp32 records by the oracle's index lists.
"""
import ctypes
import statistics

import numpy as np
import pytest

from oracle import c_oracle
from test_gpu_abi_space import (CENTER_MEDIAN, _cdt, _sfx, analyze_dev, analyze_ragged_dev, check_records, fft_dev,
                                fft_ragged_dev, fp32_bound, generic, k1_bound, k2_bound, peaks_dev, rec_dtype,
                                rows_on_device)

_p = ctypes.c_void_p
FS = 125.0
U64 = 2.0 ** -53
# (cycles per window as a fraction of min(n_samples, 1024), amplitude): distinct amplitudes, at least 5 % apart in
# frequency; the cycle counts end in .15, so each tone has one clearly highest bin and no two bins of it are near-equal
TONES = ((0.045, 1.0), (0.081, 0.85), (0.122, 0.7), (0.161, 0.6), (0.203, 0.5), (0.244, 0.42))


# ---------------------------------------------------------------------------------------------------------------
# fixtures, inputs and references
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def an():
    import torch
    import apda_fft_b200
    a = apda_fft_b200.Analyzer(0)
    a.use_stream(torch.cuda.current_stream(torch.device("cuda:0")).cuda_stream)
    yield a
    a.use_stream(None)


def own_analyzer():
    """A context of its own, closed by the caller: the largest tests must not leave their twiddle tables and
    workspaces (tens of GB) in the module's context."""
    import torch
    import apda_fft_b200
    a = apda_fft_b200.Analyzer(0)
    a.use_stream(torch.cuda.current_stream(torch.device("cuda:0")).cuda_stream)
    return a


def need_device_memory(nbytes):
    import torch
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes + (2 << 30):
        pytest.skip(f"needs {nbytes} bytes of device memory (+2 GiB margin), {free} free")


def need_host_memory(nbytes):
    with open("/proc/meminfo") as fh:
        info = {ln.split(":")[0]: int(ln.split()[1]) * 1024 for ln in fh}
    if info.get("MemAvailable", 0) < nbytes + (4 << 30):
        pytest.skip(f"needs {nbytes} bytes of host memory (+4 GiB margin), {info.get('MemAvailable')} available")


def tone_window(ns, seed=0):
    """Six Hann-tapered tones (TONES) plus Gaussian noise of 0.05, on a 2^-20 grid inside +-5: exact in fp32, and stays
    so after a shift by up to +-1 or a scale by 2 or 4.  The taper keeps the sidelobes of padded windows below the
    pickers' threshold, which keeps the reference pickers affordable at 2^24."""
    rng = np.random.default_rng(seed)
    m = min(ns, 1024)
    i = np.arange(ns, dtype=np.float64)
    x = 0.05 * rng.standard_normal(ns)
    taper = 0.5 - 0.5 * np.cos(2 * np.pi * (i + 0.5) / ns)
    for r, a in TONES:
        x += a * taper * np.sin(2 * np.pi * (np.floor(r * m) + 0.15) * i / ns + 7 * r + seed)
    return np.round(x * 2.0 ** 20) / 2.0 ** 20


def shifts(b):
    """Per-window offsets, multiples of 1/8 in [-1, 1], not periodic in any launch-set size."""
    return 0.125 * ((5 * np.arange(b)) % 17) - 1.0


def inputs(n):
    return (n,) if n < 4 else (n, n // 2 + 1)


_SPEC, _LIST, _C2C = {}, {}, {}


def oracle_spec(n, ns):
    """start_fft of tone_window(ns) at N = n (the window is exact in fp32, so this is also the oracle of the
    fp32-quantised samples), cached for the module; only the sizes of part 2 are kept after their test."""
    key = (n, ns)
    if key not in _SPEC:
        for k in [k for k in _SPEC if k[0] > 1 << 24]:
            del _SPEC[k]
        _SPEC[key] = c_oracle.start_fft_batch(tone_window(ns)[None, :], n_fft=n)[0]
    return _SPEC[key]


def oracle_list(n, ns, flexible):
    key = (n, ns, flexible)
    if key not in _LIST:
        spec = oracle_spec(n, ns)
        _LIST[key] = c_oracle.peaks_prominence(spec, FS, 4) if flexible else c_oracle.peaks_resolution(spec, FS, 5)
    return _LIST[key]


def c2c_input(n):
    z = np.zeros(n, dtype=np.complex128)
    x = tone_window(max(1, n // 2 + 1))[:n]
    z[:x.shape[0]] = x
    z.imag[:x.shape[0]] = 0.5 * np.roll(x, 3)
    return z


def median_windows(ns, dt):
    return max(1, min(256, (256 << 20) // (ns * np.dtype(dt).itemsize)))


def batch_for(n, ns, dt):
    """K1 / K3-fast: 37 windows (a tail block); K2: one more window than a median launch set, and for K3-large
    (N >= 2^16) more than its 64-window launch set; one window above 2^20."""
    if n <= 8192:
        return 37
    if n > 1 << 20:
        return 1
    b = median_windows(ns, dt) + 1
    return max(b, 65) if n >= 1 << 16 else b


def rows_bit_equal(a):
    """Every row of a [b, ...] array has the bytes of row 0."""
    v = np.ascontiguousarray(a).view(np.uint8).reshape(a.shape[0], -1)
    bad = np.flatnonzero((v != v[:1]).any(axis=1))
    assert bad.size == 0, f"windows {bad[:8]} differ from window 0"


def check_spectrum(got0, want, x0, n, dt, what):
    if dt == np.float64:
        assert np.array_equal(got0.view(np.float64), want.view(np.float64)), (what, "fp64 vs oracle")
    else:
        err = np.abs(got0.astype(np.complex128) - want).max()
        assert err <= fp32_bound(n, want, x0.astype(np.float32)), (what, err)


def check_list(raw, n, ns, flexible, dt, what):
    """raw: uint8[b, 128] records; all equal to window 0's, and window 0's equal to the reference list."""
    rows_bit_equal(raw)
    k = 4 if flexible else 5
    check_records(raw[:1], 5, k, n, flexible, [FS], lambda w: oracle_list(n, ns, flexible)[:k], exact=dt == np.float64)


def host_fft(an, x, n, dt):
    b, ns = x.shape
    out = np.empty((b, n), dtype=_cdt(dt))
    an.ctx.call(f"apda_fft_{_sfx(dt)}_host", _p(x.ctypes.data), ns, ns, b, n, CENTER_MEDIAN, _p(out.ctypes.data))
    return out


def host_analyze(an, x, n, dt, flexible):
    b, ns = x.shape
    recs = np.zeros(b, dtype=rec_dtype(5))
    recs.view(np.uint8)[:] = 0xA5
    an.ctx.call(f"apda_analyze_{_sfx(dt)}_host", _p(x.ctypes.data), ns, ns, b, n, CENTER_MEDIAN, int(flexible), FS,
                _p(0), 4 if flexible else 5, 5, _p(recs.ctypes.data))
    return recs.view(np.uint8).reshape(b, -1)


def peaks_on(an, z, b, flexible):
    """apda_peaks_*_dev on b copies of spectrum z (complex64 -> fp32 pickers)."""
    return peaks_dev(an, np.repeat(z[None, :], b, axis=0), flexible)


# ---------------------------------------------------------------------------------------------------------------
# 1. every length against the oracle
# ---------------------------------------------------------------------------------------------------------------
SWEEP = [(lg, dt, gen) for lg in range(1, 26) for dt in (np.float64, np.float32) for gen in (False, True)
         if not gen or lg <= 16]


@pytest.mark.gpu
@pytest.mark.parametrize("lg,dt,gen", SWEEP,
                         ids=[f"2^{lg}-{_sfx(dt)}{'-generic' if gen else ''}" for lg, dt, gen in SWEEP])
def test_length_sweep(lg, dt, gen, an):
    """fp64 bit-equal to the oracle, fp32 within the K1 / K2 bound; every window of the batch bit-equal to window 0
    (spectra and records), the caller's workspace and the _host pipeline bit-equal to apda_fft_*_dev, records equal to
    the reference's lists (N >= 4, N <= 2^24), pickers on the oracle's own spectrum too; apda_fft_c2c_f64_host
    bit-equal to the oracle's fft(x)."""
    import torch
    n = 1 << lg
    with generic(an, gen):
        for ns in inputs(n):
            b = batch_for(n, ns, dt)
            x0 = tone_window(ns)
            x = (x0[None, :] + shifts(b)[:, None]).astype(dt)
            want = oracle_spec(n, ns)
            buf, ptr = rows_on_device(x, ns, 0)
            spec = fft_dev(an, ptr, ns, ns, b, n, dt)
            rows_bit_equal(spec)
            check_spectrum(spec[0], want, x0, n, dt, ("fft_dev", ns, b))
            host = host_fft(an, x, n, dt)
            assert np.array_equal(host.view(np.uint8), spec.view(np.uint8)), ("fft_host", ns)
            del host
            if n < 4:       # one bin of half spectrum: the reference's pickers raise (test_oracle covers the error)
                continue
            pick = n <= 1 << 24
            for flexible in (True, False):
                own, _ = analyze_dev(an, ptr, ns, ns, b, n, dt, flexible)
                ws, wsspec = analyze_dev(an, ptr, ns, ns, b, n, dt, flexible, ws=True)
                assert np.array_equal(wsspec.view(np.uint8), spec.view(np.uint8)), ("analyze workspace", ns, flexible)
                del wsspec
                hrec = host_analyze(an, x, n, dt, flexible)
                assert np.array_equal(hrec, own), ("analyze_host", ns, flexible)
                if pick:
                    check_list(own, n, ns, flexible, dt, "analyze own")
                    check_list(ws, n, ns, flexible, dt, "analyze ws")
                    z = want.astype(_cdt(dt))
                    check_list(peaks_on(an, z, min(b, 65), flexible), n, ns, flexible, dt, "peaks on oracle spectrum")
                else:
                    rows_bit_equal(own)
                    rows_bit_equal(ws)
            del buf
            torch.cuda.empty_cache()
    if dt == np.float64 and not gen:
        z = c2c_input(n)
        if n not in _C2C:
            _C2C.clear()
            _C2C[n] = c_oracle.fft_c2c(z)
        zz = np.stack([z, 2 * z])
        out = np.empty_like(zz)
        an.ctx.call("apda_fft_c2c_f64_host", _p(zz.ctypes.data), 2, n, _p(out.ctypes.data))
        assert np.array_equal(out[0].view(np.float64), _C2C[n].view(np.float64)), "c2c vs oracle"
        assert np.array_equal(out[1].view(np.float64), (2 * _C2C[n]).view(np.float64)), "c2c, window 1"


# ---------------------------------------------------------------------------------------------------------------
# 2. the host pipeline at three-pass sizes with several windows
# ---------------------------------------------------------------------------------------------------------------
HOST = [(lg, dt) for lg in range(21, 25) for dt in (np.float64, np.float32)]


@pytest.mark.gpu
@pytest.mark.parametrize("lg,dt", HOST, ids=[f"2^{lg}-{_sfx(dt)}" for lg, dt in HOST])
def test_host_pipeline_three_pass_batches(lg, dt, an):
    """apda_fft_*_host / apda_analyze_*_host on windows 2^w * x, w = 0, 1, 2, padded (N/2 + 1 samples): at these sizes
    the pipeline runs three-pass K2 plans over chunks of three windows (2^21, and 2^22 in fp32) or one-window chunks on
    alternating streams, each stream with its own median scratch and picker workspace.  Scaling by 2^w is exact
    everywhere, so window w must be 2^w times window 0 bit for bit (spectra, magnitudes and prominences), and window 0
    must match the oracle."""
    n = 1 << lg
    ns = n // 2 + 1
    x0 = tone_window(ns)
    x = np.stack([x0 * 2.0 ** w for w in range(3)]).astype(dt)
    want = oracle_spec(n, ns)
    spec = host_fft(an, x, n, dt)
    check_spectrum(spec[0], want, x0, n, dt, "window 0")
    for w in (1, 2):
        assert np.array_equal(spec[w].view(dt), (spec[0] * dt(2.0 ** w)).view(dt)), ("window", w)
    del spec
    for flexible in (True, False):
        raw = host_analyze(an, x, n, dt, flexible)
        k = 4 if flexible else 5
        check_records(raw[:1], 5, k, n, flexible, [FS], lambda w: oracle_list(n, ns, flexible)[:k],
                      exact=dt == np.float64)
        recs = raw.view(rec_dtype(5)).reshape(3)
        assert recs["count"][0] >= 3, (flexible, recs["count"])
        for w in (1, 2):
            assert recs["count"][w] == recs["count"][0] and recs["status"][w] == recs["status"][0], (flexible, w)
            c = recs["count"][0]
            a, r = recs["pk"][w][:c], recs["pk"][0][:c]
            assert (a["idx"] == r["idx"]).all() and (a["width_bins"] == r["width_bins"]).all(), (flexible, w)
            assert (a["mag"] == r["mag"] * 2.0 ** w).all() and (a["prominence"] == r["prominence"] * 2.0 ** w).all()


# ---------------------------------------------------------------------------------------------------------------
# 3. beyond the oracle: periodic windows of 2^26 ... 2^30 samples
# ---------------------------------------------------------------------------------------------------------------
# (period P, seed): P | N, dyadic pattern values; the spikes of the half spectrum have magnitudes at least 2 % apart
DESIGNS = ((64, 8), (16, 3))
OFFSET = 2.5


def pattern(P, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(-32, 33, P) / 8.0


def exact_spikes(P, seed, n):
    """(median, spike bins m*N/P for m = 1 .. P-1, their exact values (N/P) * DFT_P(p - median)[m], rms(p - median))."""
    p = pattern(P, seed) + OFFSET
    med = statistics.median(p.tolist())
    d = np.fft.fft(p - med)
    m = np.arange(1, P)
    return med, m * (n // P), (n // P) * d[1:], float(np.sqrt(np.mean((p - med) ** 2)))


def fp64_bound(n, rms):
    """Max-bin error bound of the fp64 transform of a window with rms(x - median) = rms: ||X||_2 = N * rms times
    (4 N + 5 log2 N) u.  The twiddle recurrence's own drift is at most 4 (j + 1) u on the j-th entry of a stage (each
    complex product rounds by at most sqrt(5) u, the step by sqrt(2) u; test_twiddle_drift_premise checks it), which
    sums to 4 N u over the stages; each stage's butterflies add at most 5 u (norm-wise, first order)."""
    lg = n.bit_length() - 1
    return (4.0 * n + 5.0 * lg) * U64 * n * rms


def periodic_bounds(n, dt, want_sp, rms):
    if dt == np.float32:
        return k2_bound(want_sp)
    return fp64_bound(n, rms)


def dilated_reference(P, seed, flexible):
    n16 = 1 << 16
    x = np.tile(pattern(P, seed) + OFFSET, n16 // P)
    spec = c_oracle.start_fft_batch(x[None, :])[0]
    return c_oracle.peaks_prominence(spec, FS, 4) if flexible else c_oracle.peaks_resolution(spec, FS, 5)


def test_twiddle_drift_premise():
    """The fp64 bound of part 3 assumes the reference's recurrence twiddles drift by at most 4 (j + 1) u from
    exp(-i pi j / h) on entry j of the stage of half-span h: checked on the oracle's table at 2^20."""
    n = 1 << 20
    tw = c_oracle.twiddle_table(n)
    h = 1
    while h < n:
        j = np.arange(h)
        exact = np.exp(-1j * np.pi * j / h)
        drift = np.abs(tw[h - 1:2 * h - 1] - exact)
        assert (drift <= 4.0 * (j + 1) * U64 + 2 * U64).all(), (h, float((drift / ((j + 1) * U64)).max()))
        h *= 2


@pytest.mark.parametrize("P,seed", DESIGNS)
def test_periodic_designs_dilate(P, seed):
    """Without a GPU: the oracle at N = 2^12, 2^14, 2^16 on the periodic design equals the exact spikes within the
    fp64 bound of part 3, every other bin stays under it, and the rigid picker's list at N is the 2^16 list with its
    indices scaled by N / 2^16 (same frequencies, magnitudes scaled by N / 2^16, spikes 2 % apart so that fp32 keeps
    their order).  The flexible picker's damping gate 1 / (2 q) with q = j / width depends on the bin j itself: with
    P <= 64 every spike of N >= 2^16 sits at j >= 1024, below damping 0.001, so that list is empty at 2^16 and at every
    larger N - the dilation holds for it from 2^16 on, and only there."""
    ref16 = dilated_reference(P, seed, False)
    assert len(ref16) == 5, ref16
    mags = sorted((p["mag"] for p in ref16), reverse=True)
    assert all(a > b * 1.02 for a, b in zip(mags, mags[1:])), mags
    assert dilated_reference(P, seed, True) == []
    for lg in (12, 14, 16):
        n = 1 << lg
        x = np.tile(pattern(P, seed) + OFFSET, n // P)
        assert statistics.median(x.tolist()) == exact_spikes(P, seed, n)[0]
        spec = c_oracle.start_fft_batch(x[None, :])[0]
        med, at, want, rms = exact_spikes(P, seed, n)
        bound = fp64_bound(n, rms)
        assert np.abs(spec[at] - want).max() <= bound
        rest = spec.copy()
        rest[at] = 0
        assert np.abs(rest).max() <= bound and spec[0] == 0
        got = c_oracle.peaks_resolution(spec, FS, 5)
        s = n / (1 << 16)
        assert [p["idx"] for p in got] == [int(p["idx"] * s) for p in ref16], (lg, got)
        for a, r in zip(got, ref16):
            assert abs(a["freq"] - r["freq"]) <= 1e-12 * r["freq"]
            assert abs(a["mag"] - r["mag"] * s) <= 1e-9 * a["mag"]


LARGE = [(lg, dt) for lg in range(26, 31) for dt in (np.float32, np.float64)]


@pytest.mark.gpu
@pytest.mark.parametrize("lg,dt", LARGE, ids=[f"2^{lg}-{_sfx(dt)}" for lg, dt in LARGE])
def test_periodic_beyond_oracle(lg, dt):
    """x[i] = p[i mod P] + 2.5 at N = 2^26 ... 2^30, checked on the device: spike bins m*N/P equal (N/P) * DFT_P(p -
    median)[m] and every other bin is (near) zero, both within the K2 bound of the largest spike (fp32) or the derived
    fp64 bound (fp64_bound), bin 0 exactly 0; the rigid picker reports the 2^16 oracle's spikes dilated by N / 2^16
    (indices, half-height widths of 2 bins, magnitudes within the same bound), the flexible picker nothing."""
    import torch
    n = 1 << lg
    s = np.dtype(dt).itemsize
    # samples, spectrum, the median's bucket copy, the pickers' magnitude workspace, both twiddle tables (24 N bytes)
    need_device_memory(n * (s + 2 * s + s + 2 * s) + 24 * n)
    need_host_memory(24 * n)
    tdt = torch.float32 if dt == np.float32 else torch.float64
    a = own_analyzer()
    try:
        for P, seed in DESIGNS:
            med, at, want_sp, rms = exact_spikes(P, seed, n)
            x = torch.tensor(pattern(P, seed) + OFFSET, dtype=tdt, device="cuda:0").repeat(n // P)
            spec = torch.empty(2 * n, dtype=tdt, device="cuda:0")
            a.ctx.call(f"apda_fft_{_sfx(dt)}_dev", _p(x.data_ptr()), n, n, 1, n, CENTER_MEDIAN, _p(spec.data_ptr()))
            z = torch.view_as_complex(spec.view(n, 2))
            bound = periodic_bounds(n, dt, want_sp, rms)
            idx = torch.from_numpy(at).to("cuda:0")
            got_sp = z[idx].cpu().numpy().astype(np.complex128)
            err = np.abs(got_sp - want_sp).max()
            assert err <= bound, (P, "spikes", err, bound)
            assert float(z[0].abs()) == 0.0
            recs = {}
            for flexible in (False, True):
                raw = torch.full((128,), 0xA5, dtype=torch.uint8, device="cuda:0")
                a.ctx.call(f"apda_analyze_{_sfx(dt)}_dev", _p(x.data_ptr()), n, n, 1, n, CENTER_MEDIAN, int(flexible),
                           FS, _p(0), 4 if flexible else 5, 5, _p(spec.data_ptr()), _p(raw.data_ptr()))
                torch.cuda.synchronize()
                recs[flexible] = raw.cpu().numpy().view(rec_dtype(5))[0]
            # the caller's workspace holds the spectrum apda_fft wrote: check the bins off the spikes last
            z[idx] = 0
            rest = max(float(z[i:i + (1 << 26)].abs().max()) for i in range(0, n, 1 << 26))
            assert rest <= bound, (P, "off-spike bins", rest, bound)
            del x, spec, z
            torch.cuda.empty_cache()
            assert recs[True]["count"] == 0 and recs[True]["status"] == 0, recs[True]
            rig = recs[False]
            ref = dilated_reference(P, seed, False)
            scale = n >> 16
            assert rig["status"] == 0 and rig["count"] == len(ref), rig
            pk = rig["pk"][:rig["count"]]
            assert [int(i) for i in pk["idx"]] == [r["idx"] * scale for r in ref], (P, pk["idx"])
            assert (pk["width_bins"] == 2).all(), pk["width_bins"]
            for got_m, r in zip(pk["mag"], ref):
                assert abs(got_m - r["mag"] * scale) <= bound + 1e-9 * got_m, (P, got_m, r["mag"] * scale)
    finally:
        a.ctx.close()
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------
# 4. batches past the launch limits, and the ragged entry points at the shared-memory limit
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_batch_beyond_grid_y(dt):
    """65537 windows of N = 2^14 (n_samples = N - 3) through apda_fft_*_dev and apda_analyze_*_dev: K2 puts windows on
    gridDim.y (at most 65535), so the batch runs in two launch sets, and the median in launch sets of 256.  Window w is
    template w mod 7 (7 is prime to 256 and 65535): every window bit-equal to its template's result, the templates
    equal to the oracle (spectra and both pickers' lists)."""
    import torch
    n, ns, B, T = 1 << 14, (1 << 14) - 3, 65537, 7
    s = np.dtype(dt).itemsize
    need_device_memory(B * (ns + 2 * n) * s + B * 2 * n * s // 2)
    tdt = torch.float32 if dt == np.float32 else torch.float64
    idt = torch.int32 if dt == np.float32 else torch.int64
    tmpl = np.stack([tone_window(ns, seed=t + 1) for t in range(T)])
    want = c_oracle.start_fft_batch(tmpl, n_fft=n)
    a = own_analyzer()
    try:
        sel = torch.arange(B, device="cuda:0") % T
        x = torch.from_numpy(tmpl).to(device="cuda:0", dtype=tdt)[sel].contiguous()

        def same_as_template(v):
            """v[B, row]: every row bit-equal to row (w mod 7)."""
            for i in range(0, B, 4096):
                j = min(B, i + 4096)
                bad = (v[i:j] != v[:T][sel[i:j]]).any(dim=1)
                assert not bool(bad.any()), ("window", i + int(torch.nonzero(bad)[0]))

        spec = torch.full((B, 2 * n), float("nan"), dtype=tdt, device="cuda:0")
        a.ctx.call(f"apda_fft_{_sfx(dt)}_dev", _p(x.data_ptr()), ns, ns, B, n, CENTER_MEDIAN, _p(spec.data_ptr()))
        torch.cuda.synchronize()
        same_as_template(spec.view(idt))
        got = spec[:T].cpu().numpy().view(_cdt(dt))
        for t in range(T):
            check_spectrum(got[t], want[t], tmpl[t], n, dt, ("template", t))
        del spec
        torch.cuda.empty_cache()
        for flexible in (True, False):
            k = 4 if flexible else 5
            rec = torch.full((B, 128), 0xA5, dtype=torch.uint8, device="cuda:0")
            a.ctx.call(f"apda_analyze_{_sfx(dt)}_dev", _p(x.data_ptr()), ns, ns, B, n, CENTER_MEDIAN, int(flexible), FS,
                       _p(0), k, 5, _p(0), _p(rec.data_ptr()))
            torch.cuda.synchronize()
            same_as_template(rec)
            check_records(rec[:T].cpu().numpy(), 5, k, n, flexible, [FS] * T,
                          lambda w: (c_oracle.peaks_prominence(want[w], FS, k) if flexible
                                     else c_oracle.peaks_resolution(want[w], FS, k)), exact=dt == np.float64)
    finally:
        a.ctx.close()
        torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.float32, np.float64], ids=["f32", "f64"])
def test_ragged_at_shared_memory_limit(dt, an):
    """apda_fft_ragged / apda_analyze_ragged at N = fft_smem_max_n (fp32 2^14, the only caller of the fp32 shared-memory
    kernel at that size; fp64 2^13) with mixed lengths: spectra against the oracle at each window's own sample count
    (fp64 bit for bit, fp32 within the K1 bound), status bit 4 exactly for windows whose padded length is not N, and
    the full-length windows' records equal to the reference's lists."""
    import torch
    n = 16384 if dt == np.float32 else 8192
    b = 23
    nv = np.array([n, n - 3, n // 2 + 1, n, 3 * n // 4 + 1, n // 2, n - 1, n, 1, n // 4 + 7, n, 2] * 2, dtype=np.int32)[:b]
    x = np.full((b, n), np.nan)
    for w in range(b):
        x[w, :nv[w]] = tone_window(int(nv[w]), seed=w)
    x = x.astype(dt)
    buf, ptr = rows_on_device(x, n, 0)
    d_nv = torch.from_numpy(nv).to("cuda:0")
    spec = fft_ragged_dev(an, ptr, d_nv, n, n, b, n, dt)
    wants = [c_oracle.start_fft_batch(x[w:w + 1, :nv[w]].astype(np.float64), n_fft=n)[0] for w in range(b)]
    for w in range(b):
        if dt == np.float64:
            assert np.array_equal(spec[w].view(np.float64), wants[w].view(np.float64)), (w, nv[w])
        else:
            err = np.abs(spec[w].astype(np.complex128) - wants[w]).max()
            assert err <= k1_bound(wants[w], x[w, :nv[w]]), (w, nv[w], err)
    full = np.flatnonzero(nv == n)
    other = np.array([c_oracle.padded_len(int(v)) != n for v in nv])
    for flexible in (True, False):
        k = 4 if flexible else 5
        raw, wsspec = analyze_ragged_dev(an, ptr, d_nv, n, n, b, n, dt, flexible, ws=True)
        assert np.array_equal(wsspec.view(np.uint8), spec.view(np.uint8)), flexible
        recs = raw.view(rec_dtype(5)).reshape(b)
        assert ((recs["status"] & 4 != 0) == other).all() and ((recs["status"] & ~(4 | 16)) == 0).all(), recs["status"]
        check_records(raw[full], 5, k, n, flexible, [FS] * full.size,
                      lambda i: (c_oracle.peaks_prominence(wants[full[i]], FS, k) if flexible
                                 else c_oracle.peaks_resolution(wants[full[i]], FS, k)), exact=dt == np.float64)
    del buf
