"""T2: CUDA path (through the C ABI) vs the oracle / the committed goldens.  Needs a B200: run with -m gpu.

Bars (north_star): fp64 - spectrum bit-exact (SHA-256 of the doubles), peak indices/counts exact, magnitudes and
prominences within rel 1e-12; fp32 - indices/counts exact on the well-separated inputs, values within rel 1e-5.
"""
import os
import statistics

import numpy as np
import pytest

import cases
from oracle import c_oracle, ref_port

pytestmark = pytest.mark.gpu

TOL64 = 1e-12
TOL32 = 1e-5


@pytest.fixture(scope="module")
def an():
    import apda_fft_b200
    return apda_fft_b200.Analyzer(0)


def _dicts(rec, fs, n, flexible):
    from apda_fft_b200.records import prominence_dicts, resolution_dicts
    return prominence_dicts(rec, fs, n) if flexible else resolution_dicts(rec, fs, n)


def assert_peaks_close(got, want, tol, what=""):
    assert [p["idx"] for p in got] == [p["idx"] for p in want], what
    for g, w in zip(got, want):
        assert set(g) == set(w)
        for key in w:
            if key == "idx":
                continue
            assert cases.isclose_rel(g[key], w[key], tol), (what, key, g[key], w[key])


FFT_CASES = [c for c in cases.CASES if c["id"] not in ("n1",)]


@pytest.mark.parametrize("spec", FFT_CASES, ids=[c["id"] for c in FFT_CASES])
def test_fft_f64_bit_exact_and_peaks(spec, golden, an):
    g = golden["cases"][spec["id"]]
    x, fs = cases.build_samples(spec)
    n = g["n_fft"]
    spectrum = an.fft(x)[0]
    assert spectrum.shape == (n,)
    assert cases.spectrum_sha16(spectrum) == g["spectrum_sha"], "fp64 spectrum is not bit-identical to the reference"
    for flexible, key in ((True, "prominence"), (False, "resolution")):
        if "error" in g[key]:
            with pytest.raises(statistics.StatisticsError):
                an.peaks(spectrum, fs, flexible=flexible)
            continue
        rec = an.peaks(spectrum, fs, flexible=flexible)[0]
        assert rec["status"] == 0
        assert_peaks_close(_dicts(rec, fs, n, flexible), g[key]["ok"], TOL64, (spec["id"], key))
        # fused pipeline entry point gives the same record
        rec2 = an.analyze(x, fs, flexible=flexible)[0]
        assert rec2.tobytes() == rec.tobytes()


def test_fp64_values_are_exact_on_kats(golden, an):
    """Stronger than the 1e-12 bar: with glibc's hypot sequence and double-double statistics the fp64 tables are
    the very same doubles as the reference's on the KATs."""
    for cid in ("katA", "katB", "katC"):
        g = golden["cases"][cid]
        x, fs = cases.build_samples(g["spec"])
        assert _dicts(an.analyze(x, fs, flexible=True)[0], fs, g["n_fft"], True) == g["prominence"]["ok"]
        assert _dicts(an.analyze(x, fs, flexible=False)[0], fs, g["n_fft"], False) == g["resolution"]["ok"]


@pytest.mark.parametrize("spec", cases.SPECTRA, ids=[c["id"] for c in cases.SPECTRA])
def test_picker_only_spectra(spec, golden, an):
    g = golden["spectra"][spec["id"]]
    z, fs = cases.build_spectrum(spec)
    for k in (4, 5, 12):
        for flexible, key in ((True, "prominence"), (False, "resolution")):
            rec = an.peaks(z, fs, flexible=flexible, k=k)[0]
            assert_peaks_close(_dicts(rec, fs, len(z), flexible), g[f"{key}_k{k}"]["ok"], TOL64, (spec["id"], key, k))


def test_k_variants(golden, an):
    by_id = {c["id"]: c for c in cases.CASES}
    for row in golden["k_variants"]:
        x, fs = cases.build_samples(by_id[row["case"]])
        n = c_oracle.padded_len(len(x))
        for flexible, key in ((True, "prominence"), (False, "resolution")):
            rec = an.analyze(x, fs, flexible=flexible, k=row["k"])[0]
            assert_peaks_close(_dicts(rec, fs, n, flexible), row[key]["ok"], TOL64, (row["case"], key, row["k"]))


def test_magnitudes_bit_identical_to_glibc_hypot(an):
    """K3's magnitude follows glibc's hypot operation sequence; check through the prominence of an isolated peak:
    prominence = mag[j] - mag[valley] is exact only if both magnitudes are the reference's doubles."""
    rng = np.random.default_rng(5)
    n = 2048
    z = (rng.standard_normal(n) + 1j * rng.standard_normal(n)) * 0.01
    z[0] = 0
    for j, amp in ((100, 50.0 + 3.3j), (400, -20.0 + 31.7j), (800, 7.77 - 19.1j)):
        z[j] = amp
    rec = an.peaks(z, 125.0, flexible=True, k=4)[0]
    want = ref_port.top_peaks_prominence(z.tolist(), 125.0, 4)
    assert _dicts(rec, 125.0, n, True) == want


def test_fft_c2c_bit_exact(golden, an):
    rng = np.random.default_rng(0)
    z = np.round(rng.standard_normal(64) + 1j * rng.standard_normal(64), 6)
    assert cases.spectrum_sha16(an.fft_c2c(z)[0]) == golden["fft_c2c_64"]["sha"]
    z = np.round(rng.standard_normal(4096) + 1j * rng.standard_normal(4096), 6)
    assert np.array_equal(an.fft_c2c(z)[0].view(np.float64), c_oracle.fft_c2c(z).view(np.float64))


def test_batch_f64_vs_c_oracle_multichunk(an):
    """3.5k windows x 4096 fp64 crosses the host pipeline's chunk boundary; spectra must match the C oracle bit for bit."""
    import apda_fft_b200.synth as synth
    b, n = 3500, 4096
    x = synth.fleet_windows(5000, b, n)
    spectra = an.fft(x)
    want = c_oracle.start_fft_batch(x)
    assert np.array_equal(spectra.view(np.float64), want.view(np.float64))
    recs = an.analyze(x, 125.0, flexible=True)
    assert (recs["count"] == 3).all() and (recs["status"] == 0).all()
    recs_r = an.analyze(x, 125.0, flexible=False)
    for w in list(range(0, 24)) + list(range(b - 24, b)) + [1535, 1536, 1537, 1750]:
        assert_peaks_close(_dicts(recs[w], 125.0, n, True), c_oracle.peaks_prominence(want[w], 125.0), TOL64, w)
        assert_peaks_close(_dicts(recs_r[w], 125.0, n, False), c_oracle.peaks_resolution(want[w], 125.0), TOL64, w)


def test_per_window_fs(an):
    import apda_fft_b200.synth as synth
    x = synth.fleet_windows(0, 6, 1024)
    fs = np.array([31.25, 62.5, 125.0, 250.0, 500.0, 44100.0])
    recs = an.analyze(x, fs, flexible=True)
    spectra = c_oracle.start_fft_batch(x)
    for w in range(6):
        assert_peaks_close(_dicts(recs[w], float(fs[w]), 1024, True), c_oracle.peaks_prominence(spectra[w], float(fs[w])),
                           TOL64, w)


F32_CASES = ["katA", "katB", "katC", "fleet4096_w0", "fleet4096_w0_onbin", "fleet8192_w7_onbin", "fleet1024_w1",
             "fleet2048_w5", "fleet4096_w3", "fleet4096_w999999", "fleet16384_w9", "pad1000", "pad3000", "six_tones"]


@pytest.mark.parametrize("cid", F32_CASES)
def test_f32_indices_exact_values_1e5(cid, golden, an):
    g = golden["cases"][cid]
    x, fs = cases.build_samples(g["spec"])
    x32 = x.astype(np.float32)
    n = g["n_fft"]
    spec32 = an.fft(x32)[0]
    want = c_oracle.start_fft_batch(x)[0]
    scale = np.abs(want).max()
    assert np.abs(spec32.astype(np.complex128) - want).max() <= 2e-6 * scale
    for flexible, key in ((True, "prominence"), (False, "resolution")):
        rec = an.analyze(x32, fs, flexible=flexible)[0]
        got = _dicts(rec, fs, n, flexible)
        assert [p["idx"] for p in got] == [p["idx"] for p in g[key]["ok"]], (cid, key)
        for gp, wp in zip(got, g[key]["ok"]):
            assert cases.isclose_rel(gp["mag"], wp["mag"], TOL32 + 1e-4 / max(abs(wp["mag"]), 1.0) * flexible)
            if flexible:
                assert cases.isclose_rel(gp["prominence"], wp["prominence"], TOL32)


def test_f32_mean_centering_equals_median_when_unpadded(an):
    """SURVEY finding 5: without padding the centring constant only moves bin 0, which is zeroed."""
    import apda_fft_b200
    import apda_fft_b200.synth as synth
    x = synth.fleet_windows(40, 32, 4096, dtype=np.float32)
    a = an.analyze(x, 125.0, flexible=True, center=apda_fft_b200._cabi.CENTER_MEDIAN)
    b = an.analyze(x, 125.0, flexible=True, center=apda_fft_b200._cabi.CENTER_MEAN)
    assert (a["count"] == b["count"]).all() and (a["pk"]["idx"] == b["pk"]["idx"]).all()
    live = a["pk"]["idx"] >= 0
    assert np.allclose(a["pk"]["mag"][live], b["pk"]["mag"][live], rtol=1e-5)
    with pytest.raises(ValueError):
        an.analyze(x[:, :3000], 125.0, center=apda_fft_b200._cabi.CENTER_MEAN)


def test_helper_functions(golden, an):
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "apda-fft_b200"))
    from utils.get_peak_prominence import calculate_half_power_width_prominenceBased, calculate_prominence
    from utils.get_peak_resolution import resolution, width_half_magnitude
    for blk in golden["helpers"]:
        mags = cases.mags_case(blk["seed"], blk["n"], blk["style"]).tolist()
        for row in blk["rows"]:
            j = row["j"]
            assert calculate_prominence(mags, j) == row["prominence"]
            assert calculate_half_power_width_prominenceBased(mags, row["prominence"], j, blk["fs"], blk["n_fft"]) == row["width_hz"]
            assert width_half_magnitude(mags, j) == row["whm"]
            assert resolution(mags, j, row["other"]) == row["rs"]


def test_device_pointer_api_and_synth(an):
    """The _dev entry points on torch-owned memory and stream; device generator vs host generator."""
    import torch
    import apda_fft_b200.synth as synth
    from apda_fft_b200.records import record_dtype
    b, n = 64, 4096
    dev = torch.device("cuda:0")
    stream = torch.cuda.current_stream(dev)
    an.use_stream(stream.cuda_stream)
    try:
        for dtype, tdt in (("f64", torch.float64), ("f32", torch.float32)):
            d_x = torch.empty((b, n), dtype=tdt, device=dev)
            an.synth_device(1000, b, n, dtype, d_x.data_ptr())
            d_rec = torch.zeros((b, 128), dtype=torch.uint8, device=dev)
            d_spec = torch.empty((b, n, 2), dtype=tdt, device=dev)
            an.analyze_device(d_x.data_ptr(), b, n, n, dtype, 125.0, d_rec.data_ptr(), d_spec_ws=d_spec.data_ptr())
            torch.cuda.synchronize()
            x = d_x.cpu().numpy()
            host = synth.fleet_windows(1000, b, n)
            assert np.abs(x - host).max() <= 1.000001e-6 and (x.astype(np.float64) == host.astype(x.dtype)).mean() > 0.999
            recs = d_rec.cpu().numpy().view(record_dtype(5)).reshape(b)
            want = c_oracle.start_fft_batch(x.astype(np.float64))
            if dtype == "f64":
                assert np.array_equal(d_spec.cpu().numpy().reshape(b, 2 * n), want.view(np.float64))
            for w in range(0, b, 7):
                ref = c_oracle.peaks_prominence(want[w], 125.0)
                got = _dicts(recs[w], 125.0, n, True)
                assert [p["idx"] for p in got] == [p["idx"] for p in ref]
    finally:
        an.use_stream(None)


def test_dropin_call_sequence(tmp_path, golden):
    """The call sequence of the reference's only caller (GT_FFT_v5.py:627-659) on the drop-in modules."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "apda-fft_b200"))
    from metrics.fft_iterativa import fft, remove_dc_component, start_fft
    from utils.get_peak_prominence import get_top_peaks_prominence
    from utils.get_peak_resolution import get_top_peaks_resolution
    from utils.load_data import load_sensor

    g = golden["cases"]["katA"]
    x, fs = cases.build_samples(g["spec"])
    path = tmp_path / "0013a20041e7f6b7_Xaxis.log"
    rows = ["2_11_22_18_20_32;2 g;125.0 Hz;X axis;", "Synced;", "25.010;-0.0222;0.0110;0.9981;85.0;", "0.268262;0.0;1.0;"]
    vals = ["%8.6f" % v for v in x]
    rows += [";".join(vals[i:i + 60]) + ";" for i in range(0, len(vals), 60)]
    rows.insert(9, "* MISSING PACKETS 3-4 *")
    path.write_text("\n".join(rows) + "\n")

    data = load_sensor(str(path))
    samples, fs_file, axis = data["samples"], data["metadata"]["fs"], data["metadata"]["axis"]
    assert (len(samples), fs_file, axis) == (1024, 125.0, "X")
    keep = list(samples)
    res_fft = start_fft(samples, fs_file)
    assert samples == keep and isinstance(res_fft, list) and res_fft[0] == 0 and type(res_fft[0]) is int
    assert cases.spectrum_sha16(res_fft) == g["spectrum_sha"]
    assert get_top_peaks_prominence(res_fft, fs_file) == g["prominence"]["ok"]
    assert get_top_peaks_resolution(res_fft, fs_file) == g["resolution"]["ok"]
    assert get_top_peaks_prominence(list(res_fft), fs_file) == g["prominence"]["ok"]      # plain list path
    peaks = get_top_peaks_prominence(res_fft, fs_file)
    entry = {"peak_freq": peaks[0]["freq"], "max_mag": peaks[0]["mag"]}
    assert entry == {"peak_freq": 3.0518, "max_mag": 195.833}
    # edge behaviour of the reference
    assert start_fft([], 1.0) == [0] and start_fft([1.0], 1.0) == [0]
    assert start_fft([1.0, 2.0], 1.0) == [0, (-1 + 0j)]
    with pytest.raises(statistics.StatisticsError, match="mean requires"):
        get_top_peaks_prominence([0], 1.0)
    with pytest.raises(statistics.StatisticsError, match="stdev requires"):
        get_top_peaks_resolution([0, (-1 + 0j)], 1.0)
    assert get_top_peaks_prominence(start_fft([1.0, -2.0, 3.5, 0.25], 1.0), 1.0) == []
    med = remove_dc_component([3.0, 1.0, 2.0, 10.0])
    assert med == [0.5, -1.5, -0.5, 7.5]
    z = [complex(i, -i) for i in range(8)]
    assert fft(list(z)) == ref_port.dit_radix2(z)
    assert start_fft(keep, fs_file)[1] == complex(*g["bins"]["1"])


@pytest.mark.parametrize("n_fft", [1024, 2048, 4096, 8192])
def test_f32_fast_kernel_median_and_padding(n_fft, an):
    """The fp32 fast kernel's in-register exact median: skewed, heavily tied data, odd/even/padded lengths.
    A wrong order statistic moves the low bins by ~1e-2 of the scale; the bound below is 3e-6."""
    rng = np.random.default_rng(n_fft)
    for n_samples in (n_fft, n_fft - 1, n_fft - 2, (3 * n_fft) // 4 + 1, n_fft // 2 + 1, n_fft // 2 + 2):
        rows = []
        rows.append(np.round(np.exp(rng.standard_normal(n_samples)), 2))                 # skewed, many ties
        rows.append(np.round(rng.standard_normal(n_samples) * 0.3 + 5.0, 3))             # large offset
        rows.append((rng.random(n_samples) < 0.5).astype(np.float64))                    # two values only
        rows.append(np.round(np.sin(np.arange(n_samples) * 0.05) + 0.2 * rng.standard_normal(n_samples), 6))
        rows.append(np.zeros(n_samples))                                                 # constant
        x = np.stack(rows).astype(np.float32)
        got = an.fft(x, n_fft=n_fft)
        want = c_oracle.start_fft_batch(x.astype(np.float64), n_fft=n_fft)
        for r in range(x.shape[0]):
            scale = max(np.abs(want[r]).max(), 1e-3)
            err = np.abs(got[r].astype(np.complex128) - want[r]).max()
            # the fp32 median itself carries half an ulp of |x|, which n_samples samples add coherently into the low bins
            assert err <= 3e-6 * scale + n_samples * float(np.abs(x[r]).max()) * 1.2e-7, (n_fft, n_samples, r, err, scale)


def _real_spiky_spectra(rng, b, n):
    """Purely real bins -> magnitudes are exact in fp32 and fp64, so every picker comparison is decided identically."""
    half = n // 2
    z = np.zeros((b, n), dtype=np.complex64)
    mags = np.exp(1.6 * rng.standard_normal((b, half))).astype(np.float32)
    mags[:, 0] = 0
    z[:, :half] = mags * np.where(rng.random((b, half)) < 0.5, -1, 1)
    return z


@pytest.mark.parametrize("n", [1024, 2048, 4096, 8192])
def test_f32_fast_picker_vs_oracle_spiky(n, an):
    """Heavy-tailed spectra: many candidates whose prominence walks stop in every chunk position (exercises the
    chunk-summary skipping of the warp-per-window kernel) - decisions must equal the oracle's exactly."""
    rng = np.random.default_rng(n + 1)
    b = 96
    z = _real_spiky_spectra(rng, b, n)
    for flexible in (True, False):
        recs = an.peaks(z, 250.0, flexible=flexible)
        assert (recs["status"] == 0).all()
        for w in range(b):
            zl = z[w].astype(np.complex128).tolist()
            want = ref_port.top_peaks_prominence(zl, 250.0) if flexible else ref_port.top_peaks_resolution(zl, 250.0)
            got = _dicts(recs[w], 250.0, n, flexible)
            assert [p["idx"] for p in got] == [p["idx"] for p in want], (n, flexible, w)
            for g, wt in zip(got, want):
                if flexible:
                    assert g["damping"] == wt["damping"] and g["q-factor"] == wt["q-factor"]
                    assert cases.isclose_rel(g["prominence"], wt["prominence"], 2e-6)
                assert abs(g["mag"] - wt["mag"]) <= 1e-4 + 1e-6 * abs(wt["mag"])   # MUFU sqrt: 1 ulp before round(., 4)


def test_f32_fast_kernels_equal_general_kernels(an):
    """Specialised fp32 kernels vs the general ones (apda_ctx_set_generic_only) on tone and noise windows."""
    import apda_fft_b200.synth as synth
    for n in (1024, 4096, 8192):
        tones = synth.fleet_windows(300, 128, n, dtype=np.float32)
        noise = np.stack([synth.noise_window(w, n) for w in range(32)]).astype(np.float32)
        for x, min_same in ((tones, 1.0), (noise, 0.9)):
            for flexible in (True, False):
                fast = an.analyze(x, 125.0, flexible=flexible)
                an.ctx.set_generic_only(True)
                try:
                    slow = an.analyze(x, 125.0, flexible=flexible)
                finally:
                    an.ctx.set_generic_only(False)
                same = [(fast[w]["count"] == slow[w]["count"]) and (fast[w]["pk"]["idx"] == slow[w]["pk"]["idx"]).all()
                        for w in range(x.shape[0])]
                assert np.mean(same) >= min_same, (n, flexible, np.mean(same))
                assert (fast["status"] == 0).all()


@pytest.mark.parametrize("log2n,n_samples", [(14, None), (15, 20000), (16, None), (18, 200001), (20, None)])
def test_fft_large_f64_bit_exact(log2n, n_samples, an):
    """K2 (multi-pass): fp64 spectra of N > 2^13 are bit-identical to the reference restatement, padding included."""
    n = 1 << log2n
    ns = n if n_samples is None else n_samples
    i = np.arange(ns, dtype=np.float64)
    rng = np.random.default_rng(log2n)
    x = np.round(0.5 * np.sin(2 * np.pi * 101.6 * i / n) + 0.3 * np.sin(2 * np.pi * 252.4 * i / n + 0.3)
                 + 0.2 * np.sin(2 * np.pi * 498.0 * i / n + 1.1) + 0.01 * rng.uniform(-1, 1, ns) + 0.25, 6)
    got = an.fft(x)[0]
    want = c_oracle.start_fft_batch(x)[0]
    assert got.shape == (n,)
    assert np.array_equal(got.view(np.float64), want.view(np.float64))
    if log2n <= 16:
        rec = an.analyze(x, 250.0, flexible=True)[0]
        assert _dicts(rec, 250.0, n, True) == c_oracle.peaks_prominence(want, 250.0)
        rec = an.analyze(x, 250.0, flexible=False)[0]
        assert _dicts(rec, 250.0, n, False) == c_oracle.peaks_resolution(want, 250.0)


def test_fft_large_f32_and_c2c(an):
    n = 1 << 17
    i = np.arange(n, dtype=np.float64)
    x = np.round(0.5 * np.sin(2 * np.pi * 1001.6 * i / n) + 0.3 * np.sin(2 * np.pi * 2520.4 * i / n + 0.3), 6)
    want = c_oracle.start_fft_batch(x)[0]
    got = an.fft(x.astype(np.float32))[0]
    assert np.abs(got.astype(np.complex128) - want).max() <= 3e-6 * np.abs(want).max()
    rec = an.analyze(x.astype(np.float32), 250.0, flexible=True)[0]
    assert [p["idx"] for p in _dicts(rec, 250.0, n, True)] == [p["idx"] for p in c_oracle.peaks_prominence(want, 250.0)]
    rng = np.random.default_rng(3)
    z = np.round(rng.standard_normal(1 << 15) + 1j * rng.standard_normal(1 << 15), 6)
    assert np.array_equal(an.fft_c2c(z)[0].view(np.float64), c_oracle.fft_c2c(z).view(np.float64))


@pytest.mark.parametrize("n_fft", [1024, 2048, 4096, 8192])
def test_f64_fast_kernel_bit_exact_incl_median_and_padding(n_fft, an):
    """Register-blocked fp64 K1: bit-identical to the C oracle on skewed / tied / padded / odd-length windows."""
    rng = np.random.default_rng(n_fft + 7)
    for n_samples in (n_fft, n_fft - 1, n_fft - 2, (3 * n_fft) // 4 + 1, n_fft // 2 + 1, n_fft // 2 + 2):
        rows = [np.round(np.exp(rng.standard_normal(n_samples)), 2),
                np.round(rng.standard_normal(n_samples) * 0.3 + 5.0, 3),
                (rng.random(n_samples) < 0.5).astype(np.float64),
                np.round(np.sin(np.arange(n_samples) * 0.05) + 0.2 * rng.standard_normal(n_samples), 6),
                np.zeros(n_samples), rng.standard_normal(n_samples)]
        x = np.stack(rows)
        got = an.fft(x, n_fft=n_fft)
        want = c_oracle.start_fft_batch(x, n_fft=n_fft)
        assert np.array_equal(got.view(np.float64), want.view(np.float64)), (n_fft, n_samples)
    import apda_fft_b200.synth as synth
    x = synth.fleet_windows(77, 64, n_fft)
    fast = an.fft(x)
    an.ctx.set_generic_only(True)
    try:
        slow = an.fft(x)
    finally:
        an.ctx.set_generic_only(False)
    assert np.array_equal(fast.view(np.float64), slow.view(np.float64))


@pytest.mark.parametrize("n", [1024, 2048, 4096, 8192])
def test_f64_fast_picker_equals_general_and_oracle(n, an):
    """Warp-per-window fp64 K3 vs the general CTA-per-window kernel: byte-identical records on tone, noise and
    heavy-tailed spectra (both pickers), and the oracle's dicts on a sample; covers zero / huge / tiny / subnormal bins
    (full-range hypot path) and the candidate-list overflow hand-over (noise windows)."""
    import apda_fft_b200.synth as synth
    rng = np.random.default_rng(n + 3)
    tones = an.fft(synth.fleet_windows(500, 96, n))
    noise = an.fft(np.stack([synth.noise_window(w, n) for w in range(24)]))
    spiky = _real_spiky_spectra(rng, 48, n).astype(np.complex128)
    spiky[:, : n // 2] *= np.exp(1j * rng.uniform(0, 6.28, (48, n // 2)))
    odd = spiky[:8].copy()
    odd[0, 5:40] = 0.0                       # exact zeros (glibc: ax >= ay / EPS shortcut)
    odd[1, 7] = 1e300 + 1e300j               # scaled-down branch
    odd[2, 9:200] *= 1e-300                  # scaled-up branch
    odd[3, 11] = 5e-324 + 3e-320j            # subnormals
    odd[4, 13] = 1.0 + 1e-20j                # ay negligible
    odd[5, 100:110] = 3.0 + 4.0j             # plateau: equal magnitudes are never peaks
    for z, check in ((tones, 16), (noise, 4), (spiky, 12), (odd, 8)):
        for flexible in (True, False):
            fast = an.peaks(z, 125.0, flexible=flexible)
            an.ctx.set_generic_only(True)
            try:
                slow = an.peaks(z, 125.0, flexible=flexible)
            finally:
                an.ctx.set_generic_only(False)
            assert fast.tobytes() == slow.tobytes(), (n, flexible)
            for w in range(check):
                zl = z[w].tolist()
                want = ref_port.top_peaks_prominence(zl, 125.0) if flexible else ref_port.top_peaks_resolution(zl, 125.0)
                assert _dicts(fast[w], 125.0, n, flexible) == want, (n, flexible, w)


def test_fft_large_tma_equals_plain_tail_passes(an):
    """K2 tail passes: the TMA-staged kernel and the plain-load kernel give the same bits (fp64 and fp32)."""
    rng = np.random.default_rng(11)
    for log2n in (14, 17, 21):
        x = np.round(rng.standard_normal(1 << log2n), 6)
        for dt in (np.float64, np.float32):
            a = an.fft(x.astype(dt))
            an.ctx.set_generic_only(True)
            try:
                b = an.fft(x.astype(dt))
            finally:
                an.ctx.set_generic_only(False)
            if dt == np.float64:
                assert np.array_equal(a.view(np.float64), b.view(np.float64)), log2n
            else:
                # generic_only also swaps the fp32 small-N kernels; at these sizes both runs use K2, so bits match too
                assert np.array_equal(a.view(np.float32), b.view(np.float32)), log2n


def test_peaks_large_multi_cta_vs_general_and_oracle(an):
    """K3 large form (n >= 2^16, chip-wide): same records as the one-CTA general kernel, and as the oracle at 2^16."""
    rng = np.random.default_rng(21)
    for log2n in (16, 18):
        n = 1 << log2n
        i = np.arange(n, dtype=np.float64)
        x = np.round(0.5 * np.sin(2 * np.pi * 1001.6 * i / n) + 0.3 * np.sin(2 * np.pi * 2520.4 * i / n + 0.3)
                     + 0.2 * np.sin(2 * np.pi * 4980.0 * i / n + 1.1) + 0.01 * rng.uniform(-1, 1, n), 6)
        spec = an.fft(x)
        noise = an.fft(np.round(rng.standard_normal(n), 6))
        for z in (spec, noise):
            for flexible in (True, False):
                for dt in (np.complex128, np.complex64):
                    fast = an.peaks(z.astype(dt), 250.0, flexible=flexible)
                    an.ctx.set_generic_only(True)
                    try:
                        slow = an.peaks(z.astype(dt), 250.0, flexible=flexible)
                    finally:
                        an.ctx.set_generic_only(False)
                    assert fast.tobytes() == slow.tobytes(), (log2n, flexible, dt)
        if log2n == 16:
            assert _dicts(an.peaks(spec, 250.0, flexible=True)[0], 250.0, n, True) == c_oracle.peaks_prominence(spec[0], 250.0)
            assert _dicts(an.peaks(spec, 250.0, flexible=False)[0], 250.0, n, False) == c_oracle.peaks_resolution(spec[0], 250.0)


@pytest.mark.parametrize("n", [1024, 2048, 4096, 8192])
def test_fused_kernel_matches_pipeline_and_oracle(n, an):
    """Fused window->record kernel (no spectrum in memory) vs the two-kernel pipeline and the oracle."""
    import apda_fft_b200
    import apda_fft_b200.synth as synth
    tones = synth.fleet_windows(1200, 96, n, dtype=np.float32)
    noise = np.stack([synth.noise_window(w, n) for w in range(32)]).astype(np.float32)
    padded = synth.fleet_windows(5, 16, n, dtype=np.float32)[:, : (3 * n) // 4 + 3]
    for x, min_same in ((tones, 1.0), (padded, 1.0), (noise, 0.9)):
        for flexible in (True, False):
            for center in (apda_fft_b200._cabi.CENTER_MEDIAN, apda_fft_b200._cabi.CENTER_MEAN):
                if center == apda_fft_b200._cabi.CENTER_MEAN and x.shape[1] != n:
                    continue
                fused = an.analyze_fused(x, 125.0, flexible=flexible, center=center)
                pipe = an.analyze(x, 125.0, flexible=flexible, center=center)
                assert (fused["status"] == 0).all()
                same = [(fused[w]["count"] == pipe[w]["count"]) and (fused[w]["pk"]["idx"] == pipe[w]["pk"]["idx"]).all()
                        for w in range(x.shape[0])]
                assert np.mean(same) >= min_same, (n, flexible, center, np.mean(same))
                live = (pipe["pk"]["idx"] >= 0) & (fused["pk"]["idx"] == pipe["pk"]["idx"])
                assert np.allclose(fused["pk"]["mag"][live], pipe["pk"]["mag"][live], rtol=2e-6)
    want = c_oracle.start_fft_batch(tones[:8].astype(np.float64))
    got = an.analyze_fused(tones[:8], 125.0, flexible=True)
    for w in range(8):
        assert [p["idx"] for p in _dicts(got[w], 125.0, n, True)] == [p["idx"] for p in c_oracle.peaks_prominence(want[w], 125.0)]


def test_wire16_decode_bit_exact_and_pipeline(golden, an):
    """Wire ingest: device decode == reference decode_samples + '%8.6f' + float() (fp64 bits), and the ragged pipeline
    on the decoded windows == the oracle on the same samples."""
    rows, firsts = [], []
    for wc in cases.WIRE_CASES:
        g = golden["wire"][wc["id"]]
        pay = cases.wire_payload(wc["seed"], wc["n"], wc.get("specials", True))
        samples, nv = an.decode_wire16(pay[None, :], wc["first_value"])
        assert int(nv[0]) == g["n_valid"]
        assert cases.sha16(samples[0, : nv[0]]) == g["sha"], wc["id"]
        if wc["n"] == 4096:
            rows.append(pay)
            firsts.append(wc["first_value"])
    # a ragged batch: three 4096-sample payloads (two of them lose samples to inf/nan), fp64 and fp32
    pay = np.stack(rows)
    fv = np.asarray(firsts)
    samples, nv = an.decode_wire16(pay, fv)
    for dtype, tol in (("f64", TOL64), ("f32", TOL32)):
        for flexible in (True, False):
            recs = an.analyze_wire16(pay, fv, 125.0, dtype=dtype, flexible=flexible)
            for w in range(pay.shape[0]):
                x = samples[w, : nv[w]]
                spec = c_oracle.start_fft_batch(x, n_fft=4096)[0]
                want = c_oracle.peaks_prominence(spec, 125.0) if flexible else c_oracle.peaks_resolution(spec, 125.0)
                got = _dicts(recs[w], 125.0, 4096, flexible)
                if dtype == "f64":
                    assert_peaks_close(got, want, tol, (w, flexible))
                else:
                    assert [p["idx"] for p in got][:2] == [p["idx"] for p in want][:2] or len(want) == 0
                assert recs[w]["status"] == 0


def test_ragged_batch_device_api(an):
    """apda_analyze_ragged_*_dev: per-window sample counts, including an empty window and one whose own padded length
    differs from the batch N (status bits 3 and 2)."""
    import ctypes
    import torch
    import apda_fft_b200.synth as synth
    from apda_fft_b200.records import record_dtype
    n = 4096
    counts = [4096, 4095, 3000, 2049, 4096, 0, 1500, 4096]
    full = synth.fleet_windows(60, len(counts), n)
    dev = torch.device("cuda:0")
    an.use_stream(torch.cuda.current_stream(dev).cuda_stream)
    try:
        for name, tdt, tol in (("f64", torch.float64, TOL64), ("f32", torch.float32, TOL32)):
            d_x = torch.as_tensor(full, device=dev).to(tdt).contiguous()
            d_nv = torch.tensor(counts, dtype=torch.int32, device=dev)
            d_rec = torch.zeros((len(counts), 128), dtype=torch.uint8, device=dev)
            an.ctx.call(f"apda_analyze_ragged_{name}_dev", ctypes.c_void_p(d_x.data_ptr()), ctypes.c_void_p(d_nv.data_ptr()),
                        n, n, len(counts), n, 0, 1, 125.0, ctypes.c_void_p(0), 4, 5, ctypes.c_void_p(0),
                        ctypes.c_void_p(d_rec.data_ptr()))
            torch.cuda.synchronize()
            recs = d_rec.cpu().numpy().view(record_dtype(5)).reshape(-1)
            for w, cnt in enumerate(counts):
                if cnt == 0:
                    assert recs[w]["status"] & 8 and recs[w]["count"] == 0
                    continue
                assert bool(recs[w]["status"] & 4) == (c_oracle.padded_len(cnt) != n), (w, cnt)
                want = c_oracle.peaks_prominence(c_oracle.start_fft_batch(full[w, :cnt], n_fft=n)[0], 125.0)
                got = _dicts(recs[w], 125.0, n, True)
                if name == "f64":
                    assert_peaks_close(got, want, tol, (w, cnt))
                else:
                    assert [p["idx"] for p in got] == [p["idx"] for p in want], (w, cnt)
    finally:
        an.use_stream(None)


def test_text_ingest_matches_load_sensor(golden, tmp_path, an):
    """Batched GPU log parser == the reference's load_sensor on clean, CRLF, one-line and nasty logs."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "apda-fft_b200"))
    from utils.load_data import load_sensor, load_sensors
    paths = []
    for lc in cases.LOG_CASES:
        text = cases.log_text(lc["seed"], lc["n"], lc["nasty"], lc.get("newline", "\n"), lc.get("per_line", 60))
        path = tmp_path / (lc["id"] + ".log")
        path.write_bytes(text.encode("utf-8"))
        paths.append(str(path))
    short = tmp_path / "short.log"
    short.write_text("a;b;1 Hz;X axis;\nNo;\n")
    paths.append(str(short))
    batch = load_sensors(paths)
    assert batch[-1] is None
    for lc, got in zip(cases.LOG_CASES, batch):
        g = golden["logs"][lc["id"]]
        want = load_sensor(paths[cases.LOG_CASES.index(lc)])
        if want is None:
            assert got is None
            continue
        assert got["metadata"] == want["metadata"] and got["summary"] == want["summary"]
        assert len(got["samples"]) == g["n_samples"] and cases.sha16(np.asarray(got["samples"])) == g["sha"], lc["id"]
    # the device parser alone (no host fallback): every piece it decides must equal float(); undecided ones raise the flag
    import ctypes
    pieces = ["0.5", "-1.25", "+3", ".125", "7.", "000.500", "-0.000000", "123456789.012345", "0.000001", "nan", "x1", "", " "]
    text = (";".join(pieces) + ";\n").encode()
    off = np.array([0, len(text)], dtype=np.int64)
    out = np.zeros((1, 64)); nv = np.zeros(1, dtype=np.int32); fl = np.zeros(1, dtype=np.int32)
    buf = np.frombuffer(text, dtype=np.uint8)
    p = ctypes.c_void_p
    an.ctx.call("apda_parse_samples_f64_host", p(buf.ctypes.data), p(off.ctypes.data), 1, 64, p(out.ctypes.data),
                p(nv.ctypes.data), p(fl.ctypes.data))
    assert fl[0] == 0 and out[0, : nv[0]].tolist() == [0.5, -1.25, 3.0, 0.125, 7.0, 0.5, -0.0, 123456789.012345, 1e-06]
    assert np.signbit(out[0, 6])


def _peer_worker(rank, world, port, tmp):
    """Six steps with DIFFERENT windows per step; the owner lags (it sleeps on its stream before consuming), so the
    producers run ahead as far as the flow control lets them.  Every step's table, snapshotted by the owner between
    wait() and release(), must equal the NCCL gather of that step's records - with a single table and no
    acknowledgement a fast producer would have overwritten rows the owner had not read yet."""
    import torch
    import torch.distributed as dist
    import apda_fft_b200
    from apda_fft_b200.fleet import PeerRecordTable, gather_records
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=dev)
    an = apda_fft_b200.Analyzer(rank)
    an.use_stream(torch.cuda.current_stream(dev).cuda_stream)
    per, n, steps = 3000, 4096, 6
    x = torch.empty((steps + 1, per, n), dtype=torch.float32, device=dev)
    spec = torch.empty((per, n, 2), dtype=torch.float32, device=dev)
    rec = torch.zeros((per, 128), dtype=torch.uint8, device=dev)
    for s in range(1, steps + 1):
        an.synth_device((s * world + rank) * per, per, n, "f32", x[s].data_ptr())
    table = PeerRecordTable(an.ctx, per, 128, dev)
    snaps = {}
    for step in range(1, steps + 1):
        ptr = table.begin(step)
        an.fft_device(x[step].data_ptr(), per, n, n, "f32", spec.data_ptr())
        an.peaks_device(spec.data_ptr(), per, n, "f32", 125.0, ptr)
        table.signal(step)
        if table.owner:
            torch.cuda._sleep(20_000_000)          # ~10 ms: the consumer is slower than the producers
            snaps[step] = table.wait(step).clone()
            table.release(step)
    table.complete()
    ok = True
    for step in range(1, steps + 1):
        an.fft_device(x[step].data_ptr(), per, n, n, "f32", spec.data_ptr())
        an.peaks_device(spec.data_ptr(), per, n, "f32", 125.0, rec.data_ptr())
        want = gather_records(rec, per * world, dst=0)
        if rank == 0:
            ok = ok and bool(torch.equal(snaps[step], want))
    if rank == 0:
        assert not table.timed_out()
        assert ok
        assert not torch.equal(snaps[1], snaps[2])      # the steps really carried different data
        open(os.path.join(tmp, "ok"), "w").write("1")
    dist.barrier()
    table.close()
    dist.destroy_process_group()


def test_peer_record_table_equals_nccl_gather(tmp_path):
    """N>1 on GPUs: K3 storing its records into rank 0's table over NVLink peer memory (CUDA IPC + device-side step
    counters, double-buffered with an owner->producer acknowledgement) gives the table an NCCL gather gives, byte for
    byte, on every one of several steps with different data.  Needs two GPUs (skipped on a single-GPU box; bench.py
    repeats the equality check as a hard failure on every multi-GPU run)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    port = 29700 + os.getpid() % 200
    mp.spawn(_peer_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert os.path.exists(os.path.join(str(tmp_path), "ok"))


def _outcome(fn, *args, **kw):
    try:
        return {"ok": fn(*args, **kw)}
    except Exception as exc:  # the shim raises the reference's exception types (SURVEY 8b)
        return {"error": type(exc).__name__}


def test_fuzz_small_windows_and_spectra_vs_oracle(an):
    """The adversarial inputs that pinned the oracle to the live reference (tests/cases.py: 400 windows of length
    1..256 with ties / plateaus / offsets, 300 hand-shaped spectra with k = 1..7) through the drop-in modules, i.e.
    the reference's own call signatures on the CUDA path: spectra equal element by element (fp64 bit-exact), peak
    lists equal objects, same exception types for degenerate sizes."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "apda-fft_b200"))
    from metrics.fft_iterativa import start_fft
    from utils.get_peak_prominence import get_top_peaks_prominence
    from utils.get_peak_resolution import get_top_peaks_resolution
    for x in cases.fuzz_inputs(20260101, 400):
        want = ref_port.start_fft(list(x), 125.0)
        got = start_fft(list(x), 125.0)
        assert len(got) == len(want) and all(complex(a) == complex(b) for a, b in zip(got, want)), x
        assert _outcome(get_top_peaks_prominence, got, 125.0) == _outcome(ref_port.top_peaks_prominence, list(want), 125.0), x
        assert _outcome(get_top_peaks_resolution, got, 125.0) == _outcome(ref_port.top_peaks_resolution, list(want), 125.0), x
    for spec, fs, k in cases.fuzz_spectra(7, 300):
        assert _outcome(get_top_peaks_prominence, list(spec), fs, k) == _outcome(ref_port.top_peaks_prominence, list(spec), fs, k)
        assert _outcome(get_top_peaks_resolution, list(spec), fs, k) == _outcome(ref_port.top_peaks_resolution, list(spec), fs, k)


def test_c_host_example_runs(tmp_path):
    """examples/analyze_host.c (plain C over the C ABI): three tones per window at the expected bins."""
    import subprocess
    from test_cabi_and_host import _build_c_example
    out = subprocess.check_output([_build_c_example(tmp_path)], text=True)
    rows = [r for r in out.splitlines() if r.startswith("window")]
    assert len(rows) == 8
    for w, row in enumerate(rows):
        assert f"window {w}: 3 peaks" in row and "idx 252" in row and "idx 498" in row and f"idx {round(101.6 + w)}" in row, row
    assert "multi: 2 contexts, table identical" in out      # apda_multi_analyze_f32_host from plain C


@pytest.mark.parametrize("n_samples", [1 << 16, (1 << 16) - 1, 50_001])
def test_large_window_median_adversarial(n_samples, an):
    """K2's median (two digit passes, bucket copy, one-CTA finish) on distributions that stress it: constant windows,
    three-level plateaus (the bucket is a third of the window), half the samples equal to the median, and middle
    values that sit in different top-16-bit buckets (the upper middle comes from the buckets above).  The centred
    spectrum must stay bit-identical to the C oracle, which takes the exact statistics.median."""
    rng = np.random.default_rng(n_samples)
    n = 1 << 16
    half = n_samples // 2
    rows = [np.full(n_samples, 0.731),
            rng.integers(-1, 2, n_samples).astype(np.float64),
            np.where(rng.random(n_samples) < 0.5, 0.25, np.round(rng.standard_normal(n_samples), 6)),
            np.concatenate([np.full(half, 0.99999), np.full(n_samples - half, 1.00001)]),
            np.concatenate([np.full(half, -2.5), np.full(n_samples - half, 3.0e5)]),
            np.round(np.exp(3.0 * rng.standard_normal(n_samples)), 6)]
    for r, x in enumerate(rows):
        x = rng.permutation(x)
        got = an.fft(x[None, :], n_fft=n)
        want = c_oracle.start_fft_batch(x[None, :], n_fft=n)
        assert np.array_equal(got.view(np.float64), want.view(np.float64)), (n_samples, r)
        x32 = x.astype(np.float32)
        got32 = an.fft(x32[None, :], n_fft=n)[0]
        centred = x32 - np.float32(np.median(x32))                   # exact in fp32: midpoint of two floats
        ref32 = np.fft.fft(np.concatenate([centred.astype(np.float64), np.zeros(n - n_samples)]))
        ref32[0] = 0
        scale = np.abs(ref32).max() + 1e-30
        assert np.abs(got32 - ref32).max() <= 2e-5 * scale + 1e-3, (n_samples, r)


@pytest.mark.parametrize("dtype", ["f32", "f64"])
def test_no_out_of_bounds_writes_guard_bands(dtype, an):
    """compute-sanitizer is not available on this pool, so: every output buffer (spectra, records) sits between guard
    bands that must come back untouched, for odd batch sizes (partly filled last CTA), every fast-path size, both pickers,
    padded windows, and a K2 size."""
    import torch
    dev = torch.device("cuda:0")
    an.use_stream(torch.cuda.current_stream(dev).cuda_stream)
    tdt = torch.float32 if dtype == "f32" else torch.float64
    s = 4 if dtype == "f32" else 8
    guard = 8192
    try:
        for n, b, n_samples in ((1024, 37, 1024), (2048, 5, 2001), (4096, 33, 4096), (8192, 3, 8192), (4096, 1, 3000),
                                (1 << 15, 2, 30000)):
            x = torch.randn((b, n_samples), dtype=tdt, device=dev).round(decimals=4)
            spec_raw = torch.full((guard + b * n * 2 * s + guard,), 0xA5, dtype=torch.uint8, device=dev)
            rec_raw = torch.full((guard + b * 128 + guard,), 0x5A, dtype=torch.uint8, device=dev)
            spec_ptr, rec_ptr = spec_raw.data_ptr() + guard, rec_raw.data_ptr() + guard
            for flexible in (True, False):
                an.fft_device(x.data_ptr(), b, n_samples, n, dtype, spec_ptr)
                an.peaks_device(spec_ptr, b, n, dtype, 125.0, rec_ptr, flexible=flexible, k=4 if flexible else 5)
                an.analyze_device(x.data_ptr(), b, n_samples, n, dtype, 125.0, rec_ptr, flexible=flexible,
                                  k=4 if flexible else 5, d_spec_ws=spec_ptr)
                if dtype == "f32" and n <= 8192:
                    an.analyze_fused_device(x.data_ptr(), b, n_samples, n, 125.0, rec_ptr, flexible=flexible,
                                            k=4 if flexible else 5)
            torch.cuda.synchronize()
            for raw, fill, what in ((spec_raw, 0xA5, "spectra"), (rec_raw, 0x5A, "records")):
                assert bool((raw[:guard] == fill).all()) and bool((raw[-guard:] == fill).all()), (n, b, what)
            recs = rec_raw[guard:-guard].cpu().numpy()
            assert (recs.view(np.int32).reshape(b, 32)[:, 0] <= 5).all()      # count fields are sane
    finally:
        an.ctx.set_stream(None)
