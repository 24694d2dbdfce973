"""T0: the oracle (scalar port + C FFT) replays the committed goldens that were produced by the live reference.
CPU only.  tests/golden/make_golden.py --check re-derives the goldens where a checkout of the reference is at hand."""
import os
import statistics
import sys

import numpy as np
import pytest

import cases
from oracle import c_oracle, ref_port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(fn, *args):
    try:
        return {"ok": fn(*args)}
    except Exception as exc:
        return {"error": type(exc).__name__, "message": str(exc)}


@pytest.mark.parametrize("spec", cases.CASES, ids=[c["id"] for c in cases.CASES])
def test_port_and_c_oracle_match_golden(spec, golden):
    g = golden["cases"][spec["id"]]
    x, fs = cases.build_samples(spec)
    assert cases.sha16(x) == g["input_sha"]
    port = ref_port.start_fft(x.tolist(), fs)
    assert len(port) == g["n_fft"]
    assert cases.spectrum_sha16(port) == g["spectrum_sha"]
    assert port[0] == 0 and type(port[0]) is int
    c_spec = c_oracle.start_fft_batch(x)[0]
    assert cases.spectrum_sha16(c_spec) == g["spectrum_sha"]
    for i, (re, im) in g["bins"].items():
        assert complex(port[int(i)]) == complex(re, im)
    assert _run(ref_port.top_peaks_prominence, port, fs) == g["prominence"]
    assert _run(ref_port.top_peaks_resolution, port, fs) == g["resolution"]
    if g["n_fft"] >= 4:
        assert _run(c_oracle.peaks_prominence, c_spec, fs) == g["prominence"]
        assert _run(c_oracle.peaks_resolution, c_spec, fs) == g["resolution"]


def test_survey_known_answers(golden):
    """SURVEY.md Appendix B.1 digests (independently produced during the survey from the live reference)."""
    expect = {"katA": ("53d00f25f6dc7ef6", "8c5d9a4667584d98", [25, 63, 124]),
              "katB": ("edfc2022f3cda128", "6fc481ac7e7bcece", [102, 252, 498]),
              "katC": ("b81ccf581724a8bb", "94d3bcbf65436df0", [203, 505, 996])}
    for cid, (in_sha, sp_sha, idx) in expect.items():
        g = golden["cases"][cid]
        assert (g["input_sha"], g["spectrum_sha"]) == (in_sha, sp_sha)
        assert [p["idx"] for p in g["prominence"]["ok"]] == idx
        assert [p["idx"] for p in g["resolution"]["ok"]] == idx
    katb = golden["cases"]["katB"]["prominence"]["ok"][0]
    assert (katb["freq"], katb["mag"], katb["prominence"], katb["damping"], katb["q-factor"]) == \
        (3.1128, 772.0513, 772.0478456461883, 0.98, 51.0)
    assert ref_port.start_fft([-21, 16, -11, 26, -1, -28, 9, -18], 1.0)[1] == (-19.999999999999993 - 42.22539674441618j)
    assert [p["idx"] for p in golden["cases"]["fleet4096_w999999"]["resolution"]["ok"]] == [127, 284, 450, 123, 131]


@pytest.mark.parametrize("spec", cases.SPECTRA, ids=[c["id"] for c in cases.SPECTRA])
def test_picker_only_spectra(spec, golden):
    g = golden["spectra"][spec["id"]]
    z, fs = cases.build_spectrum(spec)
    for k in (4, 5, 12):
        assert _run(ref_port.top_peaks_prominence, z.tolist(), fs, k) == g[f"prominence_k{k}"]
        assert _run(ref_port.top_peaks_resolution, z.tolist(), fs, k) == g[f"resolution_k{k}"]


def test_k_variants(golden):
    by_id = {c["id"]: c for c in cases.CASES}
    for row in golden["k_variants"]:
        x, fs = cases.build_samples(by_id[row["case"]])
        spec = c_oracle.start_fft_batch(x)[0]
        assert _run(c_oracle.peaks_prominence, spec, fs, row["k"]) == row["prominence"]
        assert _run(c_oracle.peaks_resolution, spec, fs, row["k"]) == row["resolution"]


def test_helper_goldens(golden):
    for blk in golden["helpers"]:
        mags = cases.mags_case(blk["seed"], blk["n"], blk["style"]).tolist()
        for row in blk["rows"]:
            j = row["j"]
            assert ref_port.prominence_of(mags, j) == row["prominence"]
            assert ref_port.half_power_width(mags, row["prominence"], j, blk["fs"], blk["n_fft"]) == row["width_hz"]
            assert ref_port.half_height_bins(mags, j) == row["whm"]
            assert ref_port.resolution_between(mags, j, row["other"]) == row["rs"]


def test_pad_and_empty(golden):
    for n, padded in golden["pad"].items():
        assert len(ref_port.pad_to_pow2([1.5] * int(n))) == padded
        assert c_oracle.padded_len(int(n)) == max(padded, 1)
    assert ref_port.start_fft([], 1.0) == [0]
    assert ref_port.center_on_median([]) == []
    with pytest.raises(statistics.StatisticsError):
        ref_port.top_peaks_prominence([0, 1 + 1j], 1.0)


def test_c_oracle_batch_equals_rowwise():
    import apda_fft_b200.synth as synth
    x = synth.fleet_windows(100, 8, 1024)
    spec = c_oracle.start_fft_batch(x)
    for r in range(8):
        assert np.array_equal(spec[r].view(np.float64), c_oracle.start_fft_batch(x[r])[0].view(np.float64))
        assert cases.spectrum_sha16(ref_port.start_fft(x[r].tolist(), 125.0)) == cases.spectrum_sha16(spec[r])
    z = np.round(np.random.default_rng(0).standard_normal(64) + 1j * np.random.default_rng(0).standard_normal(64), 6)
    assert cases.spectrum_sha16(c_oracle.fft_c2c(z)) == cases.spectrum_sha16(ref_port.dit_radix2(z.tolist()))


def test_wire_decode_port_matches_golden(golden):
    for wc in cases.WIRE_CASES:
        g = golden["wire"][wc["id"]]
        pay = cases.wire_payload(wc["seed"], wc["n"], wc.get("specials", True))
        loaded = ref_port.wire_samples_as_loaded(pay.tolist(), wc["first_value"])
        assert len(loaded) == g["n_valid"] and cases.sha16(np.asarray(loaded)) == g["sha"]
        assert loaded[:6] == g["head"]
        assert ref_port.decode_wire_samples_text(pay.tolist(), wc["first_value"])[:6] == g["text_head"]


def test_log_parsing_port_and_split(golden, tmp_path):
    import io
    sys.path.insert(0, os.path.join(ROOT, "apda-fft_b200"))
    from utils.load_data import load_sensor, split_log
    for lc in cases.LOG_CASES:
        g = golden["logs"][lc["id"]]
        text = cases.log_text(lc["seed"], lc["n"], lc["nasty"], lc.get("newline", "\n"), lc.get("per_line", 60))
        lines = io.StringIO(text, newline=None).readlines()
        got = ref_port.parse_log_sample_lines(lines[4:])
        assert len(got) == g["n_samples"] and cases.sha16(np.asarray(got)) == g["sha"] and got[-4:] == g["tail"]
        path = tmp_path / (lc["id"] + ".log")
        path.write_bytes(text.encode("utf-8"))
        mine = load_sensor(str(path))
        assert mine["samples"] == got and mine["metadata"]["fs"] == g["fs"] and mine["metadata"]["axis"] == g["axis"]
        parts = split_log(text.encode("utf-8"))
        if lc["n"] == 0:
            assert parts is None or ref_port.parse_log_sample_lines(
                io.StringIO(parts[1].decode(), newline=None).readlines()) == []
        else:
            rows = io.StringIO(parts[1].decode("utf-8"), newline=None).readlines()
            assert parts[0] == lines[:4] and ref_port.parse_log_sample_lines(rows) == got
