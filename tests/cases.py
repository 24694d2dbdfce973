"""Deterministic parity cases shared by tests/golden/make_golden.py (which runs the live reference)
and the test-suite (which replays the committed answers).  A case is a small JSON-able spec; the
samples are rebuilt from the spec, never stored."""
from __future__ import annotations

import hashlib
import math

import numpy as np

import apda_fft_b200.synth as synth


def sha16(arr) -> str:
    return hashlib.sha256(np.ascontiguousarray(arr, dtype="<f8").tobytes()).hexdigest()[:16]


def spectrum_sha16(spec) -> str:
    """spec: list/array of N complex (bin 0 may be int 0) -> sha256 of N x (re, im) little-endian doubles."""
    a = np.asarray([complex(v) for v in spec] if isinstance(spec, list) else spec, dtype=np.complex128)
    return hashlib.sha256(a.view(np.float64).astype("<f8").tobytes()).hexdigest()[:16]


def _lcg_uniform(seed: int, n: int) -> np.ndarray:
    s = seed & ((1 << 64) - 1)
    out = np.empty(n)
    for i in range(n):
        s = (s * 6364136223846793005 + 1442695040888963407) & ((1 << 64) - 1)
        out[i] = (s >> 11) / 9007199254740992.0
    return out


def build_samples(spec: dict):
    """-> (samples float64[n_samples], fs)"""
    kind = spec["kind"]
    fs = float(spec.get("fs", 125.0))
    if kind == "kat0":
        return np.asarray(synth.KAT0_INPUT, dtype=np.float64), 1.0
    if kind == "kat":
        x, fs = synth.kat_window(spec["name"])
        return x, fs
    if kind == "fleet":
        x = synth.fleet_window(spec["w"], spec["n"], on_bin=spec.get("on_bin", False))
    elif kind == "noise":
        x = synth.noise_window(spec["w"], spec["n"])
    elif kind == "tones":
        # explicit tones; optional dc offset and truncation (-> zero padding inside start_fft)
        n = spec["n"]
        i = np.arange(n, dtype=np.float64)
        x = np.zeros(n)
        for (c, a, ph) in spec["tones"]:
            x = x + a * np.sin(2.0 * np.pi * c * i / n + ph)
        x = x + spec.get("noise", 0.01) * (2.0 * _lcg_uniform(spec.get("seed", 1), n) - 1.0)
        x = np.round(x + spec.get("dc", 0.0), 6)
    elif kind == "const":
        x = np.full(spec["n"], float(spec["value"]))
    elif kind == "literal":
        x = np.asarray(spec["values"], dtype=np.float64)
    else:
        raise ValueError(kind)
    if "take" in spec:
        x = x[: spec["take"]]
    return np.ascontiguousarray(x, dtype=np.float64), fs


def mags_case(seed: int, n: int, style: str) -> np.ndarray:
    """Magnitude arrays for the helper-function goldens (plateaus/ties included on purpose)."""
    u = _lcg_uniform(seed, n)
    if style == "coarse":            # few distinct values -> equal neighbours, equal-height peaks
        return np.floor(u * 6.0)
    if style == "smooth":
        i = np.arange(n)
        return np.round(np.abs(np.sin(i * 0.37 + seed)) * 5.0 + u, 3)
    return np.round(u * 10.0, 6)


CASES = [
    {"id": "kat0", "kind": "kat0"},
    {"id": "katA", "kind": "kat", "name": "A"},
    {"id": "katB", "kind": "kat", "name": "B"},
    {"id": "katC", "kind": "kat", "name": "C"},
    {"id": "fleet4096_w0", "kind": "fleet", "n": 4096, "w": 0},
    {"id": "fleet4096_w0_onbin", "kind": "fleet", "n": 4096, "w": 0, "on_bin": True},
    {"id": "fleet4096_w999999", "kind": "fleet", "n": 4096, "w": 999999},
    {"id": "fleet4096_w3", "kind": "fleet", "n": 4096, "w": 3},
    {"id": "fleet8192_w7_onbin", "kind": "fleet", "n": 8192, "w": 7, "on_bin": True},
    {"id": "fleet8192_w11", "kind": "fleet", "n": 8192, "w": 11},
    {"id": "fleet1024_w1", "kind": "fleet", "n": 1024, "w": 1},
    {"id": "fleet2048_w5", "kind": "fleet", "n": 2048, "w": 5},
    {"id": "fleet512_w2", "kind": "fleet", "n": 512, "w": 2},
    {"id": "fleet256_w4", "kind": "fleet", "n": 256, "w": 4},
    {"id": "fleet16384_w9", "kind": "fleet", "n": 16384, "w": 9},
    {"id": "pad1000", "kind": "fleet", "n": 1024, "w": 21, "take": 1000},
    {"id": "pad3000", "kind": "fleet", "n": 4096, "w": 22, "take": 3000},
    {"id": "pad1025", "kind": "fleet", "n": 2048, "w": 23, "take": 1025},
    {"id": "pad_odd777", "kind": "fleet", "n": 1024, "w": 24, "take": 777},
    {"id": "dc_offset", "kind": "tones", "n": 2048, "tones": [[60.3, 0.02, 0.1], [170.0, 0.01, 0.7]],
     "noise": 0.0005, "dc": 1.0, "seed": 5, "fs": 62.5},
    {"id": "dc_offset_padded", "kind": "tones", "n": 2048, "tones": [[60.3, 0.02, 0.1], [170.0, 0.01, 0.7]],
     "noise": 0.0005, "dc": -0.98, "seed": 6, "fs": 62.5, "take": 1500},
    {"id": "hump_pair", "kind": "tones", "n": 4096, "tones": [[200.0, 0.5, 0.0], [204.5, 0.12, 0.4], [600.0, 0.3, 0.2]],
     "noise": 0.002, "seed": 9, "fs": 250.0},
    {"id": "close_pair", "kind": "tones", "n": 4096, "tones": [[300.0, 0.5, 0.0], [303.0, 0.45, 1.0], [306.0, 0.4, 2.0]],
     "noise": 0.002, "seed": 10, "fs": 500.0},
    {"id": "low_and_high_bins", "kind": "tones", "n": 4096, "tones": [[10.0, 0.5, 0.0], [40.0, 0.4, 0.0], [1500.0, 0.4, 0.3], [990.0, 0.3, 0.3]],
     "noise": 0.001, "seed": 11, "fs": 31.25},
    {"id": "six_tones", "kind": "tones", "n": 4096, "tones": [[100.0, 0.5, 0.0], [210.0, 0.45, 0.5], [330.0, 0.4, 1.0],
                                                             [470.0, 0.35, 1.5], [610.0, 0.3, 2.0], [800.0, 0.25, 2.5]],
     "noise": 0.002, "seed": 12, "fs": 125.0},
    {"id": "noise1024", "kind": "noise", "n": 1024, "w": 0},
    {"id": "noise4096", "kind": "noise", "n": 4096, "w": 1},
    {"id": "const64", "kind": "const", "n": 64, "value": 3.25},
    {"id": "n4", "kind": "literal", "values": [1.0, -2.0, 3.5, 0.25]},
    {"id": "n8_ramp", "kind": "literal", "values": [0.0, 1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 7.0]},
    {"id": "n16_spike", "kind": "literal", "values": [0.0] * 5 + [1.0] + [0.0] * 10},
    {"id": "n3_padded", "kind": "literal", "values": [1.0, 2.0, 4.0]},
    {"id": "n2", "kind": "literal", "values": [1.0, 2.0]},
    {"id": "n1", "kind": "literal", "values": [1.0]},
]



def build_spectrum(spec: dict):
    """Picker-only cases: a hand-shaped half spectrum (exact magnitudes: purely real or purely imaginary bins),
    mirrored into a length-n complex array.  -> (complex128[n], fs)"""
    n = spec["n"]
    half = n // 2
    mags = 1.0 + np.round(_lcg_uniform(spec.get("seed", 3), half), 3) * spec.get("floor", 1.0)
    for start, shape in spec["shapes"]:
        mags[start:start + len(shape)] = shape
    mags[0] = 0.0
    z = np.zeros(n, dtype=np.complex128)
    sign = np.where(np.arange(half) % 3 == 0, -1.0, 1.0)
    z[:half] = np.where(np.arange(half) % 2 == 0, mags * sign, 1j * mags * sign)
    z[half:] = 0.5          # never read by the pickers
    return z, float(spec.get("fs", 125.0))


SPECTRA = [
    # shoulder bump (idx 207) within 5 % of the main peak (idx 200) and prominence/mag < 0.1 -> "hump" rejected
    {"id": "hump_rejected", "n": 4096, "fs": 250.0, "shapes": [
        [196, [120.0, 300.0, 700.0, 760.0, 1000.0, 720.0, 500.0, 380.0, 300.0, 290.0, 280.0, 310.0, 250.0, 180.0, 120.0, 60.0]],
        [598, [200.0, 400.0, 500.0, 390.0, 150.0]]]},
    # same bump but tall enough relative to its valley to survive (ratio >= 0.1)
    {"id": "hump_kept", "n": 4096, "fs": 250.0, "shapes": [
        [196, [120.0, 300.0, 700.0, 760.0, 1000.0, 720.0, 500.0, 380.0, 300.0, 290.0, 270.0, 310.0, 250.0, 180.0, 120.0, 60.0]],
        [598, [200.0, 400.0, 500.0, 390.0, 150.0]]]},
    # equal magnitudes: the sort is stable on round(mag, 4) -> ascending idx among ties; plateau at 900/901 is no peak
    {"id": "ties_and_plateau", "n": 2048, "fs": 125.0, "shapes": [
        [99, [200.0, 600.0, 210.0]], [299, [190.0, 600.0, 220.0]], [499, [100.0, 600.00004, 100.0]],
        [699, [150.0, 599.99996, 150.0]], [899, [300.0, 800.0, 800.0, 300.0]]]},
    # wide peak (fails the 7 % damping gate) next to narrow ones; one peak below idx 15 (fails the 0.1 % side never, 7 % side yes)
    {"id": "damping_gate", "n": 4096, "fs": 125.0, "shapes": [
        [5, [300.0, 900.0, 320.0]],
        [300, [200.0, 420.0, 640.0, 860.0, 900.0, 870.0, 650.0, 400.0, 210.0]],
        [1200, [100.0, 700.0, 120.0]], [1900, [100.0, 650.0, 90.0]]]},
    # rigid picker: close neighbours fail Rs >= 1.5; zeroing radius grows with idx
    {"id": "rigid_close", "n": 4096, "fs": 500.0, "shapes": [
        [400, [300.0, 900.0, 650.0, 640.0, 880.0, 300.0]], [1000, [500.0, 700.0, 520.0]],
        [1018, [100.0, 690.0, 100.0]], [1025, [100.0, 680.0, 100.0]], [30, [100.0, 500.0, 100.0]]]},
]

def wire_payload(seed: int, n: int, specials: bool = True) -> np.ndarray:
    """uint8[2*n]: n random 16-bit wire samples (high byte first); with `specials` a few inf/nan/subnormal/zero words."""
    s = (seed * 2654435761 + 12345) & ((1 << 64) - 1)
    words = np.empty(n, dtype=np.uint16)
    for i in range(n):
        s = (s * 6364136223846793005 + 1442695040888963407) & ((1 << 64) - 1)
        w = (s >> 33) & 0xFFFF
        if ((w >> 10) & 31) == 31 and not (specials and i % 97 == 0):
            w &= 0xBFFF                       # keep ordinary words finite
        words[i] = w
    if specials and n >= 64:
        words[3] = 0x7C00      # +inf
        words[5] = 0xFC00      # "-inf" decodes to +inf
        words[9] = 0x7E01      # nan
        words[11] = 0x0000     # +0
        words[12] = 0x8000     # sign bit, zero mantissa -> +0.0
        words[13] = 0x0001     # smallest subnormal
        words[14] = 0x83FF     # largest negative subnormal
        words[15] = 0x3C00     # 1.0
        words[16] = 0xBC00     # -1.0
    out = np.empty(2 * n, dtype=np.uint8)
    out[0::2] = words >> 8
    out[1::2] = words & 0xFF
    return out


LOG_HEADER = "2_11_22_18_20_32;2 g;125.0 Hz;X axis;\nSynced;\n25.010;-0.0222;0.0110;0.9981;85.0;\n0.268262;-0.5;1.0;\n"

NASTY_PIECES = ["+1.5", ".5", "5.", "-0.000000", "00012.500", "1e3", "1E-2", "1_0", "nan", "inf", "-inf", "Infinity", "abc",
                "* MISSING PACKETS 3-4 *", " ", "1.2.3", "--1", "1-", "0.1234567890123456789", "123456789012345678",
                "0.0000000000000000000001", "\u0661\u0662", " 7.25 ", "+", ".", "-.", "9007199254740993", "1e400", "-1e-400",
                "0x10", "1,5", "\t-3.125\t"]


def log_text(seed: int, n: int, nasty: bool, newline: str = "\n", per_line: int = 60) -> str:
    """Text of one sensor .log: 4 header lines + n '%8.6f' samples (optionally sprinkled with nasty pieces)."""
    vals = np.round(np.sin(np.arange(n) * 0.37 + seed) * 1.7 + 0.3 * (2 * _lcg_uniform(seed + 77, n) - 1), 6)
    pieces = ["%8.6f" % v for v in vals]
    if nasty:
        for i, tok in enumerate(NASTY_PIECES):
            pieces.insert(min(len(pieces), 5 + 13 * i), tok)
    rows = [";".join(pieces[i:i + per_line]) + ";" for i in range(0, len(pieces), per_line)]
    return LOG_HEADER.replace("\n", newline) + newline.join(rows) + newline


LOG_CASES = [
    {"id": "log_clean_4096", "seed": 1, "n": 4096, "nasty": False},
    {"id": "log_nasty_1000", "seed": 2, "n": 1000, "nasty": True},
    {"id": "log_crlf_2048", "seed": 3, "n": 2048, "nasty": False, "newline": "\r\n", "per_line": 7},
    {"id": "log_short_0", "seed": 4, "n": 0, "nasty": False},
    {"id": "log_oneline_300", "seed": 5, "n": 300, "nasty": True, "per_line": 100000},
]


WIRE_CASES = [
    {"id": "wire_1024_base0", "seed": 1, "n": 1024, "first_value": 0.0},
    {"id": "wire_4096_basez", "seed": 2, "n": 4096, "first_value": 0.9981234},
    {"id": "wire_4096_neg", "seed": 3, "n": 4096, "first_value": -0.5000005},
    {"id": "wire_777_tiny", "seed": 4, "n": 777, "first_value": 1e-07},
    {"id": "wire_4096_clean", "seed": 5, "n": 4096, "first_value": 0.0123456, "specials": False},
]

# cases too small for the pickers (statistics errors) are listed with the expected exception text
K_VARIANTS = [("six_tones", 2), ("six_tones", 6), ("noise4096", 10), ("noise1024", 1), ("katB", 3)]


def approx_rel(a: float, b: float) -> float:
    if a == b:
        return 0.0
    return abs(a - b) / max(abs(a), abs(b), 1e-300)


def isclose_rel(a, b, tol):
    return approx_rel(float(a), float(b)) <= tol or (math.isnan(a) and math.isnan(b))


def fuzz_inputs(seed, count):
    """Deterministic adversarial inputs: ties, plateaus, odd lengths, DC offsets, spiky magnitude spectra."""
    rng = np.random.default_rng(seed)
    for i in range(count):
        n = int(rng.integers(1, 70)) if i % 3 else int(rng.choice([2, 3, 4, 7, 8, 16, 31, 32, 64, 100, 128, 200, 256]))
        kind = i % 4
        if kind == 0:
            x = np.round(rng.standard_normal(n), 1)                       # many ties
        elif kind == 1:
            x = np.round(np.sin(np.arange(n) * rng.uniform(0.1, 2.5)) + 0.05 * rng.standard_normal(n) + rng.uniform(-3, 3), 6)
        elif kind == 2:
            x = rng.integers(-3, 4, n).astype(np.float64)                 # plateaus, repeated medians
        else:
            x = np.round(np.exp(rng.standard_normal(n)), 3)               # skewed
        yield x.tolist()


def fuzz_spectra(seed, count):
    rng = np.random.default_rng(seed)
    for i in range(count):
        n = int(rng.choice([8, 16, 32, 64, 128, 256]))
        mags = np.round(np.exp(1.4 * rng.standard_normal(n)), int(rng.integers(0, 4)))   # rounded: equal neighbours occur
        mags[0] = 0.0
        phase = np.exp(1j * rng.uniform(0, 2 * np.pi, n)) if i % 2 else np.ones(n)
        yield (mags * phase).tolist(), float(rng.choice([31.25, 62.5, 125.0, 250.0, 500.0])), int(rng.integers(1, 8))
