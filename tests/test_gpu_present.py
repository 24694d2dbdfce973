"""apda_present_{dev,host} and apda_fleet_jsonl_{dev,host}: the reference's presentation of record tables made on the
device.  Columns are held bit for bit (NaN-aware) to records.prominence_dicts / resolution_dicts, text byte for byte to
records.write_fleet_jsonl, which stay the oracle."""
import ctypes
import json
import os

import numpy as np
import pytest

from apda_fft_b200.records import prominence_dicts, record_dtype, resolution_dicts, write_fleet_jsonl

pytestmark = pytest.mark.gpu

_p = ctypes.c_void_p
SENT = 0xA5
GUARD = 4096
RATES = np.array([125.0, 100 / 3, 1e-3, 1e6, 0.7, 3200.0])
COLS = ("idx", "freq", "mag", "prominence", "damping", "q_factor")


@pytest.fixture(scope="module")
def an():
    import torch
    import apda_fft_b200
    a = apda_fft_b200.Analyzer(0)
    a.use_stream(torch.cuda.current_stream(torch.device("cuda:0")).cuda_stream)
    yield a
    a.use_stream(None)


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


def want_columns(recs, fs, n, flexible, k):
    b = len(recs)
    fs_col = np.broadcast_to(np.asarray(fs, dtype=np.float64), (b,))
    out = {c: np.full((b, k), np.nan) for c in COLS}
    out["idx"] = np.full((b, k), -1, dtype=np.int32)
    conv = prominence_dicts if flexible else resolution_dicts
    for w in range(b):
        for j, pk in enumerate(conv(recs[w], float(fs_col[w]), n)[:k]):
            out["idx"][w, j] = pk["idx"]
            out["freq"][w, j] = pk["freq"]
            out["mag"][w, j] = pk["mag"]
            if flexible:
                out["prominence"][w, j] = pk["prominence"]
                out["damping"][w, j] = pk["damping"]
                out["q_factor"][w, j] = pk["q-factor"]
    return out


def want_jsonl(tmp_path, recs, fs, n, flexible, k, first_window):
    path = os.path.join(tmp_path, "want.jsonl")
    write_fleet_jsonl(path, recs, fs, n, flexible, k, first_window)
    with open(path, "rb") as fh:
        return fh.read()


def same_bits(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64))


def check_columns(got, want, flexible):
    assert set(got) == {"idx", "freq", "mag"} | ({"prominence", "damping", "q_factor"} if flexible else set())
    assert np.array_equal(got["idx"], want["idx"])
    for c in got:
        if c != "idx":
            assert same_bits(got[c], want[c]), (c, np.argwhere(got[c].view(np.uint64) != want[c].view(np.uint64))[:5])


def windows(b, n, seed):
    """[b, n] float64: 24 tones at random bins and amplitudes plus noise."""
    rng = np.random.default_rng(seed)
    i = np.arange(n)[None, :]
    x = rng.normal(0, 0.05, size=(b, n))
    for _ in range(24):
        f = rng.uniform(3, n // 2 - 3, size=(b, 1))
        x += rng.uniform(0.2, 3.0, size=(b, 1)) * np.cos(2 * np.pi * f * i / n + rng.uniform(0, 6.3, size=(b, 1)))
    return x


# ---------------------------------------------------------------------------------------------------------------
# records made by the real routes
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1024, 2048, 4096, 8192, 16384, 65536])
@pytest.mark.parametrize("cap", [5, 16])
@pytest.mark.parametrize("flexible", [True, False])
@pytest.mark.parametrize("dtype", ["f32", "f64"])
def test_real_records(an, tmp_path, dtype, flexible, cap, n):
    b = 40 if n <= 16384 else 12
    x = windows(b, n, seed=n + cap).astype(np.float32 if dtype == "f32" else np.float64)
    fs = RATES[np.arange(b) % len(RATES)] if cap == 16 else 125.0
    recs = an.analyze(x, fs, flexible=flexible, k=cap, n_fft=n, rec_cap=cap)
    assert (recs["count"] > 0).any()                  # full slots are covered by the crafted tables below
    recs["count"][3] = 0                              # an empty record ...
    recs["pk"]["idx"][3] = -1
    recs["status"][5] = 4                             # ... and records the pipeline flagged
    recs["status"][7] = 16 | 8
    first = 2 ** 31 + 17 if cap == 16 else 0
    for k in range(1, cap + 1):
        check_columns(an.present(recs, fs, n, flexible=flexible, k=k), want_columns(recs, fs, n, flexible, k), flexible)
        assert an.fleet_jsonl(recs, fs, n, flexible=flexible, k=k, first_window=first) == \
            want_jsonl(tmp_path, recs, fs, n, flexible, k, first)


# ---------------------------------------------------------------------------------------------------------------
# crafted tables over the rounding and formatting domain
# ---------------------------------------------------------------------------------------------------------------
def domain_values():
    v = [0.0, -0.0, 1.0, -1.0, 2.0 ** 53, 1e16, 1e16 + 2, 9999999999999998.0, 1e-4, 9.999999999999999e-05, 1e-5,
         5e-324, 2.2250738585072014e-308, 2.225073858507201e-308, 1.7976931348623157e308, -1.7976931348623157e308,
         6857196096582392 / 1e4, 685719609658.2393, 0.03125, 0.015625, 2.675, 1.0005, 1e22, 1e23, 123456789.0]
    v += [k / 32 for k in range(-70, 70)] + [k / 64 for k in range(0, 200)] + [k / 1024 for k in range(0, 90)]
    v += [2.0 ** e for e in range(-1074, 1024, 7)] + [10.0 ** e for e in range(-323, 309, 3)]
    for d in (2, 4):                                 # around 2^53 / 10^d, where round() stops dividing
        c = 2.0 ** 53 / 10 ** d
        v += list(np.nextafter(c, np.inf) * np.ones(1)) + [np.nextafter(c, 0.0), c, c * (1 + 2 ** -40), c * (1 - 2 ** -40)]
        v += [(2 ** 53 - j) / 10 ** d for j in range(1, 6)] + [(2 ** 53 + j) / 10 ** d for j in range(0, 6, 2)]
    rng = np.random.default_rng(5)
    v += list(rng.integers(1, 10 ** 6, 200) / 10 ** rng.integers(0, 8, 200))   # short decimals
    v += list(rng.integers(0, 10 ** 9, 100).astype(np.float64))                # integral values
    v += [float(x) for x in np.nextafter(np.array([1e-4, 1e16, 0.5, 0.005]), [0, np.inf, 1, 0])]
    return np.array(v, dtype=np.float64)


def crafted_records(values, cap, seed):
    """Records whose magnitudes run over `values`; idx and width_bins 1..64 (q = idx / width: ties of round(q, 2))."""
    rng = np.random.default_rng(seed)
    b = (len(values) + cap - 1) // cap
    mags = np.resize(values, b * cap).reshape(b, cap)
    recs = np.zeros(b, dtype=record_dtype(cap))
    recs["count"] = rng.integers(0, cap + 1, size=b)
    recs["count"][:2] = cap
    recs["status"] = rng.choice([0, 0, 0, 1, 4, 8, 16], size=b)
    recs["pk"]["idx"] = rng.integers(1, 65, size=(b, cap))
    recs["pk"]["width_bins"] = rng.integers(1, 65, size=(b, cap))
    recs["pk"]["mag"] = mags
    recs["pk"]["prominence"] = np.roll(mags, 1)
    return recs


@pytest.mark.parametrize("flexible", [True, False])
def test_crafted_domain(an, tmp_path, flexible):
    vals = domain_values()
    recs = crafted_records(vals, 16, seed=1)
    b, n = len(recs), 4096
    for fs in (125.0, np.resize(np.concatenate([RATES, [1e300, 3e-310, 1.0 / 3]]), b)):
        for k in (1, 4, 16):
            check_columns(an.present(recs, fs, n, flexible=flexible, k=k), want_columns(recs, fs, n, flexible, k),
                          flexible)
            assert an.fleet_jsonl(recs, fs, n, flexible=flexible, k=k, first_window=2 ** 40) == \
                want_jsonl(tmp_path, recs, fs, n, flexible, k, 2 ** 40)
    # frequencies over the same domain: idx 1 and fs = n * v give df = fn = v (exact)
    recs["pk"]["idx"] = 1
    recs["pk"]["width_bins"] = 1
    fs = np.abs(vals[:b]) * n
    fs[~np.isfinite(fs) | (fs == 0)] = 1.0
    check_columns(an.present(recs, fs, n, flexible=flexible), want_columns(recs, fs, n, flexible, 16), flexible)
    assert an.fleet_jsonl(recs, fs, n, flexible=flexible, k=16) == want_jsonl(tmp_path, recs, fs, n, flexible, 16, 0)


def test_non_finite_magnitudes(an, tmp_path):
    recs = crafted_records(np.array([np.nan, np.inf, -np.inf, 1.5, -np.nan, 0.0]), 5, seed=2)
    recs["count"] = 5
    for flexible in (True, False):
        check_columns(an.present(recs, 125.0, 1024, flexible=flexible), want_columns(recs, 125.0, 1024, flexible, 5),
                      flexible)
        assert an.fleet_jsonl(recs, 125.0, 1024, flexible=flexible, k=5) == \
            want_jsonl(tmp_path, recs, 125.0, 1024, flexible, 5, 0)


def test_random_bit_patterns_repr(an, tmp_path):
    """10^7 random finite and non-finite bit patterns as the rigid picker's raw magnitudes: each printed as repr()."""
    cap, n = 16, 1024
    b = 10 ** 7 // cap
    rng = np.random.default_rng(11)
    mags = rng.integers(0, 2 ** 64, size=(b, cap), dtype=np.uint64).view(np.float64)
    recs = np.zeros(b, dtype=record_dtype(cap))
    recs["count"] = cap
    recs["pk"]["idx"] = np.arange(1, cap + 1)
    recs["pk"]["mag"] = mags
    got = an.fleet_jsonl(recs, float(n), n, flexible=False, k=cap)
    freqs = [float(i) for i in range(1, cap + 1)]
    want = "".join(json.dumps({"window": w, "fft_freqs": freqs, "fft_mags": row}) + "\n"
                   for w, row in enumerate(mags.tolist())).encode()
    assert got == want
    head = want_jsonl(tmp_path, recs[:20000], float(n), n, False, cap, 0)    # the text as the oracle writes it
    assert got[:len(head)] == head
    cols = an.present(recs, float(n), n, flexible=False)
    assert same_bits(cols["mag"], mags)


# ---------------------------------------------------------------------------------------------------------------
# device entry points, buffers, errors
# ---------------------------------------------------------------------------------------------------------------
def test_device_matches_host_and_stays_in_bounds(an):
    import torch
    cap, n, k = 16, 4096, 7
    recs = crafted_records(domain_values(), cap, seed=3)
    b = len(recs)
    fs = np.resize(RATES, b)
    d_rec = Guarded(recs.nbytes, recs)
    d_fs = torch.from_numpy(fs).cuda()
    for flexible in (True, False):
        want = an.present(recs, fs, n, flexible=flexible, k=k)
        bufs = {c: Guarded(b * k * (4 if c == "idx" else 8)) for c in COLS}
        an.present_device(d_rec.ptr, b, cap, n, 0.0, k, bufs["idx"].ptr, bufs["freq"].ptr, bufs["mag"].ptr,
                          bufs["prominence"].ptr, bufs["damping"].ptr, bufs["q_factor"].ptr, flexible=flexible,
                          d_fs=d_fs.data_ptr())
        got = {c: bufs[c].bytes().view(np.int32 if c == "idx" else np.float64).reshape(b, k) for c in COLS}
        assert np.array_equal(got["idx"], want["idx"])
        for c in COLS[1:]:
            assert same_bits(got[c], want[c] if c in want else np.full((b, k), np.nan)), c
        # a NULL column is not written
        only = Guarded(b * k * 8)
        an.present_device(d_rec.ptr, b, cap, n, 0.0, k, d_mag=only.ptr, flexible=flexible, d_fs=d_fs.data_ptr())
        assert same_bits(only.bytes().view(np.float64).reshape(b, k), want["mag"])

        text_want = an.fleet_jsonl(recs, fs, n, flexible=flexible, k=k, first_window=2 ** 33)
        cap_bytes = b * (64 + 52 * k)
        text = Guarded(cap_bytes)
        off = Guarded((b + 1) * 8)
        an.fleet_jsonl_device(d_rec.ptr, b, cap, n, 0.0, text.ptr, cap_bytes, off.ptr, flexible=flexible, k=k,
                              first_window=2 ** 33, d_fs=d_fs.data_ptr())
        offsets = off.bytes().view(np.int64)
        t = text.bytes()
        assert offsets[0] == 0 and offsets[-1] == len(text_want)
        assert t[:offsets[-1]].tobytes() == text_want
        assert (t[offsets[-1]:] == SENT).all()
        rows = text_want.split(b"\n")[:-1]
        assert np.array_equal(np.diff(offsets), [len(r) + 1 for r in rows])


def test_text_cap_too_small(an):
    from apda_fft_b200 import _cabi
    cap, n, k = 5, 1024, 4
    recs = crafted_records(domain_values()[:400], cap, seed=4)
    b = len(recs)
    exact = len(an.fleet_jsonl(recs, 125.0, n, k=k))
    d_rec = Guarded(recs.nbytes, recs)
    bound = b * _cabi.jsonl_row_bytes(k)
    text, off = Guarded(bound), Guarded((b + 1) * 8)
    with pytest.raises(ValueError):                 # _dev needs the bound of every row
        an.fleet_jsonl_device(d_rec.ptr, b, cap, n, 125.0, text.ptr, bound - 1, off.ptr, k=k)
    assert (text.bytes() == SENT).all() and (off.bytes() == SENT).all()
    # _host needs the exact size; nothing past text_cap is written
    h_text = np.full(exact + GUARD, SENT, dtype=np.uint8)
    h_off = np.zeros(b + 1, dtype=np.int64)
    for short in (exact - 1, exact // 2, 0):
        with pytest.raises(ValueError):
            an.ctx.call("apda_fleet_jsonl_host", _p(recs.ctypes.data), cap, b, n, 125.0, _p(0), 1, k, 0,
                        _p(h_text.ctypes.data), short, _p(h_off.ctypes.data))
        assert (h_text[short:] == SENT).all()
    an.ctx.call("apda_fleet_jsonl_host", _p(recs.ctypes.data), cap, b, n, 125.0, _p(0), 1, k, 0,
                _p(h_text.ctypes.data), exact, _p(h_off.ctypes.data))
    assert h_off[-1] == exact and (h_text[exact:] == SENT).all()


def test_argument_errors_and_empty_batch(an):
    import torch
    cap, n, k, b = 5, 1024, 4, 8
    recs = np.zeros(b, dtype=record_dtype(cap))
    d_rec = Guarded(recs.nbytes + 8, np.zeros(recs.nbytes + 8, dtype=np.uint8))
    col = Guarded(b * k * 8)
    text, off = Guarded(b * (64 + 52 * k)), Guarded((b + 1) * 8)
    pres = [_p(d_rec.ptr), cap, b, n, 125.0, _p(0), 1, k, _p(0), _p(col.ptr), _p(0), _p(0), _p(0), _p(0)]
    jsonl = [_p(d_rec.ptr), cap, b, n, 125.0, _p(0), 1, k, 0, _p(text.ptr), text.n, _p(off.ptr)]

    def bad(name, ok, i, v):
        a = list(ok)
        a[i] = v
        with pytest.raises(ValueError):
            an.ctx.call(name, *a)
    for name, ok in (("apda_present_dev", pres), ("apda_fleet_jsonl_dev", jsonl)):
        bad(name, ok, 0, _p(0))                     # records NULL
        bad(name, ok, 0, _p(d_rec.ptr + 4))         # records misaligned
        bad(name, ok, 1, 0)                         # rec_cap < 1
        bad(name, ok, 1, 10_000)                    # rec_cap beyond max(64, n/8 + 8)
        bad(name, ok, 7, 0)                         # k < 1
        bad(name, ok, 7, cap + 1)                   # k > rec_cap
        bad(name, ok, 3, 3)                         # n not a power of two
        bad(name, ok, 3, 2)                         # n < 4
        bad(name, ok, 2, -1)                        # batch < 0
    bad("apda_fleet_jsonl_dev", jsonl, 8, -1)       # first_window < 0
    bad("apda_fleet_jsonl_dev", jsonl, 9, _p(0))    # text NULL
    bad("apda_fleet_jsonl_dev", jsonl, 11, _p(0))   # offsets NULL
    h = np.zeros(b + 1, dtype=np.int64)
    with pytest.raises(ValueError):
        an.ctx.call("apda_fleet_jsonl_host", _p(0), cap, b, n, 125.0, _p(0), 1, k, 0, _p(h.ctypes.data), 100,
                    _p(h.ctypes.data))
    with pytest.raises(ValueError):
        an.ctx.call("apda_present_host", _p(0), cap, b, n, 125.0, _p(0), 1, k, _p(0), _p(0), _p(0), _p(0), _p(0),
                    _p(0))
    c0 = an.launch_count()                          # batch 0: nothing is launched or written
    a = list(pres)
    a[2] = 0
    an.ctx.call("apda_present_dev", *a)
    a = list(jsonl)
    a[2] = 0
    an.ctx.call("apda_fleet_jsonl_dev", *a)
    assert an.launch_count() == c0
    assert (col.bytes() == SENT).all() and (text.bytes() == SENT).all() and (off.bytes() == SENT).all()
    assert an.fleet_jsonl(recs[:0], 125.0, n) == b""
    assert all(v.shape == (0, cap) for v in an.present(recs[:0], 125.0, n).values())
    torch.cuda.synchronize()


def test_dev_calls_do_not_synchronise(an):
    """The _dev calls return while a long kernel queued in front of them on the same stream still runs."""
    import torch
    cap, n, k, b = 5, 4096, 4, 1 << 16
    recs = crafted_records(domain_values(), cap, seed=6)
    recs = np.resize(recs, b)
    d_rec = torch.from_numpy(recs.view(np.uint8)).cuda()
    cols = torch.empty((b, k), dtype=torch.float64, device="cuda:0")
    text = torch.empty(b * (64 + 52 * k), dtype=torch.uint8, device="cuda:0")
    off = torch.empty(b + 1, dtype=torch.int64, device="cuda:0")
    # warm the scratch so no call has to grow it
    an.fleet_jsonl_device(d_rec.data_ptr(), b, cap, n, 125.0, text.data_ptr(), text.numel(), off.data_ptr(), k=k)
    torch.cuda.synchronize()
    torch.cuda._sleep(2_000_000_000)                # ~1 s of GPU clock cycles in front of the calls
    done = torch.cuda.Event()
    an.present_device(d_rec.data_ptr(), b, cap, n, 125.0, k, d_freq=cols.data_ptr())
    an.fleet_jsonl_device(d_rec.data_ptr(), b, cap, n, 125.0, text.data_ptr(), text.numel(), off.data_ptr(), k=k)
    done.record()
    assert not done.query()
    torch.cuda.synchronize()
    want = an.fleet_jsonl(recs, 125.0, n, k=k)
    assert bytes(text[:int(off[-1])].cpu().numpy()) == want
    assert same_bits(cols.cpu().numpy(), an.present(recs, 125.0, n, k=k)["freq"])
