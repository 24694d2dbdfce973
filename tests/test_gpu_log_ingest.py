"""Whole sensor .log files -> records: apda_analyze_logs_{f64,f32}_host and Analyzer.analyze_logs.

  1. the Python API on a corpus of logs (LOG_CASES plus LF / CRLF / CR-only line ends, marker lines, nan / inf / blank
     pieces, with and without trailing ';', per-file rates, "125.0  Hz" spacing, a long and a non-ASCII header, a rate
     and a sample in exponent form, an empty sample region, short and over-long files, a 4-line file): metas equal
     load_sensor's, records equal apda_analyze_ragged_*_dev on load_sensor's samples (and Analyzer.analyze for files
     that pad to N, and the oracle's pickers in fp64), for both pickers, k = 1..5 and a wider record;
  2. the raw C call with no host fallback: flags, record statuses, h_fs (bit-equal to float()), h_n_valid, h_head;
  3. more files than three chunks hold and than there are reader threads: order, a repeated call, no thread left over;
  4. argument errors.
"""
import ctypes
import os
import struct
import sys

import numpy as np
import pytest

import cases
from oracle import c_oracle

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "apda-fft_b200"))
from utils.load_data import load_sensor  # noqa: E402

_p = ctypes.c_void_p
N = 4096
HEAD = 1024
EMPTY_SLOT = struct.pack("<iidd", -1, 0, 0.0, 0.0)
JUNK = ["nan", "inf", "-inf", "", " ", "* MISSING PACKETS 3-4 *", "abc", "Infinity"]


@pytest.fixture(scope="module")
def an():
    import apda_fft_b200
    return apda_fft_b200.Analyzer(0)


def rec_dtype(cap):
    from apda_fft_b200.records import record_dtype
    return record_dtype(cap)


def empty_record(cap, status):
    return struct.pack("<ii", 0, status) + EMPTY_SLOT * cap


def header(rate="125.0 Hz", nl="\n"):
    return cases.LOG_HEADER.replace("125.0 Hz", rate).replace("\n", nl)


def body(seed, n, nl="\n", per_line=60, extra=(), trailing=True):
    vals = np.round(np.sin(np.arange(n) * 0.37 + seed) * 1.7 + 0.4 * np.cos(np.arange(n) * 2.3 + 0.1 * seed), 6)
    pieces = ["%8.6f" % v for v in vals]
    for i, tok in enumerate(extra):
        pieces.insert(min(len(pieces), 7 + 31 * i), tok)
    rows = [";".join(pieces[i:i + per_line]) + (";" if trailing else "") for i in range(0, len(pieces), per_line)]
    return nl.join(rows) + (nl if trailing else "")


def corpus():
    """(name, bytes, device flag) of every test log; analyze_logs must reproduce load_sensor on each."""
    files = []
    for lc in cases.LOG_CASES:
        text = cases.log_text(lc["seed"], lc["n"], lc["nasty"], lc.get("newline", "\n"), lc.get("per_line", 60))
        files.append((lc["id"], text.encode(), 1 if lc["nasty"] else 0))
    rates = ["31.25 Hz", "62.5 Hz", "125 Hz", "250.0 Hz", "500 Hz", "100 Hz", "125.0  Hz", " 62.5 Hz ", "125"]
    lengths = [4096, 3000, 2049, 1500]
    for i, rate in enumerate(rates):
        for j, nl in enumerate(["\n", "\r\n", "\r"]):
            n = lengths[(i + j) % len(lengths)]
            extra = JUNK if (i + j) % 2 else ()
            text = header(rate, nl) + body(10 * i + j, n, nl, per_line=13 + 17 * j, extra=extra, trailing=(i % 3 != 2))
            files.append((f"rate{i}_nl{j}", text.encode(), 0))
    marker = header("250 Hz") + body(3, 2000) + "* MISSING PACKETS 12-13 *\n" + body(4, 1900)
    files.append(("marker_line", marker.encode(), 0))
    files.append(("blank_pieces", (header("500 Hz") + " ; ;;\n\n;\n").encode(), 0))
    files.append(("empty_region", (header() + "\n").encode(), 0))
    files.append(("short_500", (header("100 Hz") + body(5, 500)).encode(), 0))
    files.append(("over_long", (header("125 Hz") + body(6, N + 900)).encode(), 2))
    files.append(("four_lines", header().encode(), 4))
    files.append(("four_lines_no_end", header(nl="\r\n").rstrip("\r\n").encode(), 4))
    files.append(("rate_exponent", (header("1.25e2 Hz") + body(7, 3000)).encode(), 8))
    files.append(("sample_exponent", (header("62.5 Hz") + body(8, 3500, extra=["1.5e-3"])).encode(), 1))
    files.append(("long_header", (header().replace("2_11_22", "2" * 1100 + "_11_22") + body(9, 4096)).encode(), 8))
    files.append(("utf8_header", (header().replace("X axis", "X é axis") + body(11, 4000)).encode("utf-8"), 8))
    return files


@pytest.fixture(scope="module")
def logs(tmp_path_factory):
    d = tmp_path_factory.mktemp("logs")
    out = []
    for name, data, flag in corpus():
        path = d / (name + ".log")
        path.write_bytes(data)
        out.append((str(path), flag))
    return out


def ragged_records(an, samples, fs, dtype, flexible, k, cap, n=N):
    """apda_analyze_ragged_*_dev on the given per-file samples (at most n each), n_max = ld = n."""
    import torch
    dt = np.float64 if dtype == "f64" else np.float32
    b = len(samples)
    x = np.zeros((b, n), dtype=dt)
    nv = np.zeros(b, dtype=np.int32)
    for i, s in enumerate(samples):
        s = np.asarray(s, dtype=dt)[:n]
        x[i, :s.size] = s
        nv[i] = s.size
    d_x, d_nv = torch.from_numpy(x).cuda(), torch.from_numpy(nv).cuda()
    d_fs = torch.from_numpy(np.asarray(fs, dtype=np.float64)).cuda()
    d_rec = torch.zeros(b * (8 + 24 * cap), dtype=torch.uint8, device="cuda")
    an.ctx.call(f"apda_analyze_ragged_{dtype}_dev", _p(d_x.data_ptr()), _p(d_nv.data_ptr()), n, n, b, n, 0, int(flexible),
                0.0, _p(d_fs.data_ptr()), k, cap, _p(0), _p(d_rec.data_ptr()))
    an.sync()
    return d_rec.cpu().numpy().view(rec_dtype(cap))


def raw_call(an, paths, n=N, dtype="f64", flexible=True, k=4, cap=5):
    b = len(paths)
    recs = np.zeros(b, dtype=rec_dtype(cap))
    fs = np.full(b, -1.0)
    nv = np.full(b, -1, dtype=np.int32)
    fl = np.full(b, -1, dtype=np.int32)
    head = np.full((b, HEAD), 0xA5, dtype=np.uint8)
    arr = (ctypes.c_char_p * max(b, 1))(*[os.fsencode(p) for p in paths])
    an.ctx.call(f"apda_analyze_logs_{dtype}_host", ctypes.cast(arr, _p), b, n, 0, int(flexible), k, cap,
                _p(recs.ctypes.data), _p(fs.ctypes.data), _p(nv.ctypes.data), _p(fl.ctypes.data), _p(head.ctypes.data))
    return recs, fs, nv, fl, head


def same_peaks(a, b):
    """Equal count, status and peak indices; magnitudes within fp32 rounding."""
    c = int(a["count"])
    return (c == int(b["count"]) and int(a["status"]) == int(b["status"])
            and (a["pk"]["idx"] == b["pk"]["idx"]).all()
            and np.allclose(a["pk"]["mag"][:c], b["pk"]["mag"][:c], rtol=1e-5, atol=0))


def thread_count():
    return len(os.listdir("/proc/self/task"))


# ---------------------------------------------------------------------------------------------------------------
# 1. Analyzer.analyze_logs == load_sensor -> start_fft -> picker
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("flexible", [True, False], ids=["prominence", "resolution"])
def test_analyze_logs_matches_load_sensor(an, logs, dtype, flexible):
    from apda_fft_b200.records import gateway_entry, prominence_dicts, resolution_dicts
    paths = [p for p, _ in logs]
    wants = [load_sensor(p) for p in paths]
    samples = [w["samples"] if w else [] for w in wants]
    fss = [w["metadata"]["fs"] if w else 0.0 for w in wants]
    flag = [f for _, f in logs]
    assert set(flag) == {0, 1, 2, 4, 8}
    for k in (1, 2, 3, 4, 5, 7):
        cap = max(5, k)
        recs, metas = an.analyze_logs(paths, N, flexible=flexible, k=k, dtype=dtype)
        ref = ragged_records(an, samples, fss, dtype, flexible, k, cap)
        for i, (path, want) in enumerate(zip(paths, wants)):
            got = recs[i:i + 1].tobytes()
            if want is None:
                assert metas[i] is None, path
                assert got == empty_record(cap, 8), path
                continue
            assert metas[i] == {"metadata": want["metadata"], "summary": want["summary"]}, path
            if len(want["samples"]) > N:
                assert got == empty_record(cap, 4), path
                continue
            n = len(want["samples"])
            if flag[i] & (1 | 8) and dtype == "f32" and n != N:
                # the host route transforms a window shorter than N on K1's fast fp32 kernel, the ragged path on the
                # general one: the same peaks, magnitudes within fp32 rounding
                assert same_peaks(recs[i], ref[i]), (path, k, recs[i], ref[i])
            else:
                assert got == ref[i:i + 1].tobytes(), (path, k, recs[i], ref[i])
            if n == 0 or c_oracle.padded_len(n) != N:
                continue
            x = np.asarray(want["samples"], dtype=np.float64 if dtype == "f64" else np.float32)
            one = an.analyze(x[None, :], fss[i], flexible=flexible, k=k, n_fft=N, rec_cap=cap, resolve_ties=False)
            if dtype == "f64" or n == N:
                assert got == one.tobytes(), (path, k)
            else:
                assert same_peaks(recs[i], one[0]), (path, k)
            if dtype == "f64":
                spec = c_oracle.start_fft_batch(np.asarray(want["samples"], dtype=np.float64), n_fft=N)[0]
                if flexible:
                    mine, oracle = prominence_dicts(recs[i], fss[i], N), c_oracle.peaks_prominence(spec, fss[i], k)
                else:
                    mine, oracle = resolution_dicts(recs[i], fss[i], N), c_oracle.peaks_resolution(spec, fss[i], k)
                assert mine == oracle, (path, k)
                assert gateway_entry(mine) == gateway_entry(oracle)


def test_analyze_logs_strict_and_errors(an, logs, tmp_path):
    paths = [p for p, f in logs if f in (0, 1)]
    recs, _ = an.analyze_logs(paths, N)
    assert (recs["status"] != 0).any()          # short files pad to another length
    with pytest.raises(Exception, match="not reference-equivalent"):
        an.analyze_logs(paths, N, strict=True)
    full = [p for p, f in logs if f == 0 and len(load_sensor(p)["samples"]) in range(N // 2 + 1, N + 1)]
    recs, _ = an.analyze_logs(full, N, strict=True)
    assert (recs["status"] == 0).all()
    missing = str(tmp_path / "missing.log")
    with pytest.raises(FileNotFoundError):
        an.analyze_logs([paths[0], missing], N)
    with pytest.raises(IsADirectoryError):
        an.analyze_logs([str(tmp_path), paths[0]], N)
    bad_fields = tmp_path / "fields.log"
    bad_fields.write_text("a;b;125 Hz\nSynced;\n1;2;3;4;5;\n1;2;3;\n1.0;2.0;\n")
    with pytest.raises(ValueError):
        an.analyze_logs([str(bad_fields)], N)
    bad_summary = tmp_path / "summary.log"
    bad_summary.write_text("a;b;125 Hz;X axis;\nSynced;\n1;2\n1;2;3;\n1.0;2.0;\n")
    with pytest.raises(IndexError):
        an.analyze_logs([str(bad_summary)], N)
    with pytest.raises(ValueError):
        an.analyze_logs(paths, N, dtype="f16")
    recs, metas = an.analyze_logs([], N)
    assert recs.shape == (0,) and metas == []


# ---------------------------------------------------------------------------------------------------------------
# 2. the raw C call: flags, statuses, rates, counts, header bytes
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_raw_call_flags_rates_and_heads(an, logs, tmp_path, dtype):
    from utils.load_data import split_log
    fields = tmp_path / "fields.log"
    fields.write_text("a;b;125 Hz\nSynced;\n1;2;3;4;5;\n1;2;3;\n1.0;2.0;\n")
    nan_rate = tmp_path / "nan_rate.log"
    nan_rate.write_text(header("nan Hz") + "1.0;2.0;\n")
    cases_ = logs + [(str(fields), 8), (str(nan_rate), 8), (str(tmp_path / "missing.log"), 16), (str(tmp_path), 16)]
    paths = [p for p, _ in cases_]
    recs, fs, nv, fl, head = raw_call(an, paths, dtype=dtype, k=3, cap=6)
    assert fl.tolist() == [f for _, f in cases_]
    status_of = {1: 0, 2: 4, 4: 8, 8: 0, 16: 0}
    for i, (path, flag) in enumerate(cases_):
        if flag:
            assert recs[i:i + 1].tobytes() == empty_record(6, status_of[flag]), path
        if flag & (4 | 8 | 16):
            assert fs[i] == 0.0 and nv[i] == 0 and not head[i].any(), path
            continue
        with open(path, "rb") as fh:
            data = fh.read()
        rows, region = split_log(data)
        want_head = data[:len(data) - len(region)]          # the raw bytes, line ends as in the file
        raw = head[i].tobytes()
        assert raw[:len(want_head)] == want_head and not any(raw[len(want_head):]), path
        rate = rows[0].strip().split(";")[2]
        assert struct.pack("<d", fs[i]) == struct.pack("<d", float(rate.replace(" Hz", ""))), path
        if flag == 0:
            assert nv[i] == len(load_sensor(path)["samples"]), path
        if flag == 2:
            assert nv[i] == N, path


def test_raw_call_rate_grammar(an, tmp_path):
    """h_fs is bit-equal to float() on every rate field the device decides; the others raise flag 8."""
    decided = ["125.0 Hz", "31.25 Hz", " 0.5 Hz", "+1000 Hz", "-62.5 Hz", "7.", ".5 Hz ", "00012.500 Hz",
               "123456789.012345 Hz", "0.0000000000000000000001 Hz", "1 Hz Hz", "\t250\t", "25 Hz0"]
    undecided = ["1e2 Hz", "1_0 Hz", "Hz", "", " Hz", "inf Hz", "nan", "12 Hz x", "1.2.3 Hz", "9" * 16 + " Hz",
                 "1" * 70 + " Hz"]
    paths = []
    for i, rate in enumerate(decided + undecided):
        p = tmp_path / f"r{i}.log"
        p.write_bytes((header(rate) + "1.0;2.0;3.0;\n").encode())
        paths.append(str(p))
    recs, fs, nv, fl, head = raw_call(an, paths, n=64)
    for i, rate in enumerate(decided):
        assert fl[i] == 0, rate
        assert struct.pack("<d", fs[i]) == struct.pack("<d", float(rate.replace(" Hz", ""))), rate
        assert nv[i] == 3
    for i, rate in enumerate(undecided, len(decided)):
        assert fl[i] == 8, rate


# ---------------------------------------------------------------------------------------------------------------
# 3. many chunks, order, repeatability, threads
# ---------------------------------------------------------------------------------------------------------------
def test_many_chunks_order_repeat_and_threads(an, tmp_path):
    """N = 8192 fp64: a chunk holds 768 files, so 2600 files make four chunks (and many more files than readers).
    Sizes run from 5 lines to N samples; every 97th file holds up to 16 N samples (flag 2)."""
    n = 8192
    rng = np.random.default_rng(5)
    counts = rng.integers(0, n + 1, size=2600)
    counts[::97] = rng.integers(n + 1, 16 * n + 1, size=counts[::97].size)
    counts[5] = n
    rates = np.array([31.25, 62.5, 125.0, 250.0, 500.0, 100.0])[rng.integers(0, 6, size=counts.size)]
    paths, samples = [], []
    for i, (c, r) in enumerate(zip(counts, rates)):
        vals = np.round(np.sin(np.arange(c) * (0.05 + 0.001 * (i % 50))) + 0.01 * (i % 7), 6)
        text = header(f"{r} Hz") + ";".join("%8.6f" % v for v in vals) + ";\n"
        p = tmp_path / f"f{i:05d}.log"
        p.write_bytes(text.encode())
        paths.append(str(p))
        samples.append([float("%8.6f" % v) for v in vals[:n]])
    raw_call(an, paths[:3], n=n)                     # the CUDA runtime's own threads exist from here on
    before = thread_count()
    first = raw_call(an, paths, n=n)
    assert thread_count() == before
    second = raw_call(an, paths, n=n)
    assert thread_count() == before
    for a, b in zip(first, second):
        assert a.tobytes() == b.tobytes()
    recs, fs, nv, fl, _ = first
    big = counts > n
    assert (fl == np.where(big, 2, 0)).all()
    assert (nv == np.minimum(counts, n)).all()
    assert (fs == rates).all()
    ref = ragged_records(an, samples, rates, "f64", True, 4, 5, n=n)
    for i in np.flatnonzero(big):
        assert recs[i:i + 1].tobytes() == empty_record(5, 4)
    ok = np.flatnonzero(~big)
    assert recs[ok].tobytes() == ref[ok].tobytes()
    with pytest.raises(ValueError):
        raw_call(an, paths, n=3)
    assert thread_count() == before


# ---------------------------------------------------------------------------------------------------------------
# 4. argument errors
# ---------------------------------------------------------------------------------------------------------------
def test_argument_errors(an, logs):
    path = logs[0][0]
    recs = np.zeros(2, dtype=rec_dtype(64))
    fs, nv, fl = np.zeros(2), np.zeros(2, dtype=np.int32), np.zeros(2, dtype=np.int32)
    head = np.zeros((2, HEAD), dtype=np.uint8)
    good = (ctypes.c_char_p * 2)(path.encode(), path.encode())
    holey = (ctypes.c_char_p * 2)(path.encode(), None)

    def call(paths=ctypes.cast(good, _p), n_files=2, n=N, flags=0, k=4, cap=5, dtype="f64", out=True):
        ptr = _p(recs.ctypes.data) if out else _p(0)
        an.ctx.call(f"apda_analyze_logs_{dtype}_host", paths, n_files, n, flags, 1, k, cap, ptr, _p(fs.ctypes.data),
                    _p(nv.ctypes.data), _p(fl.ctypes.data), _p(head.ctypes.data))

    call()
    call(dtype="f32", n=16384)
    for kw in [dict(paths=_p(0)), dict(paths=ctypes.cast(holey, _p)), dict(n_files=-1), dict(n=0), dict(n=2),
               dict(n=3), dict(n=6144), dict(n=16384), dict(n=32768, dtype="f32"), dict(flags=1), dict(flags=7),
               dict(k=0), dict(k=6, cap=5), dict(cap=N), dict(out=False)]:
        with pytest.raises(ValueError):
            call(**kw)
