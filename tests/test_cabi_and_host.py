"""CPU-side tests: the C-ABI library loads and exports every symbol of include/apda_b200.h, there is no silent
fallback, and the host logic (record decoding, sharding, gather, log parser) behaves like the reference."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import cases
from oracle import ref_port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "apda-fft_b200")


@pytest.fixture(scope="module")
def lib():
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.build()
    import apda_fft_b200
    return apda_fft_b200.load()


def test_library_exports_every_declared_symbol(lib):
    import apda_fft_b200._cabi as cabi
    header = open(os.path.join(ROOT, "include", "apda_b200.h")).read()
    declared = set(re.findall(r"\b(apda_[a-z0-9_]+)\s*\(", header))
    assert declared == set(cabi.SIGNATURES), declared ^ set(cabi.SIGNATURES)
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.apda_version() >= 100


def test_no_cpu_fallback(lib):
    """Without a CUDA device the product path must fail loudly (and never route through oracle/)."""
    import torch
    import apda_fft_b200
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible; the loud-failure path is exercised on the CPU box")
    with pytest.raises(apda_fft_b200.ApdaError, match="no CPU fallback"):
        apda_fft_b200.Analyzer(0)
    sys.path.insert(0, PKG)
    from metrics.fft_iterativa import start_fft
    with pytest.raises(apda_fft_b200.ApdaError):
        start_fft([1.0, 2.0, 3.0, 4.0], 1.0)
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), f"{f} imports the oracle"


def test_record_layout_and_decoding(golden):
    from apda_fft_b200.records import prominence_dicts, record_dtype, resolution_dicts
    from oracle import c_oracle
    assert record_dtype(5).itemsize == 128 and record_dtype(12).itemsize == 8 + 24 * 12
    for cid in ("katA", "katB", "katC", "pad3000", "noise4096", "six_tones"):
        g = golden["cases"][cid]
        x, fs = cases.build_samples(g["spec"])
        n = g["n_fft"]
        mags = c_oracle.half_magnitudes(c_oracle.start_fft_batch(x)[0]).tolist()
        rec = np.zeros(1, dtype=record_dtype(5))[0]
        want = g["prominence"]["ok"]
        rec["count"] = len(want)
        for a, p in enumerate(want):
            rec["pk"][a] = (p["idx"], ref_port.half_power_bins(mags, p["prominence"], p["idx"]), mags[p["idx"]], p["prominence"])
        assert prominence_dicts(rec, fs, n) == want
        want = g["resolution"]["ok"]
        rec["count"] = len(want)
        for a, p in enumerate(want):
            rec["pk"][a] = (p["idx"], 2, p["mag"], 0.0)
        assert resolution_dicts(rec, fs, n) == want


def test_shard_bounds():
    from apda_fft_b200.fleet import shard_bounds, shard_capacity
    for total in (0, 1, 7, 8, 1000, 1_000_000):
        for world in (1, 2, 3, 4, 8):
            spans = [shard_bounds(total, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert all(hi - lo <= shard_capacity(total, world) for lo, hi in spans)


def _gloo_worker(rank, world, port, total, tmp):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from apda_fft_b200.fleet import gather_records, shard_bounds, shard_capacity
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    lo, hi = shard_bounds(total, world, rank)
    local = torch.zeros((shard_capacity(total, world), 128), dtype=torch.uint8)
    for i in range(hi - lo):          # a record that encodes its own window index
        local[i] = torch.tensor(np.frombuffer(np.int64(lo + i).tobytes() * 16, dtype=np.uint8).copy())
    table = gather_records(local, total, dst=0)
    if rank == 0:
        np.save(os.path.join(tmp, "table.npy"), table.numpy())
    else:
        assert table is None
    # the sliced, overlapped gather used by the fleet sweep gives the same table (two consecutive steps reuse it)
    from apda_fft_b200.fleet import RecordGatherer
    g = RecordGatherer(shard_capacity(total, world), 128, local.device)
    for _ in range(2):
        for a, z in g.slices(3):
            g.start(local, a, z)
        sliced = g.finish()
        if rank == 0:
            assert np.array_equal(sliced[:total].numpy(), table.numpy())
        else:
            assert sliced is None
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,total", [(2, 10), (2, 7), (3, 8)])
def test_gather_records_gloo(tmp_path, world, total):
    """N>1 path on CPU: world_size ranks over gloo; the gathered table is in window order, byte for byte."""
    import torch.multiprocessing as mp
    port = 29500 + (os.getpid() * 7 + world * 13 + total) % 2000
    mp.spawn(_gloo_worker, args=(world, port, total, str(tmp_path)), nprocs=world, join=True)
    table = np.load(os.path.join(str(tmp_path), "table.npy"))
    assert table.shape == (total, 128)
    assert (table.view(np.int64)[:, 0] == np.arange(total)).all()


LOG_TEXT = """2_11_22_18_20_32;2 g;31.25 Hz;Z axis;
Synced2;
25.010;-0.0222;0.0110;0.9981;85.0;
0.268262;-0.5;1.0;
0.100000;0.200000;-0.300000;
* MISSING PACKETS 3-4 *
0.400000;nan;inf;;0.500000
-0.000000;1e3;abc;
"""


def test_load_sensor(tmp_path):
    sys.path.insert(0, PKG)
    from utils.load_data import load_sensor
    path = tmp_path / "a.log"
    path.write_text(LOG_TEXT)
    got = load_sensor(str(path))
    assert got["metadata"] == {"timestamp": "2_11_22_18_20_32", "sensitivity": "2g", "fs": 31.25, "axis": "Z",
                               "sync_type": "Synced2", "is_synced": 1.0}
    assert list(got["metadata"]) == ["timestamp", "sensitivity", "fs", "axis", "sync_type", "is_synced"]
    assert got["summary"] == {"temperature": 25.01, "rms_x": -0.0222, "rms_y": 0.011, "rms_z": 0.9981, "humidity": 85.0,
                              "first_x": 0.268262, "first_y": -0.5, "first_z": 1.0}
    assert got["samples"] == [0.1, 0.2, -0.3, 0.4, 0.5, -0.0, 1000.0]
    short = tmp_path / "b.log"
    short.write_text("a;b;1 Hz;X axis;\nNo;\n")
    assert load_sensor(str(short)) is None


def test_pure_host_helpers():
    sys.path.insert(0, PKG)
    from metrics.fft_iterativa import Spectrum, bit_reversal, pad, pack_spectrum
    assert pad([]) == [0] and pad([1]) == [1] and pad([1, 2, 3]) == [1, 2, 3, 0] and len(pad([0.5] * 1025)) == 2048
    assert bit_reversal(list(range(16))) == [ref_port.bitrev_indices(16)[i] for i in range(16)]
    s = Spectrum([0, 1j, 2j, 3j], np.array([0, 1j, 2j, 3j]))
    assert pack_spectrum(s) is s._packed
    s[1] = 5j
    assert s._packed is None and pack_spectrum(s)[1] == 5j


def test_synth_device_twin_constants():
    """Host generator: every row of the vectorised generator equals the scalar one (the device twin is checked on GPU)."""
    import apda_fft_b200.synth as synth
    block = synth.fleet_windows(123, 3, 256, on_bin=True, dtype=np.float32)
    for r in range(3):
        assert np.array_equal(block[r], synth.fleet_window(123 + r, 256, on_bin=True).astype(np.float32))


def test_gateway_entry_and_fleet_table(golden):
    from apda_fft_b200.records import fleet_table, gateway_entry, record_dtype
    peaks = golden["cases"]["katA"]["prominence"]["ok"]
    entry = gateway_entry(peaks)
    assert entry["peak_freq"] == 3.0518 and entry["max_mag"] == 195.833 and entry["peak_freq_3"] == 15.1367
    assert gateway_entry([]) == {"peak_freq": -1, "max_mag": -1}
    recs = np.zeros(2, dtype=record_dtype(5))
    recs["pk"]["idx"] = -1
    recs[0]["count"] = 2
    recs[0]["pk"][0] = (25, 2, 195.8, 195.7)
    recs[0]["pk"][1] = (63, 2, 149.3, 149.1)
    count, idx, freq, mag = fleet_table(recs, 125.0, 1024)
    assert count.tolist() == [2, 0] and idx[0, :2].tolist() == [25, 63] and freq[0, 0] == 25 * (125.0 / 1024)
    assert np.isnan(freq[1]).all() and mag[0, 1] == 149.3


def _build_c_example(tmp_path):
    import subprocess
    exe = os.path.join(str(tmp_path), "analyze_host")
    libdir = os.path.join(ROOT, "apda-fft_b200")
    subprocess.check_call(["gcc", "-O2", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "analyze_host.c"), "-L", libdir, "-lapda_b200",
                           f"-Wl,-rpath,{libdir}", "-lm", "-o", exe])
    return exe


def test_c_host_example_compiles_and_links(lib, tmp_path):
    """include/apda_b200.h is a plain-C header and the library links from C (no CUDA headers, no Python)."""
    assert os.path.exists(_build_c_example(tmp_path))


def test_result_packing_arrow_jsonl_and_upload_metrics(golden, tmp_path):
    """SURVEY 8f rank 4: columnar / JSONL packing of a record batch and the uploader's `metriche` block."""
    import json
    from apda_fft_b200.records import (fleet_arrow, gateway_entry, record_dtype, upload_metrics, write_fleet_jsonl,
                                       prominence_dicts)
    recs = np.zeros(3, dtype=record_dtype(5))
    recs["pk"]["idx"] = -1
    recs[0]["count"] = 2
    recs[0]["pk"][0] = (25, 2, 195.8331234, 195.7)
    recs[0]["pk"][1] = (63, 2, 149.3, 149.1)
    recs[2]["count"] = 1
    recs[2]["pk"][0] = (100, 3, 12.5, 12.0)
    tab = fleet_arrow(recs, 125.0, 1024, first_window=40)
    assert tab.column("window").to_pylist() == [40, 41, 42] and tab.column("count").to_pylist() == [2, 0, 1]
    assert tab.column("idx").to_pylist() == [[25, 63], [], [100]]
    assert tab.column("freq").to_pylist()[0] == [25 * (125.0 / 1024), 63 * (125.0 / 1024)]
    assert tab.column("mag").to_pylist()[2] == [12.5]
    path = os.path.join(str(tmp_path), "fleet.jsonl")
    assert write_fleet_jsonl(path, recs, 125.0, 1024, first_window=40) == 3
    rows = [json.loads(ln) for ln in open(path)]
    want0 = prominence_dicts(recs[0], 125.0, 1024)
    assert rows[0] == {"window": 40, "fft_freqs": [want0[0]["freq"], want0[1]["freq"], 0.0, 0.0],
                       "fft_mags": [want0[0]["mag"], want0[1]["mag"], 0.0, 0.0]}
    assert rows[1]["fft_freqs"] == [0.0] * 4 and rows[2]["fft_mags"][0] == 12.5

    summary = {"temperature": 25.01, "rms_x": -0.0222, "rms_y": 0.011, "rms_z": 0.9981, "humidity": 85.0}
    entry = gateway_entry(golden["cases"]["katA"]["prominence"]["ok"])
    got = upload_metrics(summary, "Z", entry)
    assert got["rms_asse"] == 0.9981 and got["fft_freqs"][:3] == [3.0518, 7.6904, 15.1367] and got["fft_freqs"][3] == 0.0
    assert got == {"temp": 25.01, "humidity": 85.0, "phi": 153.64179189369935, "theta": 1.4219587307998718,
                   "rms_asse": 0.9981, "fft_freqs": [3.0518, 7.6904, 15.1367, 0.0],
                   "fft_mags": [195.833, 149.3667, 65.4201, 0.0]}


def test_dropins_never_hand_out_a_record_with_nonzero_status():
    """The drop-in modules return reference-equivalent results or raise (VERDICT r1, weak 4): every record batch they
    decode goes through _cabi.check_record_status, which raises on any status bit (truncated candidate list, window of
    another padded length, empty window, fp32 tie) and names the first offending window."""
    from apda_fft_b200 import _cabi
    from apda_fft_b200.records import record_dtype
    recs = np.zeros(4, dtype=record_dtype(5))
    _cabi.check_record_status(recs)                      # all clean: no exception
    for bit in (_cabi.STATUS_TRUNCATED if hasattr(_cabi, "STATUS_TRUNCATED") else 1, 4, 8, _cabi.STATUS_FP32_TIE):
        recs["status"][:] = 0
        recs["status"][2] = bit
        with pytest.raises(_cabi.ApdaError) as err:
            _cabi.check_record_status(recs)
        assert "window 2" in str(err.value) and f"status {bit}" in str(err.value)
    # and both picker drop-ins really call it on what the library returns
    here = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "apda-fft_b200", "utils")
    for mod in ("get_peak_prominence.py", "get_peak_resolution.py"):
        with open(os.path.join(here, mod)) as fh:
            assert "check_record_status" in fh.read(), mod
