"""What presenting a record table costs on the device against the Python presentation it replaces (DESIGN.md, present.cu).

    python scripts/present_probe.py [--out FILE.json]

Records: the cfg5 fleet (1M x 4096 fp32 windows of apda_synth_f32_dev, seed 42) through apda_analyze_f32_dev, once per
picker (flexible k = 4, rigid k = 5, rec_cap 5).  For each picker:
  - apda_present_dev (all columns) and apda_fleet_jsonl_dev: CUDA events after warm-up, records already in HBM;
  - apda_present_host and apda_fleet_jsonl_host from host records: wall clock, H2D + kernels + D2H included;
  - records.write_fleet_jsonl and a prominence_dicts / resolution_dicts loop on this host over the first 100k windows;
  - equality: the _host text of all windows equals the _dev text, the first 100k windows' text equals
    write_fleet_jsonl's, and their columns equal the dicts' fields bit for bit.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import apda_fft_b200  # noqa: E402
from apda_fft_b200 import _cabi  # noqa: E402
from apda_fft_b200.records import prominence_dicts, record_dtype, resolution_dicts, write_fleet_jsonl  # noqa: E402
from test_gpu_present import check_columns, want_columns  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    name, power = [s.strip() for s in q.split(",")]
    return {"gpu": name, "power_limit": power}


def event_ms(fn, reps):
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out))


def wall_ms(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--py-windows", type=int, default=100_000)
    args = ap.parse_args()
    an = apda_fft_b200.Analyzer(0)
    an.use_stream(torch.cuda.current_stream().cuda_stream)
    res = {"card": card(), "cpus": os.cpu_count()}
    b, n, fs, cap = 1_000_000, 4096, 125.0, 5
    d_x = torch.empty((b, n), dtype=torch.float32, device="cuda:0")
    an.synth_device(0, b, n, "f32", d_x.data_ptr(), seed=42)
    d_rec = torch.zeros((b, record_dtype(cap).itemsize), dtype=torch.uint8, device="cuda:0")
    res["pickers"] = []
    for flexible, k in ((True, 4), (False, 5)):
        an.analyze_device(d_x.data_ptr(), b, n, n, "f32", fs, d_rec.data_ptr(), flexible=flexible, k=k, rec_cap=cap)
        torch.cuda.synchronize()
        recs = d_rec.cpu().numpy().view(record_dtype(cap)).reshape(b)
        cols = {c: torch.empty((b, k), dtype=torch.int32 if c == "idx" else torch.float64, device="cuda:0")
                for c in ("idx", "freq", "mag", "prominence", "damping", "q")}
        ptr = {c: t.data_ptr() for c, t in cols.items()}
        cap_bytes = b * _cabi.jsonl_row_bytes(k)
        d_text = torch.empty(cap_bytes, dtype=torch.uint8, device="cuda:0")
        d_off = torch.empty(b + 1, dtype=torch.int64, device="cuda:0")

        def present_dev():
            an.present_device(d_rec.data_ptr(), b, cap, n, fs, k, ptr["idx"], ptr["freq"], ptr["mag"], ptr["prominence"],
                              ptr["damping"], ptr["q"], flexible=flexible)

        def jsonl_dev():
            an.fleet_jsonl_device(d_rec.data_ptr(), b, cap, n, fs, d_text.data_ptr(), cap_bytes, d_off.data_ptr(),
                                  flexible=flexible, k=k)
        for _ in range(3):
            present_dev()
            jsonl_dev()
        torch.cuda.synchronize()
        row = {"flexible": flexible, "k": k, "windows": b, "n": n,
               "present_dev_ms": event_ms(present_dev, args.reps), "fleet_jsonl_dev_ms": event_ms(jsonl_dev, args.reps)}
        dev_text = bytes(d_text[:int(d_off[-1])].cpu().numpy())
        row["text_bytes"] = len(dev_text)
        host_text = an.fleet_jsonl(recs, fs, n, flexible=flexible, k=k)
        an.present(recs, fs, n, flexible=flexible, k=k)
        row["present_host_ms"] = wall_ms(lambda: an.present(recs, fs, n, flexible=flexible, k=k), max(3, args.reps // 3))
        row["fleet_jsonl_host_ms"] = wall_ms(lambda: an.fleet_jsonl(recs, fs, n, flexible=flexible, k=k),
                                             max(3, args.reps // 3))
        assert host_text == dev_text, "fleet_jsonl _host and _dev texts differ"

        m = args.py_windows
        head = recs[:m]
        conv = prominence_dicts if flexible else resolution_dicts
        t0 = time.perf_counter()
        for w in range(m):
            conv(head[w], fs, n)
        t1 = time.perf_counter()
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "fleet.jsonl")
            write_fleet_jsonl(path, head, fs, n, flexible, k)
            t2 = time.perf_counter()
            with open(path, "rb") as fh:
                py_text = fh.read()
        assert dev_text.startswith(py_text), "device text differs from write_fleet_jsonl"
        check_columns(an.present(head, fs, n, flexible=flexible, k=k), want_columns(head, fs, n, flexible, k), flexible)
        row.update({"python_windows": m, "python_dicts_us_per_window": 1e6 * (t1 - t0) / m,
                    "python_write_fleet_jsonl_us_per_window": 1e6 * (t2 - t1) / m,
                    "equal": True})
        res["pickers"].append(row)
        del cols, d_text, d_off
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)
            fh.write("\n")


if __name__ == "__main__":
    main()
