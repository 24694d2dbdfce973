"""How fast a directory of sensor .log files becomes one record per file, by three routes on the same files.

    python scripts/log_ingest_probe.py --out DIR [--files 20000] [--n 4096] [--reps 3]

The logs (4 header lines + n '%8.6f' samples, rates drawn from 31.25 / 62.5 / 100 / 125 / 250 / 500 Hz, seeded) are
written to a temporary directory that is removed afterwards.  Every route runs once as a warm-up, so the page cache holds
the files, then --reps times; the median is reported.
  (a) utils.load_data.load_sensors (Python reads and splits the files, GPU sample parser) + grouping by fs +
      Analyzer.analyze per group (samples kept as numpy arrays, the route's fastest form);
  (b) Analyzer.analyze_logs (reader threads, device header/rate/sample decode, ragged analysis);
  (c) file bytes alone: min(16, CPUs) threads doing what the library's readers do (open, fstat, pread into pinned
      memory, close), no kernels.  It bounds (b) from below on this host.
(a) and (b) must give byte-equal records.  Prints one JSON object (also written to <out>/log_ingest_probe.json) with the
GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "apda-fft_b200"))

HEADER = "2_11_22_18_20_32;2 g;{rate} Hz;X axis;\nSynced;\n25.010;-0.0222;0.0110;0.9981;85.0;\n0.268262;-0.5;1.0;\n"
RATES = [31.25, 62.5, 100.0, 125.0, 250.0, 500.0]
BODIES = 256  # distinct sample bodies (formatting 20 000 x 4096 values in Python would dominate the set-up)


def write_logs(d: str, files: int, n: int, seed: int) -> tuple[list[str], int]:
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    bodies = []
    for _ in range(BODIES):
        f1, f2 = rng.uniform(0.01, 0.45, size=2)
        vals = np.round(np.sin(2 * np.pi * f1 * t) + 0.5 * np.sin(2 * np.pi * f2 * t) + 0.2 * rng.standard_normal(n), 6)
        pieces = ["%8.6f" % v for v in vals]
        bodies.append("\n".join(";".join(pieces[i:i + 60]) + ";" for i in range(0, n, 60)) + "\n")
    pick = rng.integers(0, BODIES, size=files)
    rates = rng.integers(0, len(RATES), size=files)
    paths, total = [], 0
    for i in range(files):
        data = (HEADER.format(rate=RATES[rates[i]]) + bodies[pick[i]]).encode()
        p = os.path.join(d, f"sensor_{i:06d}.log")
        with open(p, "wb") as fh:
            fh.write(data)
        paths.append(p)
        total += len(data)
    return paths, total


def route_a(an, paths, n):
    from utils.load_data import load_sensors
    from apda_fft_b200.records import record_dtype
    loaded = load_sensors(paths, as_arrays=True)
    recs = np.zeros(len(paths), dtype=record_dtype(5))
    groups: dict[float, list[int]] = {}
    for i, d in enumerate(loaded):
        groups.setdefault(d["metadata"]["fs"], []).append(i)
    for fs, idx in groups.items():
        x = np.stack([loaded[i]["samples"] for i in idx])
        recs[idx] = an.analyze(x, fs, n_fft=n, resolve_ties=False)
    return recs


def route_b(an, paths, n):
    return an.analyze_logs(paths, n)[0]


def route_c(paths, pinned):
    sizes = [os.stat(p).st_size for p in paths]
    offs = np.concatenate([[0], np.cumsum(sizes)])
    view = memoryview(pinned.numpy()).cast("B")
    nxt = iter(range(len(paths)))
    lock = threading.Lock()

    def work():
        while True:
            with lock:
                i = next(nxt, None)
            if i is None:
                return
            fd = os.open(paths[i], os.O_RDONLY)
            os.fstat(fd)
            os.preadv(fd, [view[offs[i]:offs[i + 1]]], 0)
            os.close(fd)
    threads = [threading.Thread(target=work) for _ in range(min(16, os.cpu_count() or 1))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()


def timed(fn, reps):
    fn()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        times.append(time.perf_counter() - t0)
    return statistics.median(times), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=20000)
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", required=True, help="directory for log_ingest_probe.json")
    args = ap.parse_args()
    import torch
    import apda_fft_b200
    if not torch.cuda.is_available():
        raise SystemExit("log_ingest_probe: no CUDA device; nothing is measured without one")
    gpu = torch.cuda.get_device_name(0)
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True).stdout.strip()
    an = apda_fft_b200.Analyzer(0)
    with tempfile.TemporaryDirectory(prefix="apda_logs_") as d:
        paths, total = write_logs(d, args.files, args.n, args.seed)
        pinned = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        ta, ra = timed(lambda: route_a(an, paths, args.n), args.reps)
        tb, rb = timed(lambda: route_b(an, paths, args.n), args.reps)
        tc, _ = timed(lambda: route_c(paths, pinned), args.reps)
    equal = ra.tobytes() == rb.tobytes()
    res = {"gpu": gpu, "power_limit": power, "cpus": os.cpu_count(), "files": args.files, "n": args.n,
           "text_bytes": total, "page_cache": "warm (one untimed pass of each route first)", "reps": args.reps,
           "records_equal": equal}
    for key, t in (("a_load_sensors_group_analyze", ta), ("b_analyze_logs", tb), ("c_reader_threads_only", tc)):
        res[key] = {"seconds": round(t, 4), "logs_per_s": round(args.files / t, 1), "text_GB_per_s": round(total / t / 1e9, 3)}
    res["b_over_a"] = round(ta / tb, 2)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "log_ingest_probe.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))
    if not equal:
        raise SystemExit("log_ingest_probe: routes (a) and (b) give different records")


if __name__ == "__main__":
    main()
