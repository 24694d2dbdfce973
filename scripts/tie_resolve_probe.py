"""What apda_resolve_fp32_ties_{dev,host} cost (DESIGN.md, K-ties).

    python scripts/tie_resolve_probe.py [--out FILE.json]

(a) apda_resolve_fp32_ties_dev on the records of the cfg5 fleet (1M x 4096 fp32, K1 + K3 split pipeline, generator seed 42),
    restored before every timed call so each one meets the fleet's own ties;
(b) the same call on tie-rich batches (100k windows at N = 4096 and 8192): time per resolved window;
(c) apda_analyze_f32_host followed by apda_resolve_fp32_ties_host against apda_analyze_f32_host alone (100k x 4096).
Device times are CUDA events after warm-up; host times are wall clock around calls that return synchronised.  The card's
name and power limit are read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import apda_fft_b200  # noqa: E402
from test_gpu_fp32_ties import tie_windows  # noqa: E402

_p = ctypes.c_void_p
TIE = 16


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    name, power = [s.strip() for s in q.split(",")]
    return {"gpu": name, "power_limit": power}


def event_ms(fn, reps, before=None):
    """Median of `reps` CUDA-event timings of fn() (before() runs outside the timed span)."""
    out = []
    for _ in range(reps):
        if before:
            before()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.median(out))


def resolve(an, d_x, b, n, d_rec):
    an.resolve_fp32_ties_device(d_x.data_ptr(), b, n, n, 125.0, d_rec.data_ptr(), flexible=True, k=4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    an = apda_fft_b200.Analyzer(0)
    an.use_stream(torch.cuda.current_stream().cuda_stream)
    res = {"card": card()}

    # (a) the cfg5 fleet
    b, n = 1_000_000, 4096
    d_x = torch.empty((b, n), dtype=torch.float32, device="cuda:0")
    an.synth_device(0, b, n, "f32", d_x.data_ptr(), seed=42)
    d_spec = torch.empty((b, n, 2), dtype=torch.float32, device="cuda:0")
    d_rec = torch.zeros((b, 128), dtype=torch.uint8, device="cuda:0")
    an.fft_device(d_x.data_ptr(), b, n, n, "f32", d_spec.data_ptr())
    an.peaks_device(d_spec.data_ptr(), b, n, "f32", 125.0, d_rec.data_ptr(), flexible=True, k=4)
    step_ms = event_ms(lambda: (an.fft_device(d_x.data_ptr(), b, n, n, "f32", d_spec.data_ptr()),
                                an.peaks_device(d_spec.data_ptr(), b, n, "f32", 125.0, d_rec.data_ptr(), flexible=True, k=4)),
                       5)
    del d_spec
    saved = d_rec.clone()
    ties = int((saved.view(torch.int32)[:, 1] == TIE).sum())
    restore = lambda: d_rec.copy_(saved)  # noqa: E731
    for _ in range(3):
        restore()
        resolve(an, d_x, b, n, d_rec)
    res["a_fleet"] = {"windows": b, "n": n, "ties": ties, "k1_k3_step_ms": step_ms,
                      "resolve_dev_ms": event_ms(lambda: resolve(an, d_x, b, n, d_rec), args.reps, restore)}
    del d_x, d_rec, saved
    torch.cuda.empty_cache()

    # (b) tie-rich batches
    res["b_tie_rich"] = []
    for n in (4096, 8192):
        b = 100_000
        d_x = torch.empty((b, n), dtype=torch.float32, device="cuda:0")
        for lo in range(0, b, 10_000):
            d_x[lo:lo + 10_000] = torch.from_numpy(tie_windows(10_000, n, seed=lo + n)[0]).cuda()
        d_rec = torch.zeros((b, 128), dtype=torch.uint8, device="cuda:0")
        an.analyze_device(d_x.data_ptr(), b, n, n, "f32", 125.0, d_rec.data_ptr(), flexible=True, k=4)
        torch.cuda.synchronize()
        saved = d_rec.clone()
        ties = int((saved.view(torch.int32)[:, 1] == TIE).sum())
        restore = lambda: d_rec.copy_(saved)  # noqa: E731
        for _ in range(2):
            restore()
            resolve(an, d_x, b, n, d_rec)
        ms = event_ms(lambda: resolve(an, d_x, b, n, d_rec), max(3, args.reps // 4), restore)
        res["b_tie_rich"].append({"windows": b, "n": n, "ties": ties, "resolve_dev_ms": ms,
                                  "us_per_resolved_window": 1e3 * ms / max(ties, 1)})
        del d_x, d_rec, saved
        torch.cuda.empty_cache()

    # (c) host entry points on tie-rich host windows
    b, n = 100_000, 4096
    x = np.concatenate([tie_windows(10_000, n, seed=lo)[0] for lo in range(0, b, 10_000)])
    recs = np.zeros((b, 128), dtype=np.uint8)

    def analyze():
        an.ctx.call("apda_analyze_f32_host", _p(x.ctypes.data), n, n, b, n, 0, 1, 125.0, _p(0), 4, 5, _p(recs.ctypes.data))

    def resolve_host():
        an.ctx.call("apda_resolve_fp32_ties_host", _p(x.ctypes.data), _p(0), n, n, b, n, 0, 1, 125.0, _p(0), 4, 5,
                    _p(recs.ctypes.data))
    analyze()
    resolve_host()
    t_a, t_ar = [], []
    for _ in range(5):
        t0 = time.perf_counter()
        analyze()
        t1 = time.perf_counter()
        ties = int((recs.view(np.int32).reshape(b, -1)[:, 1] == TIE).sum())
        resolve_host()
        t2 = time.perf_counter()
        t_a.append(t1 - t0)
        t_ar.append(t2 - t0)
    res["c_host"] = {"windows": b, "n": n, "ties": ties, "analyze_host_ms": 1e3 * float(np.median(t_a)),
                     "analyze_plus_resolve_host_ms": 1e3 * float(np.median(t_ar))}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
