"""bench.py contract checks: the reference arm needs no GPU (oracle port on the host cores) and prints one JSON line with
the keys a caller reads; the output dump of the GPU arm needs a B200."""
# the arm times the unmodified reference from oracle/_ref when that build-time copy exists, else the oracle port
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                                   "--warmup", "0"], text=True, cwd=ROOT, timeout=600)
    lines = [ln for ln in out.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "windows/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("FFT+peak windows/sec at N=4096")
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                                   "--steps", "1", "--warmup", "0"], text=True, cwd=ROOT, env=env, timeout=120)
    assert out.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_do_not_depend_on_the_step_count(tmp_path):
    """--dump-outputs writes the last timed step's records and a sample of its spectra; two runs that time a different
    number of steps (reported as "steps") dump the same arrays, and each dumped peak is the magnitude of its bin."""
    import numpy as np

    def run(steps):
        out_dir = tmp_path / f"steps{steps}"
        out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                                       "--warmup", "1", "--windows", "20000", "--no-variants", "--no-e2e", "--no-configs",
                                       "--no-cpu-baseline", "--dump-outputs", str(out_dir)], text=True, cwd=ROOT, timeout=600)
        assert json.loads([ln for ln in out.splitlines() if ln.startswith("{")][-1])["steps"] == steps
        assert sum(f.stat().st_size for f in out_dir.iterdir()) <= 64 << 20
        return {f.stem: np.load(f) for f in out_dir.iterdir()}

    one, three = run(1), run(3)
    assert set(one) == {"record_window", "record_count", "record_status", "peak_idx", "peak_width_bins", "peak_mag",
                        "peak_prominence", "spectrum_window", "spectrum"}
    for name, a in one.items():
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, three[name]), name
    assert np.array_equal(one["record_window"], np.arange(20000)) and one["spectrum"].shape == (1024, 4096, 2)
    rows = one["spectrum_window"].astype(np.int64)
    idx = one["peak_idx"][rows].astype(np.int64)
    live = idx >= 0
    spec = one["spectrum"].astype(np.float64)
    mag = np.hypot(*np.moveaxis(np.take_along_axis(spec, np.maximum(idx, 0)[:, :, None], axis=1), 2, 0))
    np.testing.assert_allclose(mag[live], one["peak_mag"][rows][live], rtol=1e-5)
