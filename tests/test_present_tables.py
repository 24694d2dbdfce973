"""CPU tests of present.cu's power-of-five tables (apda-fft_b200/csrc/present_tables.cuh): the committed header is what
scripts/gen_present_tables.py generates, and every entry meets its definition in Python's exact integer arithmetic."""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GEN = os.path.join(ROOT, "scripts", "gen_present_tables.py")
HEADER = os.path.join(ROOT, "apda-fft_b200", "csrc", "present_tables.cuh")


def committed_tables():
    text = open(HEADER).read()
    tables = {}
    for name, body in re.findall(r"unsigned long long (\w+)\[\d+\]\[2\] = \{(.*?)\n\};", text, re.S):
        pairs = re.findall(r"\{0x([0-9a-f]{16})ull, 0x([0-9a-f]{16})ull\}", body)
        tables[name] = [int(lo, 16) | (int(hi, 16) << 64) for lo, hi in pairs]
    return tables


def test_generator_reproduces_the_committed_header():
    res = subprocess.run([sys.executable, GEN, "--check"], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr


def test_entries_match_exact_powers_of_five():
    t = committed_tables()
    inv, pos = t["kPow5InvSplit"], t["kPow5Split"]
    assert len(inv) == 342 and len(pos) == 326
    for i, v in enumerate(inv):
        p = 5 ** i
        j = p.bit_length() - 1 + 125
        # the smallest integer above 2^j / 5^i, 125 or 126 bits
        assert (v - 1) * p <= (1 << j) < v * p, i
        assert v < 1 << 126
    for i, v in enumerate(pos):
        p = 5 ** i
        assert v.bit_length() == 125, i
        s = p.bit_length() - 125
        assert v == (p >> s if s >= 0 else p << -s), i
        if s > 0:  # the truncated bits are below the kept 125
            assert v << s <= p < (v + 1) << s


def test_index_helpers_match_exact_logarithms():
    """repr.cuh's pow5bits / log10_pow2 / log10_pow5 over the exponent ranges the formatter uses."""
    for e in range(0, 3529):
        assert ((e * 1217359) >> 19) + 1 == max(1, (5 ** e).bit_length()), e
    for e in range(0, 1651):
        assert (e * 78913) >> 18 == len(str(2 ** e)) - 1, e
    for e in range(0, 2621):
        assert (e * 732923) >> 20 == len(str(5 ** e)) - 1, e
