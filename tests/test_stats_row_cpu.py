"""The row composer of k_stats_rows (the __host__ __device__ stats_row_len / stats_row_put of csrc/stats_row.cuh) against the host
formatter rbh::append_row, on the CPU: random names up to 3 KB, coordinates up to u64 max, random counters, identities from random
bits, exact decimal ties, NaN, 0 and 100, both column orders."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "rustybam_b200", "host")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("native") / "stats_row_check")
    srcs = [os.path.join(HOST, f) for f in sorted(os.listdir(HOST)) if f.endswith(".cpp") and f != "rb_main.cpp"]
    subprocess.check_call(
        ["g++", "-O1", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "rustybam_b200", "csrc"), "-I", HOST, "-I",
         os.path.join(ROOT, "include"), "-o", exe, os.path.join(ROOT, "tests", "native", "stats_row_check.cpp")] + srcs + ["-lz"])
    return exe


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_composer_matches_host_formatter(harness, seed):
    r = subprocess.run([harness, str(seed), "30000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "FAIL=0" in r.stdout
    counts = dict(kv.split("=") for kv in r.stdout.split() if "=" in kv)
    # every kind of input is exercised
    assert int(counts["tie_values"]) > 0 and int(counts["ties"]) > 1000, r.stdout
    assert int(counts["long_names"]) > 300 and int(counts["negative"]) > 1000, r.stdout
