"""The line rules k_paf_fields runs on the GPU (the __host__ __device__ core in csrc/paf_parse_core.cuh) against the host reader
rbh::Paf::from_text, on the CPU: seeded random lines with CRLF, stray form feeds, runs of mixed separators, '+17', 20-digit numbers
and u64 overflow, 2-byte strands, missing / duplicated / prefixed / empty cg tags, non-tag tokens, 11 columns and empty lines."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "rustybam_b200", "host")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("native") / "paf_parse_check")
    srcs = [os.path.join(HOST, f) for f in sorted(os.listdir(HOST)) if f.endswith(".cpp") and f != "rb_main.cpp"]
    subprocess.check_call(
        ["g++", "-O1", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "rustybam_b200", "csrc"), "-I", HOST, "-I",
         os.path.join(ROOT, "include"), "-o", exe, os.path.join(ROOT, "tests", "native", "paf_parse_check.cpp")] + srcs + ["-lz"])
    return exe


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_line_core_matches_host_reader(harness, seed):
    r = subprocess.run([harness, str(seed), "20000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "FAIL=0" in r.stdout
    counts = dict(kv.split("=") for kv in r.stdout.split() if "=" in kv)
    # every outcome is exercised
    assert int(counts["kept"]) > 1000 and int(counts["skipped"]) > 100 and int(counts["panics"]) > 100, r.stdout
