"""The line rules k_bed_fields / k_bed_judge run on the GPU (the __host__ __device__ core in csrc/bed_parse_core.cuh) against the host
packer rbh::Windows::pack_text, on the CPU: seeded random BED files with '\\r\\n', lone '\\r', runs of blank lines, no final newline,
'#' lines anywhere, a first line of another field count, rows of 2 / 4 / 5 fields, empty fields, spaces inside fields, '+5',
20-digit numbers and u64 overflow, absent contigs, names that exist only as query names, empty ids and duplicate rows."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "rustybam_b200", "host")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("native") / "bed_parse_check")
    srcs = [os.path.join(HOST, f) for f in sorted(os.listdir(HOST)) if f.endswith(".cpp") and f != "rb_main.cpp"]
    subprocess.check_call(
        ["g++", "-O1", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "rustybam_b200", "csrc"), "-I", HOST, "-I",
         os.path.join(ROOT, "include"), "-o", exe, os.path.join(ROOT, "tests", "native", "bed_parse_check.cpp")] + srcs + ["-lz"])
    return exe


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_line_core_matches_host_packer(harness, seed):
    r = subprocess.run([harness, str(seed), "20000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "FAIL=0" in r.stdout
    counts = dict(kv.split("=") for kv in r.stdout.split() if "=" in kv)
    # every outcome is exercised
    assert int(counts["kept"]) > 1000 and int(counts["skipped"]) > 100 and int(counts["absent"]) > 100, r.stdout
    assert int(counts["comments"]) > 100 and int(counts["files"]) > 5, r.stdout
