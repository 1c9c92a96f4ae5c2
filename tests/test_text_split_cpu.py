"""The line split of rb_liftover_text (csrc/text_split.hpp), on the CPU: a text cut into 1-9 byte ranges at arbitrary places, some of
them empty, must be planned into per-device buffers that hold every line exactly once, whole and in order."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("native") / "text_split_check")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "rustybam_b200", "csrc"), "-o", exe,
                           os.path.join(ROOT, "tests", "native", "text_split_check.cpp")])
    return exe


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_split_plan_keeps_every_line_once(harness, seed):
    r = subprocess.run([harness, str(seed), "20000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "FAIL=0" in r.stdout
    counts = dict(kv.split("=") for kv in r.stdout.split() if "=" in kv)
    assert int(counts["cases"]) > 20000 and int(counts["lines"]) > 100000, r.stdout
