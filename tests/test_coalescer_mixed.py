"""The C++ query coalescer under mixed (Limit, SearchSize) traffic (tests/cpp/coalescer_mixed_test.cpp):
one batch takes every waiting request whatever its parameters, each result equals the request served
alone, an invalid request fails alone. The driver is compiled into a temporary directory."""
import os
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
LIB = ROOT / "semadb_b200" / "lib"


@pytest.mark.gpu
def test_coalescer_mixed(tmp_path):
    exe = tmp_path / "coalescer_mixed_test"
    subprocess.run([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-Wall", "-Wextra", "-pthread", "-o", str(exe),
                    str(ROOT / "tests" / "cpp" / "coalescer_mixed_test.cpp"), f"-L{LIB}", "-lsemadb_b200",
                    f"-Wl,-rpath,{LIB}"], check=True, capture_output=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr + r.stdout
    assert "coalescer_mixed_test: ok" in r.stdout
