"""Host-side plan of a batched decode on the CPU (zstdlite_b200/csrc/zl_batch_plan.h): slice counts and cuts, frame order, copy runs of host
buffers, arena shares, descriptors and the copies back from staging, for the benchmark's batch shapes, every planning switch and random
batches."""
import os
import subprocess

import pytest

from tests.test_host_copy import ROOT, _cuda_include


def test_batch_plan(tmp_path):
    inc = _cuda_include()
    if inc is None:
        pytest.skip("cuda_runtime.h not found (the header includes it)")
    exe = str(tmp_path / "batch_plan_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-Wall", "-Wextra", "-Wno-unknown-pragmas", "-I", os.path.join(ROOT, "zstdlite_b200", "csrc"),
                           "-isystem", inc, os.path.join(ROOT, "tests", "host", "batch_plan_check.cpp"), "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "bad=0" in out.stdout, out.stdout + out.stderr
