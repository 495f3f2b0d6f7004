"""Host-side plan of a compress batch on the CPU (zstdlite_b200/csrc/zl_enc_plan.h): wave and part cuts, slot sizes, descriptors, far
tables and frame headers, placement and staged upload of host buffers, gather tables and the frames and chunks of zl_compress_split, for
the benchmark's shapes, every planning switch and random batches."""
import os
import subprocess

import pytest

from tests.test_host_copy import ROOT, _cuda_include


def test_enc_plan(tmp_path):
    inc = _cuda_include()
    if inc is None:
        pytest.skip("cuda_runtime.h not found (the header includes it)")
    exe = str(tmp_path / "enc_plan_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-Wall", "-Wextra", "-Wno-unknown-pragmas", "-I", os.path.join(ROOT, "zstdlite_b200", "csrc"),
                           "-isystem", inc, os.path.join(ROOT, "tests", "host", "enc_plan_check.cpp"), "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "bad=0" in out.stdout, out.stdout + out.stderr
