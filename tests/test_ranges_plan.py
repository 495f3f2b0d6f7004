"""Many ranges of seekable streams on the CPU: the plan of zstdlite_b200/csrc/zl_seek.h that turns a list of ranges into one batch
(tests/host/ranges_check.cpp), and zl_decompress_ranges / zstd_decompress_ranges failing loudly without a GPU."""
import ctypes as C
import os
import subprocess

import pytest

from tests.test_host_copy import ROOT, _cuda_include
from tests.test_seek_plan import seek_table


def test_ranges_plan(tmp_path):
    inc = _cuda_include()
    if inc is None:
        pytest.skip("cuda_runtime.h not found (the header includes it)")
    exe = str(tmp_path / "ranges_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-Wall", "-Wextra", "-Wno-unknown-pragmas", "-I", os.path.join(ROOT, "zstdlite_b200", "csrc"),
                           "-isystem", inc, os.path.join(ROOT, "tests", "host", "ranges_check.cpp"), "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "bad=0" in out.stdout, out.stdout + out.stderr


def test_ranges_calls_fail_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    import zstdlite_b200 as z
    from zstdlite_b200 import _lib
    L = _lib.lib()
    frame = open(os.path.join(ROOT, "tests", "golden", "data.json.zst"), "rb").read()
    s = frame + seek_table([(len(frame), 172, 0)], False)
    with pytest.raises(z.ZstdError):
        z.zstd_decompress_ranges(s, [(10, 20), (0, 172)])
    d = z.zstd_dctx()
    dst = C.create_string_buffer(4096)
    src = C.cast(C.c_char_p(s), C.c_void_p)
    srcs, sizes = (C.c_void_p * 1)(src), (C.c_size_t * 1)(len(s))
    offs, lens, caps, res = (C.c_size_t * 1)(0), (C.c_size_t * 1)(172), (C.c_size_t * 1)(4096), (C.c_size_t * 1)(0)
    dsts = (C.c_void_p * 1)(C.cast(dst, C.c_void_p))
    assert L.ZSTD_isError(L.zl_decompress_ranges(d._p, srcs, sizes, offs, lens, dsts, caps, res, 1, 0))
    assert L.zl_decompress_ranges(d._p, srcs, sizes, offs, lens, dsts, caps, res, 0, 0) == 0     # nothing to do
