"""The frame index of a stream in device memory, on the CPU: the per-thread bodies of zstdlite_b200/csrc/zl_stream_index.h run with the
kernels' pass structure against the serial host walk (tests/host/stream_index_check.cpp), and zl_device_frames / zl_decompress_device /
the tensor API failing loudly without a GPU."""
import ctypes as C
import os
import subprocess

import pytest

from tests.test_host_copy import ROOT, _cuda_include


def test_stream_index(tmp_path):
    inc = _cuda_include()
    if inc is None:
        pytest.skip("cuda_runtime.h not found (the header includes it)")
    exe = str(tmp_path / "stream_index_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-Wall", "-Wextra", "-Wno-unknown-pragmas", "-I", os.path.join(ROOT, "zstdlite_b200", "csrc"),
                           "-isystem", inc, os.path.join(ROOT, "tests", "host", "stream_index_check.cpp"), "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "bad=0" in out.stdout, out.stdout + out.stderr


def test_device_stream_calls_fail_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    import zstdlite_b200 as z
    from zstdlite_b200 import _lib
    L = _lib.lib()
    frame = open(os.path.join(ROOT, "tests", "golden", "data.json.zst"), "rb").read()
    src = C.cast(C.c_char_p(frame), C.c_void_p)
    d = z.zstd_dctx()
    dst = C.create_string_buffer(4096)
    assert L.ZSTD_isError(L.zl_device_frames(d._p, src, len(frame), None, None, None, 0))
    assert L.ZSTD_isError(L.zl_decompress_device(d._p, C.cast(dst, C.c_void_p), 4096, src, len(frame)))
    assert L.ZSTD_isError(L.zl_device_frames(None, src, len(frame), None, None, None, 0))
    assert L.ZSTD_isError(L.zl_decompress_device(None, C.cast(dst, C.c_void_p), 4096, src, len(frame)))
    with pytest.raises(z.ZstdError):
        z.zstd_frames(frame)                                              # a bytes source has no device to index on
    with pytest.raises(z.ZstdError):
        z.zstd_decompress(frame, out=bytearray(10))                       # out= is for CUDA sources
