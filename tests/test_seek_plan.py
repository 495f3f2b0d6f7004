"""Seekable streams on the CPU: the seek table and range plan of zstdlite_b200/csrc/zl_seek.h (tests/host/seek_check.cpp), the host-only
calls of the C ABI (zl_seekable_frames on host memory, zl_compress_seekable_bound), and the compute calls failing loudly without a GPU."""
import ctypes as C
import os
import struct
import subprocess

import pytest

from tests.test_host_copy import ROOT, _cuda_include


def test_seek_plan(tmp_path):
    inc = _cuda_include()
    if inc is None:
        pytest.skip("cuda_runtime.h not found (the header includes it)")
    exe = str(tmp_path / "seek_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", "-Wall", "-Wextra", "-Wno-unknown-pragmas", "-I", os.path.join(ROOT, "zstdlite_b200", "csrc"),
                           "-isystem", inc, os.path.join(ROOT, "tests", "host", "seek_check.cpp"), "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "bad=0" in out.stdout, out.stdout + out.stderr


def seek_table(entries, checksums):
    """the seek table frame of Zstandard's seekable format for [(compressed_size, decompressed_size, checksum)]"""
    body = b"".join(struct.pack("<III", c, d, k) if checksums else struct.pack("<II", c, d) for c, d, k in entries)
    footer = struct.pack("<IBI", len(entries), 0x80 if checksums else 0, 0x8F92EAB1)
    return struct.pack("<II", 0x184D2A5E, len(body) + len(footer)) + body + footer


def _frames(L, src, cap):
    cs, ds, ck, has = (C.c_uint * max(1, cap))(), (C.c_uint * max(1, cap))(), (C.c_uint * max(1, cap))(), C.c_int(-1)
    n = L.zl_seekable_frames(src, len(src), 0, cs, ds, ck, cap, C.byref(has))
    return n, list(cs)[:cap], list(ds)[:cap], list(ck)[:cap], has.value


def test_seekable_frames_on_host_memory():
    import zstdlite_b200 as z
    from zstdlite_b200 import _lib
    L = _lib.lib()
    frame = open(os.path.join(ROOT, "tests", "golden", "data.json.zst"), "rb").read()      # 172 bytes of content, with a trailer
    trailer = struct.unpack("<I", frame[-4:])[0]
    for checksums in (False, True):
        s = frame * 3 + seek_table([(len(frame), 172, trailer)] * 3, checksums)
        assert L.zl_seekable_frames(s, len(s), 0, None, None, None, 0, None) == 3
        n, cs, ds, ck, has = _frames(L, s, 3)
        assert (n, cs, ds, has) == (3, [len(frame)] * 3, [172] * 3, int(checksums))
        assert ck == ([trailer] * 3 if checksums else [0] * 3)
        n, cs, _, _, _ = _frames(L, s, 2)                           # too small a capacity: N only, nothing written
        assert n == 3 and cs == [0, 0]
        assert z.zstd_seek_table(s) == [(len(frame), 172, trailer if checksums else None)] * 3
        assert z.zstd_seek_table(bytearray(s)) == z.zstd_seek_table(memoryview(s))
    err = lambda name: (1 << 64) - {"prefix_unknown": 10, "corruption_detected": 20}[name]
    s = frame + seek_table([(len(frame), 172, 0)], False)
    assert L.zl_seekable_frames(frame, len(frame), 0, None, None, None, 0, None) == err("prefix_unknown")
    assert L.zl_seekable_frames(s[1:], len(s) - 1, 0, None, None, None, 0, None) == err("corruption_detected")
    assert L.zl_seekable_frames(s[:-9] + struct.pack("<IBI", 1, 0x40, 0x8F92EAB1), len(s), 0, None, None, None, 0, None) == err("corruption_detected")
    with pytest.raises(z.ZstdError, match="Unknown frame descriptor"):
        z.zstd_seek_table(frame)


def test_seekable_bound():
    from zstdlite_b200 import _lib
    L = _lib.lib()
    B = L.ZSTD_compressBound
    assert L.zl_compress_seekable_bound(0, 1000, 0) == B(0) + 8 + 8 + 9          # one empty frame
    assert L.zl_compress_seekable_bound(2500, 1000, 0) == 2 * B(1000) + B(500) + 8 + 3 * 8 + 9
    assert L.zl_compress_seekable_bound(2000, 1000, 1) == 2 * (B(1000) + 4) + 8 + 2 * 12 + 9
    assert L.zl_compress_seekable_bound(1 << 30, 1 << 30, 0) == B(1 << 30) + 25
    for bad in (0, (1 << 30) + 1):
        assert L.ZSTD_getErrorName(L.zl_compress_seekable_bound(100, bad, 0)) == b"Parameter is out of bound"
    assert L.ZSTD_isError(L.zl_compress_seekable_bound(0x8000001, 1, 0))         # more than 0x8000000 frames


def test_seekable_compute_calls_fail_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    import zstdlite_b200 as z
    from zstdlite_b200 import _lib
    L = _lib.lib()
    frame = open(os.path.join(ROOT, "tests", "golden", "data.json.zst"), "rb").read()
    s = frame + seek_table([(len(frame), 172, 0)], False)
    with pytest.raises(z.ZstdError):
        z.zstd_compress(b"no silent CPU path" * 100, frame_size=256, seekable=True)
    with pytest.raises(z.ZstdError):
        z.zstd_decompress_range(s, 10, 20)
    c = z.zstd_cctx()
    dst = C.create_string_buffer(4096)
    assert L.ZSTD_isError(L.zl_compress_seekable(c._p, dst, 4096, b"x" * 100, 100, 10, 0))
    d = z.zstd_dctx()
    assert L.ZSTD_isError(L.zl_decompress_range(d._p, dst, 4096, s, len(s), 0, 172, 0))
