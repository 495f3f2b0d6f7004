"""ctypes driver of oracle/libzl_cpubench.so (oracle/cpu_bench.c).  TEST / BENCH INFRA ONLY.

Times the system's libzstd (libzstd.so.1) frame-parallel on the host cores:
one context per thread, frames pulled from a shared counter, no Python in the timed region.
Used by bench.py (`cpu_baseline` leg and `--impl reference`) and by nothing in the product.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_PATH = os.path.join(_HERE, "libzl_cpubench.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        from oracle import ref
        ref.lib()                                      # the harness links the same libzstd.so.1: refuse an unchecked release
        if not os.path.exists(_PATH):
            subprocess.check_call(["make", "-s", "-C", _HERE, "libzl_cpubench.so"])
        L = C.CDLL(_PATH, mode=os.RTLD_LOCAL)
        vp, sz = C.c_void_p, C.c_size_t
        L.zlb_run.argtypes = [C.c_int, vp, vp, vp, vp, vp, vp, vp, sz, C.c_int, C.c_int, vp, sz, C.c_int]
        L.zlb_run.restype = C.c_double
        L.zlb_run_workers.argtypes = [vp, sz, vp, sz, C.c_int, C.c_int, C.c_int, vp]
        L.zlb_run_workers.restype = C.c_double
        _lib = L
    return _lib


def _offsets(sizes):
    offs = np.zeros(len(sizes), dtype=np.uint64)
    if len(sizes) > 1:
        offs[1:] = np.cumsum(np.asarray(sizes[:-1], dtype=np.uint64))
    return offs


class FrameSet:
    """Packed frames: `blob` (uint8 array), per-frame sizes.  Offsets are derived (back to back)."""

    def __init__(self, blob, sizes):
        self.blob = np.ascontiguousarray(blob, dtype=np.uint8)
        self.sizes = np.asarray(sizes, dtype=np.uint64)
        self.offs = _offsets(self.sizes)


def run(mode, src, dst_caps, threads, level=3, checksum=False, dict=None, passes=1):
    """mode 'decompress' | 'compress' over FrameSet `src`; dst_caps per frame.

    Returns (best seconds over `passes`, result sizes array, dst blob, dst offsets)."""
    L = lib()
    n = len(src.sizes)
    caps = np.asarray(dst_caps, dtype=np.uint64)
    doffs = _offsets(caps)
    dst = np.zeros(int(caps.sum()) + 64, dtype=np.uint8)
    dst[::4096] = 1                                    # fault the pages in before the timed region
    res = np.zeros(n, dtype=np.uint64)
    d = np.frombuffer(dict, dtype=np.uint8) if dict else None
    best = None
    for _ in range(passes):
        t = L.zlb_run(1 if mode == "compress" else 0, src.blob.ctypes.data, src.offs.ctypes.data, src.sizes.ctypes.data,
                      dst.ctypes.data, doffs.ctypes.data, caps.ctypes.data, res.ctypes.data, n, int(level),
                      1 if checksum else 0, d.ctypes.data if d is not None else None, len(d) if d is not None else 0, int(threads))
        if t < 0:
            raise RuntimeError("reference libzstd reported an error inside the CPU baseline")
        best = t if best is None else min(best, t)
    return best, res, dst, doffs


def run_workers(buf, level=3, workers=0, passes=2):
    """ONE frame from `buf` (uint8 array) with ZSTD_c_nbWorkers = workers (the reference's num_threads semantics, src/cctx.c:269-277).
    Returns (best seconds, frame size)."""
    L = lib()
    buf = np.ascontiguousarray(buf, dtype=np.uint8)
    cap = buf.size + (buf.size >> 7) + 1024
    dst = np.zeros(cap, dtype=np.uint8)
    dst[::4096] = 1
    out = C.c_size_t(0)
    t = L.zlb_run_workers(buf.ctypes.data, buf.size, dst.ctypes.data, cap, int(level), int(workers), int(passes), C.byref(out))
    if t < 0:
        raise RuntimeError("reference libzstd reported an error inside the CPU baseline (nbWorkers)")
    return t, int(out.value)
