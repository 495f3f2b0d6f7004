"""Seekable streams on one GPU (DESIGN.md, "Seekable streams"): a device-resident seekable stream of the benchmark's corpus mix -- 4 GiB of
content made on the device, 64 KiB frames, level 3 -- written by zl_compress_seekable and read back by zl_decompress_range.  Reports
  * zl_decompress_range(0, total) against zl_decompress_batch over the same frames (the difference is the table read and the plan),
  * the per-call time of 1 MiB ranges at seeded random offsets,
  * writer throughput: zl_compress_seekable against zl_compress_split on the same input,
with the card's name and power limit.  Every call synchronises before it returns, so host clocks time whole calls.
usage: python tools/probe_seekable.py [--gib 4] [--ranges 200] [--json PATH]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import zstdlite_b200 as z  # noqa: E402
from zstdlite_b200 import _lib, corpus  # noqa: E402

MIX = (("text", 0.4), ("rdf", 0.4), ("lowent", 0.1), ("rand", 0.1))      # bench.py's mix
FB = 64 << 10


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True)
    return torch.cuda.get_device_name(), (q.stdout.strip().split(", ")[-1] if q.returncode == 0 else "unknown")


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return ts


def check(r, what):
    if z.is_error(r):
        raise RuntimeError(f"{what}: {z.error_name(r)}")
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=4.0)
    ap.add_argument("--ranges", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "probe_seekable needs a CUDA device"
    L = _lib.lib()
    nf = int(a.gib * (1 << 30)) // FB
    plain, _, _ = corpus.device_mixed_slabs(nf, FB, MIX, index=11)
    plain = plain.reshape(-1)
    n = plain.numel()
    cctx = z.zstd_cctx(level=3)
    cap = check(L.zl_compress_seekable_bound(n, FB, 0), "bound")
    dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    size = {}

    def seekable():
        size["seekable"] = check(L.zl_compress_seekable(cctx._p, dst.data_ptr(), cap, plain.data_ptr(), n, FB, 1), "zl_compress_seekable")

    def split():
        size["split"] = check(L.zl_compress_split(cctx._p, dst.data_ptr(), cap, plain.data_ptr(), n, FB, None, 1), "zl_compress_split")

    split(); seekable()                                                                         # warm-up
    w_seek, w_split = [], []
    for _ in range(a.reps):                                                                     # alternating
        w_split += timed(split, 1)
        w_seek += timed(seekable, 1)
    s = dst[:size["seekable"]]
    table = z.zstd_seek_table(s)
    assert len(table) == nf and sum(t[1] for t in table) == n
    coff = np.concatenate([[0], np.cumsum([t[0] for t in table])]).astype(np.int64)
    doff = np.concatenate([[0], np.cumsum([t[1] for t in table])]).astype(np.int64)
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    dctx = z.zstd_dctx()
    plan = z.BatchPlan([s.data_ptr() + int(o) for o in coff[:-1]], [t[0] for t in table], [out.data_ptr() + int(o) for o in doff[:-1]], [t[1] for t in table])

    def batch():
        res = plan.decompress(dctx)
        assert res[0] == FB

    def whole():
        check(L.zl_decompress_range(dctx._p, out.data_ptr(), n, s.data_ptr(), s.numel(), 0, n, 1), "zl_decompress_range")

    batch(); whole()
    assert torch.equal(out, plain)
    d_batch, d_range = [], []
    for _ in range(a.reps):
        d_batch += timed(batch, 1)
        d_range += timed(whole, 1)
    rng = np.random.default_rng(20261022)
    offs = [int(x) for x in rng.integers(0, n - (1 << 20), a.ranges)]
    small = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    for o in offs[:8]:                                                                          # warm-up and check
        check(L.zl_decompress_range(dctx._p, small.data_ptr(), 1 << 20, s.data_ptr(), s.numel(), o, 1 << 20, 1), "range")
        assert torch.equal(small, plain[o:o + (1 << 20)])
    t_ranges = []
    for o in offs:
        t0 = time.perf_counter()
        L.zl_decompress_range(dctx._p, small.data_ptr(), 1 << 20, s.data_ptr(), s.numel(), o, 1 << 20, 1)
        t_ranges.append((time.perf_counter() - t0) * 1e3)
    name, power = card()
    med = lambda v: float(np.median(v))
    r = {"card": name, "power_limit": power, "content_bytes": n, "frames": nf, "frame_bytes": FB, "level": 3,
         "stream_bytes": size["seekable"], "table_bytes": size["seekable"] - size["split"],
         "write_ms": {"zl_compress_split": [round(x, 2) for x in w_split], "zl_compress_seekable": [round(x, 2) for x in w_seek]},
         "write_GBps_median": {"zl_compress_split": n / med(w_split) / 1e6, "zl_compress_seekable": n / med(w_seek) / 1e6},
         "decode_ms": {"zl_decompress_batch": [round(x, 2) for x in d_batch], "zl_decompress_range_whole": [round(x, 2) for x in d_range]},
         "decode_GBps_median": {"zl_decompress_batch": n / med(d_batch) / 1e6, "zl_decompress_range_whole": n / med(d_range) / 1e6},
         "range_1MiB_ms": {"calls": len(t_ranges), "median": med(t_ranges), "mean": float(np.mean(t_ranges)),
                           "p10": float(np.percentile(t_ranges, 10)), "p90": float(np.percentile(t_ranges, 90))}}
    print(json.dumps(r, indent=1))
    if a.json:
        with open(a.json, "w") as fh:
            json.dump(r, fh, indent=1)


if __name__ == "__main__":
    main()
