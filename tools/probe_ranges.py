"""Many ranges of a seekable stream in one call (DESIGN.md §2.2, "Many ranges"): a device-resident seekable stream of the benchmark's
corpus mix -- 4 GiB of content made on the device, 64 KiB frames, level 3 -- read with one zl_decompress_ranges call against the same
ranges through zl_decompress_range one by one.  Reports medians of alternating repetitions of
  (a) 1,000 ranges of 1 MiB at seeded random offsets: one call against the loop;
  (b) 10,000 ranges of 4 KiB at seeded random offsets (a data-loader step): one call against the loop (the loop is timed once: ~20 s);
  (c) 4,096 contiguous 1 MiB ranges from byte 1,000 -- every range has two edge frames, each shared with its neighbour -- against
      zl_decompress_batch over all the table's frames: the cost of the plan, the scratch and the copy-out,
with the card's name and power limit.  Every call synchronises before it returns, so host clocks time whole calls.
usage: python tools/probe_ranges.py [--gib 4] [--reps 5] [--json PATH]"""
import argparse
import ctypes as C
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import zstdlite_b200 as z  # noqa: E402
from zstdlite_b200 import _lib, corpus  # noqa: E402
from tools.probe_seekable import FB, MIX, card, check, timed  # noqa: E402


class Ranges:
    """the argument arrays of one zl_decompress_ranges call over stream s, the ranges packed back to back into out"""

    def __init__(self, s, offs, lens, out):
        n = len(offs)
        self.n, self.offs, self.lens = n, offs, lens
        at = np.concatenate(([0], np.cumsum(lens))).astype(np.uint64)
        assert int(at[-1]) <= out.numel()
        self.at = at
        self.a = [np.full(n, s.data_ptr(), dtype=np.uint64), np.full(n, s.numel(), dtype=np.uint64), np.asarray(offs, dtype=np.uint64),
                  np.asarray(lens, dtype=np.uint64), out.data_ptr() + at[:-1], np.asarray(lens, dtype=np.uint64), np.zeros(n, dtype=np.uint64)]
        pp, psz = C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)
        self.args = [x.ctypes.data_as(pp if k in (0, 4) else psz) for k, x in enumerate(self.a)]

    def run(self, L, dctx):
        check(L.zl_decompress_ranges(dctx._p, *self.args, self.n, 1), "zl_decompress_ranges")
        res = self.a[6]
        assert (res == np.asarray(self.lens, dtype=np.uint64)).all(), "a range failed"

    def loop(self, L, dctx, s):
        for k in range(self.n):
            L.zl_decompress_range(dctx._p, int(self.a[4][k]), int(self.lens[k]), s.data_ptr(), s.numel(), int(self.offs[k]), int(self.lens[k]), 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=4.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "probe_ranges needs a CUDA device"
    L = _lib.lib()
    nf = int(a.gib * (1 << 30)) // FB
    plain, _, _ = corpus.device_mixed_slabs(nf, FB, MIX, index=11)
    plain = plain.reshape(-1)
    n = plain.numel()
    cctx = z.zstd_cctx(level=3)
    cap = check(L.zl_compress_seekable_bound(n, FB, 0), "bound")
    dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    s = dst[:check(L.zl_compress_seekable(cctx._p, dst.data_ptr(), cap, plain.data_ptr(), n, FB, 1), "zl_compress_seekable")]
    table = z.zstd_seek_table(s)
    assert len(table) == nf and sum(t[1] for t in table) == n
    dctx = z.zstd_dctx()
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    rng = np.random.default_rng(20261022)
    med = lambda v: float(np.median(v))
    ms = lambda v: [round(x, 3) for x in v]
    r = {"content_bytes": n, "frames": nf, "frame_bytes": FB, "level": 3}

    # (a) and (b): one call against the loop
    for key, count, size in (("a_1000x1MiB", 1000, 1 << 20), ("b_10000x4KiB", 10000, 4096)):
        offs = [int(x) for x in rng.integers(0, n - size, count)]
        R = Ranges(s, offs, [size] * count, out)
        R.run(L, dctx)
        for k in range(0, count, max(1, count // 50)):
            o, at = offs[k], int(R.at[k])
            assert torch.equal(out[at:at + size], plain[o:o + size]), (key, k)
        loop_reps = a.reps if count <= 1000 else 1
        if loop_reps > 1:
            R.loop(L, dctx, s)                                                                  # warm-up of the loop
        one, loop = [], []
        for rep in range(a.reps):                                                               # alternating
            one += timed(lambda: R.run(L, dctx), 1)
            if rep < loop_reps:
                loop += timed(lambda: R.loop(L, dctx, s), 1)
        r[key] = {"ranges": count, "range_bytes": size, "one_call_ms": ms(one), "loop_ms": ms(loop),
                  "one_call_median_ms": med(one), "loop_median_ms": med(loop), "speedup": med(loop) / med(one)}

    # (c): contiguous ranges with shared edge frames against the batch over every frame
    start, size, count = 1000, 1 << 20, 4096
    offs = [start + k * size for k in range(count)]
    lens = [max(0, min(size, n - o)) for o in offs]
    R = Ranges(s, offs, lens, out)
    coff = np.concatenate([[0], np.cumsum([t[0] for t in table])]).astype(np.int64)
    doff = np.concatenate([[0], np.cumsum([t[1] for t in table])]).astype(np.int64)
    plan = z.BatchPlan([s.data_ptr() + int(o) for o in coff[:-1]], [t[0] for t in table], [out.data_ptr() + int(o) for o in doff[:-1]],
                       [t[1] for t in table])

    def batch():
        res = plan.decompress(dctx)
        assert res[0] == FB

    batch()
    assert torch.equal(out, plain)
    R.run(L, dctx)
    assert torch.equal(out[:n - start], plain[start:])
    d_batch, d_ranges = [], []
    for _ in range(a.reps):
        d_batch += timed(batch, 1)
        d_ranges += timed(lambda: R.run(L, dctx), 1)
    r["c_4096x1MiB_contiguous"] = {"ranges": count, "first_offset": start, "batch_ms": ms(d_batch), "ranges_ms": ms(d_ranges),
                                   "batch_median_ms": med(d_batch), "ranges_median_ms": med(d_ranges),
                                   "ranges_over_batch": med(d_ranges) / med(d_batch)}
    name, power = card()
    r = {"card": name, "power_limit": power, **r}
    print(json.dumps(r, indent=1))
    if a.json:
        with open(a.json, "w") as fh:
            json.dump(r, fh, indent=1)


if __name__ == "__main__":
    main()
