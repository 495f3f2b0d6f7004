"""Streams in device memory (DESIGN.md §2.3): the frame index on the device and the whole-stream decode, against the decode with every
frame boundary known and against today's workaround (copy the stream to the host, walk it with ZSTD_findFrameCompressedSize, then
zl_decompress_batch).  Inputs, all device-resident:
  (a) 4 GiB of the benchmark's mix in 64 KiB frames at level 3 (zl_compress_split; the input of tools/probe_ranges.py), and
      I1's count pass alone on as many zero bytes;
  (b) one 1.5 GiB frame written by libzstd (level 1): more than ZL_IDX_W blocks, so its walk is the frontier's; the index and the
      host walk are timed whatever the decode returns, and the existing engine is tried on libzstd frames of growing size;
  (c) 256 MiB of raw-block frames whose content is "magic then zeros" every 256 bytes: a million look-alike candidates.
Each timing is the median of --reps alternating repetitions; every call synchronises before it returns, so host clocks time whole
calls.  "workaround" and "walk_on_host" include a Python loop of one ctypes call per frame and, for "workaround", building the batch
from Python lists; "batch_known" is planned before it is timed.  The card's name and power limit are read in the same run.
usage: python tools/probe_device_stream.py [--gib 4] [--reps 5] [--json PATH]"""
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


def frames_of(L, dctx, s):
    k = check(L.zl_device_frames(dctx._p, C.c_void_p(s.data_ptr()), s.numel(), None, None, None, 0), "zl_device_frames")
    a = [np.zeros(max(1, k), dtype=np.uint64) for _ in range(3)]
    p = C.POINTER(C.c_ulonglong)
    check(L.zl_device_frames(dctx._p, C.c_void_p(s.data_ptr()), s.numel(), *[x.ctypes.data_as(p) for x in a], k), "zl_device_frames")
    return a[0][:k], a[1][:k], a[2][:k]


def case(L, dctx, s, plain, reps):
    n = plain.numel()
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    coff, csize, dsize = frames_of(L, dctx, s)
    doff = np.concatenate(([0], np.cumsum(dsize.astype(np.int64))))
    plan = z.BatchPlan([s.data_ptr() + int(o) for o in coff], [int(x) for x in csize], [out.data_ptr() + int(o) for o in doff[:-1]],
                       [int(x) for x in dsize])

    def index():
        check(L.zl_device_frames(dctx._p, C.c_void_p(s.data_ptr()), s.numel(), None, None, None, 0), "zl_device_frames")

    def device():
        assert check(L.zl_decompress_device(dctx._p, C.c_void_p(out.data_ptr()), n, C.c_void_p(s.data_ptr()), s.numel()), "decode") == n

    def batch():
        res = plan.decompress(dctx)
        assert int(res[0]) == int(dsize[0])

    def walk():
        host = s.cpu().numpy()
        base, pos, total = host.ctypes.data, 0, host.size
        offs, sizes = [], []
        while pos < total:
            k = check(L.ZSTD_findFrameCompressedSize(base + pos, total - pos), "walk")
            offs.append(pos); sizes.append(k); pos += k
        return offs, sizes, [L.ZSTD_getFrameContentSize(base + o, k) for o, k in zip(offs, sizes)]

    def workaround():
        offs, sizes, caps = walk()
        at = np.concatenate(([0], np.cumsum(caps))).astype(np.int64)
        res = z.BatchPlan([s.data_ptr() + o for o in offs], sizes, [out.data_ptr() + int(a) for a in at[:-1]], caps).decompress(dctx)
        assert int(res[0]) == caps[0]

    r = {"stream_bytes": s.numel(), "content_bytes": n, "frames": len(coff)}
    host = s.cpu().numpy()
    hout = np.empty(max(1, n), dtype=np.uint8)
    hr = L.ZSTD_decompressDCtx(dctx._p, hout.ctypes.data, n, host.ctypes.data, host.size)
    dr = L.zl_decompress_device(dctx._p, C.c_void_p(out.data_ptr()), n, C.c_void_p(s.data_ptr()), s.numel())
    del host, hout
    assert dr == hr, (z.error_name(dr) if z.is_error(dr) else dr, z.error_name(hr) if z.is_error(hr) else hr)     # the contract
    decodes = dr == n
    if decodes:
        assert torch.equal(out, plain)
        out.zero_()
        batch()
        assert torch.equal(out, plain)
    else:
        r["decode_result"] = z.error_name(dr)
    fns = {"index": index, "walk_on_host": walk}
    if decodes:
        fns.update({"decompress_device": device, "batch_known": batch, "workaround": workaround})
    t = {k: [] for k in fns}
    for fn in fns.values():
        fn()                                                              # warm-up
    for _ in range(reps):                                                 # alternating
        for k, fn in fns.items():
            t[k] += timed(fn, 1)
    for k, v in t.items():
        r[k + "_ms"] = [round(x, 3) for x in v]
        r[k + "_median_ms"] = float(np.median(v))
    if decodes:
        r["index_over_batch"] = r["index_median_ms"] / r["batch_known_median_ms"]
    return r


def engine_bracket(L, dctx, ref, data):
    """ZSTD_decompressDCtx (host copies, the existing engine) on single libzstd frames of growing prefixes of `data`"""
    out = {}
    for mib in (256, 512, 768, 1024, 1280, 1536):
        x = data[:mib << 20]
        for lvl in (1, 3):
            f = ref.compress(x, lvl)
            dst = np.empty(len(x), dtype=np.uint8)
            r = L.ZSTD_decompressDCtx(dctx._p, dst.ctypes.data, len(x), f, len(f))
            out[f"{mib}MiB_level{lvl}"] = "ok" if r == len(x) and dst.tobytes() == x else (z.error_name(r) if z.is_error(r) else f"{r} bytes, differ")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=4.0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "probe_device_stream needs a CUDA device"
    from oracle import ref
    L = _lib.lib()
    dctx = z.zstd_dctx()
    r = {}

    # (a)
    nf = int(a.gib * (1 << 30)) // FB
    plain, _, _ = corpus.device_mixed_slabs(nf, FB, MIX, index=11)
    plain = plain.reshape(-1)
    cap = nf * L.ZSTD_compressBound(FB)
    dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    cctx = z.zstd_cctx(level=3)
    s = dst[:check(L.zl_compress_split(cctx._p, dst.data_ptr(), cap, plain.data_ptr(), plain.numel(), FB, None, 1), "split")]
    r["a_64KiB_frames"] = case(L, dctx, s, plain, a.reps)
    # what I1's count pass alone costs on as many bytes: a stream of zeros has no candidate, so the index stops after it
    zeros = torch.zeros(s.numel(), dtype=torch.uint8, device="cuda")
    assert L.zl_device_frames(dctx._p, C.c_void_p(zeros.data_ptr()), zeros.numel(), None, None, None, 0) == 2**64 - 10
    t = timed(lambda: L.zl_device_frames(dctx._p, C.c_void_p(zeros.data_ptr()), zeros.numel(), None, None, None, 0), a.reps)
    r["a_64KiB_frames"]["i1_count_pass_only_median_ms"] = float(np.median(t))
    del dst, s, plain, zeros

    # (b)
    big = corpus.device_mixed_slabs(int(1.5 * (1 << 30)) // FB, FB, MIX, index=5)[0].reshape(-1)
    host = big.cpu().numpy().tobytes()
    f = ref.compress(host, 1)
    s = torch.from_numpy(np.frombuffer(f, dtype=np.uint8).copy()).cuda()
    r["b_one_1.5GiB_libzstd_frame"] = case(L, dctx, s, big, a.reps)
    del s, big, f
    r["b_engine_bracket"] = engine_bracket(L, dctx, ref, host)
    del host

    # (c)
    blk, per = 128 << 10, 8
    content = np.zeros(blk, dtype=np.uint8)
    content.reshape(-1, 256)[:, :4] = np.frombuffer(b"\x28\xB5\x2F\xFD", dtype=np.uint8)
    frame = bytearray(b"\x28\xB5\x2F\xFD\xA0" + (blk * per).to_bytes(4, "little"))      # single segment, 4-byte content size
    for k in range(per):
        frame += ((blk << 3) | (1 if k == per - 1 else 0)).to_bytes(3, "little") + content.tobytes()
    nfr = (256 << 20) // (blk * per)
    s = torch.from_numpy(np.frombuffer(bytes(frame) * nfr, dtype=np.uint8).copy()).cuda()
    plain = torch.from_numpy(np.tile(content, per * nfr)).cuda()
    r["c_256MiB_lookalikes"] = case(L, dctx, s, plain, a.reps)

    name, power = card()
    r = {"card": name, "power_limit": power, **r}
    print(json.dumps(r, indent=1))
    if a.json:
        with open(a.json, "w") as fh:
            json.dump(r, fh, indent=1)


if __name__ == "__main__":
    main()
