"""-m gpu tests of seekable streams (Zstandard's seekable format): the writer (zl_compress_seekable) checked against libzstd
(oracle/ref.py), the C restatement's XXH64 and zl_compress_split; range decoding (zl_decompress_range) of foreign streams over a grid
of ranges from host and device memory; that only the touched frames are decoded; the table's checksums and sizes; the tensor API."""
import ctypes as C
import struct

import numpy as np
import pytest

from tests.test_seek_plan import seek_table

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def z():
    import torch
    assert torch.cuda.is_available()
    import zstdlite_b200 as zz
    return zz


def lib():
    from zstdlite_b200 import _lib
    return _lib.lib()


def walk(ref, stream):
    """libzstd's frame walk: the frames in front of the table frame, and the table frame"""
    L, frames, pos = ref.lib(), [], 0
    while pos < len(stream):
        if struct.unpack_from("<I", stream, pos)[0] == 0x184D2A5E:
            break
        rest = stream[pos:]
        n = L.ZSTD_findFrameCompressedSize(rest, len(rest))
        assert not L.ZSTD_isError(n)
        frames.append(stream[pos:pos + n])
        pos += n
    return frames, stream[pos:]


def compress_seekable(z, data, frame_size, level=3, checksum=False, device=False):
    import torch
    from tests.gpu_util import to_dev
    L, c = lib(), z.zstd_cctx(level=level, include_checksum=checksum)
    cap = L.zl_compress_seekable_bound(len(data), frame_size, 1 if checksum else 0)
    if not device:
        dst = C.create_string_buffer(cap)
        r = L.zl_compress_seekable(c._p, dst, cap, data, len(data), frame_size, 0)
        assert not z.is_error(r), z.error_name(r)
        return dst.raw[:r]
    src, dst = to_dev(data), torch.empty(cap, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    r = L.zl_compress_seekable(c._p, dst.data_ptr(), cap, src.data_ptr(), len(data), frame_size, 1)
    assert not z.is_error(r), z.error_name(r)
    return dst[:r].cpu().numpy().tobytes()


def compress_split(z, data, frame_size, level, checksum):
    L, c = lib(), z.zstd_cctx(level=level, include_checksum=checksum)
    cap = L.zl_compress_seekable_bound(len(data), frame_size, 1 if checksum else 0)
    dst = C.create_string_buffer(cap)
    r = L.zl_compress_split(c._p, dst, cap, data, len(data), frame_size, None, 0)
    assert not z.is_error(r), z.error_name(r)
    return dst.raw[:r]


@pytest.mark.parametrize("family", ["text", "rdf", "rle", "rand"])
@pytest.mark.parametrize("shape", [(300000, 65536), (262144, 65536), (1000, 65536), (0, 4096), (70000, 1000)])
@pytest.mark.parametrize("checksum", [False, True])
@pytest.mark.parametrize("device", [False, True])
def test_writer(z, ref, restate, family, shape, checksum, device):
    from zstdlite_b200 import corpus
    n, fs = shape
    data = corpus.make(family, n, 5).tobytes()
    s = compress_seekable(z, data, fs, 3, checksum, device)
    assert ref.decompress(s, all_frames=True, cap=n) == data
    frames, table = walk(ref, s)
    chunks = [data[i:i + fs] for i in range(0, n, fs)] or [b""]
    entries = z.zstd_seek_table(s)
    assert len(frames) == len(chunks) == len(entries)
    assert len(table) == 8 + len(frames) * (12 if checksum else 8) + 9
    for f, ch, (cs, ds, ck) in zip(frames, chunks, entries):
        assert (cs, ds) == (len(f), len(ch)) and restate.frame_content_size(f) == len(ch)
        assert ck == ((restate.xxh64(ch) & 0xFFFFFFFF) if checksum else None)
    assert s[:len(s) - len(table)] == compress_split(z, data, fs, 3, checksum)
    # every Zstandard reader skips the table: ZSTD_decompressDCtx and zstd_decompress(all_frames=True) read the whole input
    assert z.zstd_decompress(s, all_frames=True) == data
    if not device:
        assert z.zstd_compress(data, frame_size=fs, seekable=True, include_checksum=checksum) == s


def test_writer_rejects_frame_sizes(z):
    L, c = lib(), z.zstd_cctx()
    dst = C.create_string_buffer(1 << 16)
    for fs in (0, (1 << 30) + 1):
        assert L.ZSTD_getErrorName(L.zl_compress_seekable(c._p, dst, 1 << 16, b"abc" * 100, 300, fs, 0)) == b"Parameter is out of bound"
    # the frames fit but the table does not
    s = compress_seekable(z, b"abc" * 1000, 1000)
    assert L.ZSTD_getErrorName(L.zl_compress_seekable(c._p, dst, len(s) - 1, b"abc" * 1000, 3000, 1000, 0)) == b"Destination buffer is too small"


def foreign(ref, restate, data, cuts, checksums, dict=None):
    """libzstd frames of data[cuts[k]:cuts[k+1]] at several levels, every other one with a trailer, and a table built here"""
    frames, entries = [], []
    for k in range(len(cuts) - 1):
        ch = data[cuts[k]:cuts[k + 1]]
        f = ref.CCtx(level=(1, 3, 9, 19)[k % 4], include_checksum=k % 2 == 0, dict=dict).compress(ch)
        frames.append(f)
        entries.append((len(f), len(ch), restate.xxh64(ch) & 0xFFFFFFFF))
    return b"".join(frames) + seek_table(entries, checksums), entries


def grid(cuts):
    """the offsets and lengths of the range grid: every frame boundary +-1, mid-frame; 0, 1, inside a frame, across 2, many, to and past the end"""
    total = cuts[-1]
    offs = {0, total, total // 3}
    for k, c in enumerate(cuts):
        offs |= {c - 1, c, c + 1}
        if k + 1 < len(cuts):
            offs.add((c + cuts[k + 1]) // 2)
    for o in sorted(x for x in offs if 0 <= x <= total):
        later = [c - o for c in cuts if c > o]
        lens = {0, 1, 7, total - o, total - o + 100, 1 << 40}
        if len(later) >= 2:
            lens |= {later[1], later[1] + 1, later[0] + 1}
        if later:
            lens |= {max(1, later[0] // 2), later[-1] - 1}
        for n in sorted(lens):
            yield o, n


def cuts_for(rng, total, nframes):
    inner = sorted(int(x) for x in rng.integers(0, total + 1, nframes - 1))
    return [0] + inner + [total]


@pytest.mark.parametrize("checksums", [False, True])
@pytest.mark.parametrize("with_dict", [False, True])
def test_foreign_streams_range_grid(z, ref, restate, checksums, with_dict):
    import torch
    from zstdlite_b200 import corpus
    rng = np.random.default_rng(7 + with_dict)
    if with_dict:
        objs = corpus.small_objects(3000)
        dic = ref.train_dict(objs[:2000], 8192)
        data = b"".join(objs[2000:2200])
    else:
        dic = None
        data = corpus.make("text", 150000, 3).tobytes() + corpus.make("rdf", 150000, 4).tobytes()
    cuts = cuts_for(rng, len(data), 12)
    cuts[3] = cuts[4]                                                     # a frame of zero bytes
    s, _ = foreign(ref, restate, data, cuts, checksums, dic)
    dctx = z.zstd_dctx(dict=dic)
    dsrc = torch.from_numpy(np.frombuffer(s, dtype=np.uint8).copy()).cuda()
    count = 0
    for o, n in grid(cuts):
        want = data[o:o + n]
        assert z.zstd_decompress_range(s, o, n, dctx=dctx) == want, (o, n)
        got = z.zstd_decompress_range(dsrc, o, n, dctx=dctx)
        assert got.is_cuda and got.cpu().numpy().tobytes() == want, (o, n)
        count += 1
    assert count > 200
    for src in (s, dsrc):
        with pytest.raises(z.ZstdError, match="Parameter is out of bound"):
            z.zstd_decompress_range(src, len(data) + 1, 1, dctx=dctx)


def corrupt_block_type(frame):
    """the first block of the frame gets the reserved block type 3: decoding it must fail"""
    L = lib()
    from zstdlite_b200 import _lib
    fh = _lib.FrameHeader()
    assert L.ZSTD_getFrameHeader(C.byref(fh), frame, len(frame)) == 0
    b = bytearray(frame)
    b[fh.headerSize] |= 0x06
    return bytes(b)


@pytest.mark.parametrize("device", [False, True])
def test_only_touched_frames_are_decoded(z, ref, restate, device):
    import torch
    from zstdlite_b200 import corpus
    data = corpus.make("text", 8 * 20000, 9).tobytes()
    cuts = list(range(0, len(data) + 1, 20000))
    frames = [ref.compress(data[a:b], 3) for a, b in zip(cuts, cuts[1:])]
    frames[5] = corrupt_block_type(frames[5])
    s = b"".join(frames) + seek_table([(len(f), 20000, 0) for f in frames], False)
    src = torch.from_numpy(np.frombuffer(s, dtype=np.uint8).copy()).cuda() if device else s
    get = lambda o, n: (lambda r: r.cpu().numpy().tobytes() if device else r)(z.zstd_decompress_range(src, o, n))
    for o, n in ((0, 100000), (10, 19990), (99998, 2), (120000, 40000), (130000, 100), (0, 1)):
        assert get(o, n) == data[o:o + n], (o, n)
    for o, n in ((100000, 20000), (110000, 5), (99999, 3), (0, 160000)):
        with pytest.raises(z.ZstdError):
            get(o, n)


@pytest.mark.parametrize("device", [False, True])
def test_table_checksums(z, ref, restate, device):
    import torch
    from zstdlite_b200 import corpus
    data = corpus.make("rdf", 6 * 30000, 2).tobytes()
    cuts = list(range(0, len(data) + 1, 30000))
    s, entries = foreign(ref, restate, data, cuts, True)             # frames 0, 2, 4 carry a trailer; 1, 3, 5 do not
    for k in (1, 2):
        bad = list(entries)
        bad[k] = (bad[k][0], bad[k][1], bad[k][2] ^ 0x10)
        sb = s[:len(s) - len(seek_table(entries, True))] + seek_table(bad, True)
        src = torch.from_numpy(np.frombuffer(sb, dtype=np.uint8).copy()).cuda() if device else sb
        get = lambda o, n, **kw: (lambda r: r.cpu().numpy().tobytes() if device else r)(z.zstd_decompress_range(src, o, n, **kw))
        lo = cuts[k]
        for o, n in ((lo, 30000), (lo + 10, 5), (lo - 5, 10), (0, len(data))):
            with pytest.raises(z.ZstdError, match="doesn't match checksum"):
                get(o, n)
            assert get(o, n, validate_checksum=False) == data[o:o + n]
        other = cuts[k + 2]
        assert get(other, 30000) == data[other:other + 30000]


@pytest.mark.parametrize("device", [False, True])
def test_wrong_table_sizes_are_errors(z, ref, restate, device):
    import torch
    from zstdlite_b200 import corpus
    data = corpus.make("text", 5 * 40000, 6).tobytes()
    cuts = list(range(0, len(data) + 1, 40000))
    s, entries = foreign(ref, restate, data, cuts, False)
    body = s[:len(s) - len(seek_table(entries, False))]
    cases = []
    for k in (0, 2, 4):
        for dd in (1, -1, 1000):
            e = list(entries); e[k] = (e[k][0], e[k][1] + dd, 0); cases.append((k, e))
    for k in (0, 2, 3):
        for dc in (1, -1, 7):                                         # sizes still add up: the frame's neighbour takes the difference
            e = list(entries); j = k + 1
            e[k] = (e[k][0] + dc, e[k][1], 0); e[j] = (e[j][0] - dc, e[j][1], 0); cases.append((k, e))
        e = list(entries); e[k] = (e[k][0] + 1, e[k][1], 0); cases.append((k, e))         # they do not
    for k, e in cases:
        sb = body + seek_table(e, False)
        src = torch.from_numpy(np.frombuffer(sb, dtype=np.uint8).copy()).cuda() if device else sb
        o = sum(x[1] for x in e[:k])
        for n in (e[k][1] if e[k][1] > 0 else 1, 3):
            with pytest.raises(z.ZstdError):
                z.zstd_decompress_range(src, o, n)


def test_device_round_trip_and_out(z, ref, restate):
    import torch
    from zstdlite_b200 import corpus
    data = corpus.make("text", 1 << 20, 8).tobytes()
    s = compress_seekable(z, data, 65536, checksum=True)
    dsrc = torch.from_numpy(np.frombuffer(s, dtype=np.uint8).copy()).cuda()
    assert z.zstd_seek_table(dsrc) == z.zstd_seek_table(s)
    for o, n in ((0, 1 << 20), (1000, 200000), (65535, 2), ((1 << 20) - 1, 10)):
        host = z.zstd_decompress_range(s, o, n)
        dev = z.zstd_decompress_range(dsrc, o, n)
        assert dev.is_cuda and dev.dtype == torch.uint8 and dev.cpu().numpy().tobytes() == host == data[o:o + n]
    out = torch.full((300000,), 7, dtype=torch.uint8, device="cuda")
    got = z.zstd_decompress_range(dsrc, 5000, 250000, out=out)
    assert got.data_ptr() == out.data_ptr() and got.numel() == 250000
    assert out[:250000].cpu().numpy().tobytes() == data[5000:255000] and int(out[250000:].min()) == 7
    with pytest.raises(z.ZstdError, match="Destination buffer is too small"):
        z.zstd_decompress_range(dsrc, 0, 400000, out=out)
    assert z.zstd_decompress_range(s, 10, 20, type="string") == data[10:30].decode()


def test_large_device_stream(z):
    """a device-resident stream of a few hundred MiB: written on the device, a 1 MiB range and the full range read back on the device"""
    import torch
    from zstdlite_b200 import corpus
    fb = 65536
    plain, _, _ = corpus.device_mixed_slabs(4096, fb, (("text", 0.4), ("rdf", 0.4), ("lowent", 0.1), ("rand", 0.1)), index=17)
    plain = plain.reshape(-1)
    n = plain.numel()
    L, c = lib(), z.zstd_cctx(level=3, include_checksum=True)
    cap = L.zl_compress_seekable_bound(n, fb, 1)
    dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    r = L.zl_compress_seekable(c._p, dst.data_ptr(), cap, plain.data_ptr(), n, fb, 1)
    assert not z.is_error(r), z.error_name(r)
    s = dst[:r]
    table = z.zstd_seek_table(s)
    assert len(table) == 4096 and sum(t[1] for t in table) == n and all(t[2] is not None for t in table)
    dctx = z.zstd_dctx()
    rng = np.random.default_rng(3)
    for o in [int(x) for x in rng.integers(0, n - (1 << 20), 4)] + [n - (1 << 20)]:
        got = z.zstd_decompress_range(s, o, 1 << 20, dctx=dctx)
        assert torch.equal(got, plain[o:o + (1 << 20)]), o
    full = z.zstd_decompress_range(s, 0, n, dctx=dctx)
    assert torch.equal(full, plain)
    assert torch.equal(z.zstd_decompress_range(s, n - 5, 1 << 30, dctx=dctx), plain[n - 5:])
