"""-m gpu tests of many ranges of seekable streams in one call (zl_decompress_ranges, zstd_decompress_ranges): every item's result and
bytes equal a separate zl_decompress_range call and the data, for libzstd-written streams and our own, from host and device memory;
several streams in one call; errors that fail only the items they concern; the tensor API; a large device-resident stream."""
import ctypes as C

import numpy as np
import pytest

from tests.test_gpu_seekable import compress_seekable, corrupt_block_type, cuts_for, foreign, grid, lib
from tests.test_seek_plan import seek_table

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def z():
    import torch
    assert torch.cuda.is_available()
    import zstdlite_b200 as zz
    return zz


def dev_copy(b):
    import torch
    return torch.from_numpy(np.frombuffer(b, dtype=np.uint8).copy()).cuda()


def addr(src):
    return src.data_ptr() if hasattr(src, "data_ptr") else C.cast(C.c_char_p(src), C.c_void_p).value


def call_ranges(dctx, items, device):
    """items: [(src, offset, length, capacity)] -> (results, the bytes of each item's destination up to min(result, capacity))"""
    import torch
    L, n = lib(), len(items)
    at = np.concatenate(([0], np.cumsum([it[3] for it in items]))).astype(np.int64)
    if device:
        out = torch.empty(max(1, int(at[-1])), dtype=torch.uint8, device="cuda")
        dsts = [out.data_ptr() + int(at[i]) for i in range(n)]
    else:
        out = C.create_string_buffer(max(1, int(at[-1])))
        dsts = [C.addressof(out) + int(at[i]) for i in range(n)]
    torch.cuda.synchronize()
    srcs = (C.c_void_p * n)(*[addr(it[0]) for it in items])
    sizes = (C.c_size_t * n)(*[(it[0].numel() if device else len(it[0])) for it in items])
    offs, lens = (C.c_size_t * n)(*[it[1] for it in items]), (C.c_size_t * n)(*[it[2] for it in items])
    caps, res = (C.c_size_t * n)(*[it[3] for it in items]), (C.c_size_t * n)()
    r = L.zl_decompress_ranges(dctx._p, srcs, sizes, offs, lens, (C.c_void_p * n)(*dsts), caps, res, n, 1 if device else 0)
    assert r == 0, L.ZSTD_getErrorName(r)
    raw = out.cpu().numpy().tobytes() if device else out.raw
    got = [raw[int(at[i]):int(at[i]) + (min(res[i], items[i][3]) if not L.ZSTD_isError(res[i]) else 0)] for i in range(n)]
    return list(res), got


def call_single(dctx, src, o, n, cap, device):
    import torch
    L = lib()
    if device:
        out = torch.empty(max(1, cap), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        r = L.zl_decompress_range(dctx._p, out.data_ptr(), cap, src.data_ptr(), src.numel(), o, n, 1)
        return r, (out.cpu().numpy().tobytes()[:r] if not L.ZSTD_isError(r) else b"")
    out = C.create_string_buffer(max(1, cap))
    r = L.zl_decompress_range(dctx._p, out, cap, src, len(src), o, n, 0)
    return r, (out.raw[:r] if not L.ZSTD_isError(r) else b"")


def check_against_single(dctx, items, device, datas):
    """every item: the same result as zl_decompress_range alone and, when it succeeds, the data's bytes"""
    L = lib()
    res, got = call_ranges(dctx, items, device)
    for (src, o, n, cap), r, g, data in zip(items, res, got, datas):
        r1, g1 = call_single(dctx, src, o, n, cap, device)
        assert r == r1, (o, n, cap, L.ZSTD_getErrorName(r), L.ZSTD_getErrorName(r1))
        if data is not None and not L.ZSTD_isError(r):
            assert g == g1 == data[o:o + n], (o, n)
    return res


@pytest.mark.parametrize("device", [False, True])
@pytest.mark.parametrize("checksums", [False, True])
@pytest.mark.parametrize("with_dict", [False, True])
def test_range_grid_in_one_call(z, ref, restate, device, checksums, with_dict):
    from zstdlite_b200 import corpus
    rng = np.random.default_rng(11 + with_dict + 2 * checksums)
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
    src = dev_copy(s) if device else s
    dctx = z.zstd_dctx(dict=dic)
    pairs = list(grid(cuts))
    pairs += [pairs[int(i)] for i in rng.integers(0, len(pairs), len(pairs) // 4)]          # duplicates
    rng.shuffle(pairs)
    items = [(src, o, n, max(0, min(n, len(data) - o))) for o, n in pairs]
    res = check_against_single(dctx, items, device, [data] * len(items))
    assert sum(not z.is_error(r) for r in res) > 200


@pytest.mark.parametrize("device", [False, True])
def test_own_streams_many_ranges(z, device):
    from zstdlite_b200 import corpus
    data = corpus.make("text", 1 << 20, 8).tobytes()
    s = compress_seekable(z, data, 65536, checksum=True)
    src = dev_copy(s) if device else s
    rng = np.random.default_rng(5)
    pairs = [(int(o), int(n)) for o, n in zip(rng.integers(0, len(data), 300), rng.integers(0, 200000, 300))]
    pairs += [(65536 * k - 10, 20) for k in range(1, 16)] + [(65536 * k, 65536) for k in range(16)] + [(0, len(data))] * 2
    items = [(src, o, n, max(0, min(n, len(data) - o))) for o, n in pairs]
    check_against_single(z.zstd_dctx(), items, device, [data] * len(items))


@pytest.mark.parametrize("device", [False, True])
def test_several_streams_interleaved(z, ref, restate, device):
    """a stream with table checksums, one without (two engine calls), and a copy of the first at another address, in one call"""
    from zstdlite_b200 import corpus
    rng = np.random.default_rng(21)
    da = corpus.make("rdf", 200000, 1).tobytes()
    db = corpus.make("text", 170000, 2).tobytes()
    sa, _ = foreign(ref, restate, da, cuts_for(rng, len(da), 9), True)
    sb, _ = foreign(ref, restate, db, cuts_for(rng, len(db), 7), False)
    if device:
        a, b, a2 = dev_copy(sa), dev_copy(sb), dev_copy(sa)
    else:
        a, b, a2 = sa, sb, bytes(bytearray(sa))
        assert addr(a) != addr(a2)
    streams = [(a, da), (b, db), (a2, da)]
    items, datas = [], []
    for k in range(400):
        src, data = streams[k % 3]
        o = int(rng.integers(0, len(data) + 1))
        n = int(rng.integers(0, 60000))
        items.append((src, o, n, max(0, min(n, len(data) - o))))
        datas.append(data)
    res = check_against_single(z.zstd_dctx(), items, device, datas)
    assert all(not z.is_error(r) for r in res)


@pytest.mark.parametrize("device", [False, True])
def test_errors_fail_only_their_items(z, ref, restate, device):
    from zstdlite_b200 import corpus
    L = lib()
    data = corpus.make("text", 6 * 30000, 6).tobytes()
    cuts = list(range(0, len(data) + 1, 30000))
    good, entries = foreign(ref, restate, data, cuts, True)
    body = good[:len(good) - len(seek_table(entries, True))]
    frames = [body[sum(e[0] for e in entries[:k]):sum(e[0] for e in entries[:k + 1])] for k in range(6)]
    # frame 1 corrupted; frame 3's table checksum wrong; frame 4's Decompressed_Size wrong
    corrupt = b"".join(frames[:1] + [corrupt_block_type(frames[1])] + frames[2:]) + seek_table(entries, True)
    bad_sum = list(entries); bad_sum[3] = (bad_sum[3][0], bad_sum[3][1], bad_sum[3][2] ^ 1)
    wrong_sum = body + seek_table(bad_sum, True)
    bad_size = list(entries); bad_size[4] = (bad_size[4][0], bad_size[4][1] + 7, bad_size[4][2])
    wrong_size = body + seek_table(bad_size, True)
    broken = body + seek_table(entries, True)[:-5] + bytes([0x84]) + seek_table(entries, True)[-4:]
    mk = dev_copy if device else (lambda b: b)
    srcs = {name: mk(b) for name, b in (("good", good), ("corrupt", corrupt), ("sum", wrong_sum), ("size", wrong_size), ("broken", broken))}
    f = lambda k: cuts[k]
    cases = [  # (stream, offset, length, capacity, expected error, "*" for the decoder's own, or None)
        ("corrupt", f(1) + 5, 10, 10, "*"), ("corrupt", f(0), 60000, 60000, "*"),
        ("corrupt", f(0) + 3, 1000, 1000, None), ("corrupt", f(2), 30000, 30000, None), ("corrupt", f(2) - 1, 2, 2, "*"),
        ("sum", f(3) + 10, 100, 100, "Restored data doesn't match checksum"), ("sum", f(2), 90000, 90000, "Restored data doesn't match checksum"),
        ("sum", f(0), 90000, 90000, None), ("sum", f(4), 1000, 1000, None),
        ("size", f(4) + 100, 50, 50, "Data corruption detected"), ("size", f(5) - 5, 10, 10, "Data corruption detected"), ("size", f(0), 1000, 1000, None),
        ("broken", 0, 100, 100, "Data corruption detected"), ("broken", f(3), 10, 10, "Data corruption detected"),
        ("good", 0, 1000, 999, "Destination buffer is too small"), ("good", len(data) + 1, 1, 1, "Parameter is out of bound"),
        ("good", len(data), 10, 0, None), ("good", f(1) - 10, 30020, 30020, None), ("good", 0, len(data), len(data), None),
    ]
    order = list(range(len(cases))) * 2
    np.random.default_rng(2).shuffle(order)
    items = [(srcs[cases[k][0]], cases[k][1], cases[k][2], cases[k][3]) for k in order]
    res = check_against_single(z.zstd_dctx(), items, device, [data] * len(items))
    for k, r in zip(order, res):
        want = cases[k][4]
        if want is None:
            assert not z.is_error(r), (cases[k], z.error_name(r))
        else:
            assert z.is_error(r) and want in ("*", L.ZSTD_getErrorName(r).decode()), (cases[k], z.error_name(r) if z.is_error(r) else r)
    # without checksum validation the wrong table checksum is no error
    res, got = call_ranges(z.zstd_dctx(validate_checksum=False), [(srcs["sum"], f(3) + 10, 100, 100), (srcs["sum"], f(2), 90000, 90000)], device)
    assert res == [100, 90000] and got == [data[f(3) + 10:f(3) + 110], data[f(2):f(2) + 90000]]


def test_tensor_api(z, ref, restate):
    import torch
    from zstdlite_b200 import corpus
    data = corpus.make("text", 400000, 4).tobytes()
    s = compress_seekable(z, data, 65536, checksum=True)
    dsrc = dev_copy(s)
    ranges = [(0, 10), (65530, 20), (100, 0), (len(data) - 5, 100), (1000, 200000), (65530, 20)]
    want = [data[o:o + n] for o, n in ranges]
    got = z.zstd_decompress_ranges(dsrc, ranges)
    assert len(got) == len(ranges) and all(g.is_cuda and g.dtype == torch.uint8 for g in got)
    assert [g.cpu().numpy().tobytes() for g in got] == want
    base = got[0].untyped_storage().data_ptr()                            # views into one tensor, back to back in request order
    pos = 0
    for g, w in zip(got, want):
        assert g.untyped_storage().data_ptr() == base and g.storage_offset() == pos
        pos += len(w)
    assert z.zstd_decompress_ranges(s, ranges) == want
    assert z.zstd_decompress_ranges(s, [(10, 20), (5, 3)], type="string") == [data[10:30].decode(), data[5:8].decode()]
    assert z.zstd_decompress_ranges(s, []) == [] and z.zstd_decompress_ranges(dsrc, []) == []
    total = sum(len(w) for w in want)
    out = torch.full((total + 100,), 7, dtype=torch.uint8, device="cuda")
    got = z.zstd_decompress_ranges(dsrc, ranges, out=out)
    assert [g.cpu().numpy().tobytes() for g in got] == want and got[0].data_ptr() == out.data_ptr()
    assert out[:total].cpu().numpy().tobytes() == b"".join(want) and int(out[total:].min()) == 7
    with pytest.raises(z.ZstdError, match="Destination buffer is too small"):
        z.zstd_decompress_ranges(dsrc, ranges, out=out[:total - 1])
    with pytest.raises(z.ZstdError, match=r"zstd_decompress_ranges\(\): range 2: Parameter is out of bound"):
        z.zstd_decompress_ranges(dsrc, [(0, 1), (5, 5), (len(data) + 1, 1), (len(data) + 2, 1)])
    frames = z.zstd_seek_table(s)
    bad = bytearray(s)
    at = frames[0][0] + frames[1][0]                                      # frame 2
    bad[at:at + frames[2][0]] = corrupt_block_type(bytes(bad[at:at + frames[2][0]]))
    for src in (bytes(bad), dev_copy(bytes(bad))):
        with pytest.raises(z.ZstdError, match=r"zstd_decompress_ranges\(\): range 17: "):
            z.zstd_decompress_ranges(src, [(0, 100)] * 17 + [(2 * 65536 + 5, 10)] + [(0, 5)])


def test_large_device_stream_many_ranges(z):
    """a device-resident stream of a few hundred MiB: 1,000 random ranges of 1 byte to 4 MiB, duplicates included, in one call"""
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
    rng = np.random.default_rng(9)
    lens = np.exp(rng.uniform(0, np.log(4 << 20), 900)).astype(np.int64)
    ranges = [(int(rng.integers(0, n)), int(k)) for k in lens]
    ranges += [ranges[int(i)] for i in rng.integers(0, len(ranges), 100)]
    rng.shuffle(ranges)
    got = z.zstd_decompress_ranges(s, ranges, dctx=z.zstd_dctx())
    assert len(got) == 1000
    for (o, k), g in zip(ranges, got):
        assert torch.equal(g, plain[o:o + k]), (o, k)
