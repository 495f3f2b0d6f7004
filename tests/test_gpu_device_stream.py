"""-m gpu tests of Zstandard streams decoded in device memory (zl_device_frames, zl_decompress_device, the tensor API).  The reference is
this library's own ZSTD_decompressDCtx on a host copy -- same return value for every stream and capacity, same bytes on success -- and,
where libzstd accepts the stream, libzstd itself.  Streams: libzstd at several levels, with checksums and a dictionary, frames without a
content size, zl_compress_split and zl_compress_seekable output, concatenations with skippable frames, a frame of more than ZL_IDX_W
blocks, magic look-alikes and a whole stream inside a raw block, every single structural fault, and 4 GiB in 65,536 frames."""
import ctypes as C
import struct

import numpy as np
import pytest

from tests.gpu_util import to_dev

pytestmark = pytest.mark.gpu

CONTENTSIZE_ERROR = 2**64 - 2
MAGIC = struct.pack("<I", 0xFD2FB528)


@pytest.fixture(scope="module")
def z():
    import torch
    assert torch.cuda.is_available()
    import zstdlite_b200 as zz
    return zz


def lib():
    from zstdlite_b200 import _lib
    return _lib.lib()


def host_decompress(dctx, s, cap):
    """(return value, bytes written) of this library's ZSTD_decompressDCtx on a host copy"""
    dst = C.create_string_buffer(max(1, cap))
    r = lib().ZSTD_decompressDCtx(dctx._p, dst, cap, s, len(s))
    return r, (dst.raw[:r] if not lib().ZSTD_isError(r) else None)


def device_decompress(dctx, s, cap):
    import torch
    src = to_dev(s)
    out = torch.empty(max(1, cap) + 64, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    r = lib().zl_decompress_device(dctx._p, C.c_void_p(out.data_ptr()), cap, C.c_void_p(src.data_ptr()), len(s))
    return r, (out[:r].cpu().numpy().tobytes() if not lib().ZSTD_isError(r) else None)


def host_walk(s):
    """the frames as ZSTD_findFrameCompressedSize / ZSTD_getFrameContentSize see them, or the walk's error"""
    L, out, pos = lib(), [], 0
    while len(s) - pos >= 5:
        rest = s[pos:]
        n = L.ZSTD_findFrameCompressedSize(rest, len(rest))
        if L.ZSTD_isError(n):
            return None
        out.append((pos, n, L.ZSTD_getFrameContentSize(rest, n)))
        pos += n
    return out if pos == len(s) else None


def device_frames(dctx, s):
    src = to_dev(s)
    L = lib()
    k = L.zl_device_frames(dctx._p, C.c_void_p(src.data_ptr()), len(s), None, None, None, 0)
    if L.ZSTD_isError(k):
        return k, None
    a = [(C.c_ulonglong * max(1, k))() for _ in range(3)]
    assert L.zl_device_frames(dctx._p, C.c_void_p(src.data_ptr()), len(s), a[0], a[1], a[2], k) == k
    return k, [(a[0][i], a[1][i], a[2][i]) for i in range(k)]


def same_as_host(z, s, dctx=None, caps=None):
    """zl_decompress_device == ZSTD_decompressDCtx for stream s at several capacities; returns the host result at the exact size"""
    dctx = dctx or z.zstd_dctx()
    total = lib().ZSTD_findDecompressedSize(s, len(s))
    size = total
    if total >= CONTENTSIZE_ERROR:                                         # frames without a content size: the decoded size, if any
        r, _ = host_decompress(dctx, s, 4 * len(s) + (1 << 20))
        size = r if not lib().ZSTD_isError(r) else 4 * len(s) + (1 << 20)
    first = None
    for cap in caps or (size, max(0, size - 1), size + 100):
        h = host_decompress(dctx, s, cap)
        d = device_decompress(dctx, s, cap)
        assert d[0] == h[0], (cap, z.error_name(d[0]) if z.is_error(d[0]) else d[0], z.error_name(h[0]) if z.is_error(h[0]) else h[0])
        assert d[1] == h[1], cap
        first = first or h
    return first


def libzstd_stream_frame(ref, data, level=3, checksum=False):
    """a libzstd frame written by ZSTD_compressStream2 without a pledged size: ZSTD_e_continue, then ZSTD_e_end -- no content size"""
    from zstdlite_b200 import _lib
    L = C.CDLL(ref._PATH)
    L.ZSTD_createCCtx.restype = C.c_void_p
    L.ZSTD_freeCCtx.argtypes = [C.c_void_p]
    L.ZSTD_CCtx_setParameter.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.ZSTD_CCtx_setParameter.restype = C.c_size_t
    L.ZSTD_compressStream2.argtypes = [C.c_void_p, C.POINTER(_lib.OutBuffer), C.POINTER(_lib.InBuffer), C.c_int]
    L.ZSTD_compressStream2.restype = C.c_size_t
    L.ZSTD_isError.argtypes = [C.c_size_t]
    c = L.ZSTD_createCCtx()
    L.ZSTD_CCtx_setParameter(c, 100, level)
    L.ZSTD_CCtx_setParameter(c, 201, 1 if checksum else 0)
    out = C.create_string_buffer(len(data) + (len(data) >> 7) + 4096)
    ob = _lib.OutBuffer(C.cast(out, C.c_void_p), len(out), 0)
    src = C.create_string_buffer(bytes(data), len(data))
    half = len(data) // 2
    for lo, hi, mode in ((0, half, 0), (half, len(data), 2)):
        ib = _lib.InBuffer(C.c_void_p(C.addressof(src) + lo), hi - lo, 0)
        while True:
            r = L.ZSTD_compressStream2(c, C.byref(ob), C.byref(ib), mode)
            assert not L.ZSTD_isError(r)
            if (mode == 0 and ib.pos == ib.size) or (mode == 2 and r == 0):
                break
    L.ZSTD_freeCCtx(c)
    f = out.raw[:ob.pos]
    assert lib().ZSTD_getFrameContentSize(f, len(f)) == 2**64 - 1
    return f


def skippable(payload, nibble=0):
    return struct.pack("<II", 0x184D2A50 + nibble, len(payload)) + payload


def raw_frame(content, blocks):
    """a frame of raw blocks (16 MiB window, 4-byte content size), content cut into `blocks` pieces"""
    cuts = np.linspace(0, len(content), blocks + 1).astype(int)
    body = b""
    for k in range(blocks):
        piece = content[cuts[k]:cuts[k + 1]]
        body += struct.pack("<I", (len(piece) << 3) | (1 if k == blocks - 1 else 0))[:3] + piece
    return MAGIC + bytes([0x80, 0x70]) + struct.pack("<I", len(content)) + body


def data_of(family, n, index=0):
    from zstdlite_b200 import corpus
    return corpus.make(family, n, index).tobytes()


@pytest.fixture(scope="module")
def streams(z, ref):
    """named streams; each is checked against the host path"""
    rng = np.random.default_rng(20261022)
    d = [data_of(f, 50000 + 7919 * k, k) for k, f in enumerate(("text", "rdf", "lowent", "rand", "rle"))]
    s = {}
    for lvl in (-3, 1, 3, 9, 19):
        s[f"libzstd_l{lvl}"] = b"".join(ref.compress(x, lvl, include_checksum=bool(lvl & 1)) for x in d)
    s["libzstd_unknown_size"] = b"".join(libzstd_stream_frame(ref, x, 3, checksum=k % 2 == 1) for k, x in enumerate(d))
    s["mixed_known_unknown"] = ref.compress(d[0], 3) + libzstd_stream_frame(ref, d[1]) + ref.compress(d[2], 3) + libzstd_stream_frame(ref, d[4])
    big = data_of("text", 3 << 20, 5)
    cc = z.zstd_cctx(level=3)
    s["split"] = z.zstd_compress(big, cctx=cc, frame_size=65536)
    s["seekable"] = z.zstd_compress(big, cctx=cc, frame_size=100000, seekable=True)
    s["with_skippable"] = (skippable(b"") + ref.compress(d[0], 3) + skippable(bytes(rng.integers(0, 256, 77, dtype=np.uint8)), 7)
                           + s["seekable"] + skippable(b"x" * 13, 15))
    s["skippable_only"] = skippable(b"abc") + skippable(b"", 3)
    s["empty_frame"] = ref.compress(b"", 3) + ref.compress(d[0][:100], 1)
    # a frame of more than ZL_IDX_W (1,024) blocks: the chain's walk is finished by the frontier
    s["long_frame"] = ref.compress(d[0], 3) + raw_frame(data_of("rand", 1500 * 20, 9), 1500) + ref.compress(d[1], 3)
    # ten frames of 1,100 blocks each: eight frontier rounds, then the serial walk finishes the chain
    s["many_long_frames"] = b"".join(raw_frame(data_of("rand", 1100 * 4, 20 + k), 1100) for k in range(10))
    # magic look-alikes in raw blocks, "magic then zeros", and a whole stream inside a raw block that ends exactly on the next frame
    inner = ref.compress(d[0][:3000], 3) + ref.compress(d[1][:2000], 3)
    looks = bytearray(data_of("rand", 40000, 3))
    for at in rng.integers(0, len(looks) - 8, 50):
        looks[at:at + 4] = MAGIC if at % 2 else struct.pack("<I", 0x184D2A53)
    looks[20000:20004] = MAGIC
    looks[20004:30000] = bytes(9996)
    s["lookalikes"] = raw_frame(bytes(looks), 3) + raw_frame(inner, 1) + ref.compress(d[2], 3)
    return s


NAMES = ["libzstd_l-3", "libzstd_l1", "libzstd_l3", "libzstd_l9", "libzstd_l19", "libzstd_unknown_size", "mixed_known_unknown", "split",
         "seekable", "with_skippable", "skippable_only", "empty_frame", "long_frame", "many_long_frames", "lookalikes"]


@pytest.mark.parametrize("name", NAMES)
def test_stream_matches_host_path(z, ref, streams, name):
    s = streams[name]
    r, out = same_as_host(z, s)
    assert not z.is_error(r), z.error_name(r)
    if name != "skippable_only":
        assert out == ref.decompress(s, cap=max(1, r + 4 * len(s)), all_frames=True)
    k, frames = device_frames(z.zstd_dctx(), s)
    want = host_walk(s)
    assert frames == want, name
    assert k == len(want)


def test_dictionary_stream(z, ref):
    from zstdlite_b200 import corpus
    objs = corpus.small_objects(400)
    dic = ref.train_dict(objs[:300], 4096)
    rc = ref.CCtx(level=3, dict=dic, include_checksum=True)
    s = b"".join(rc.compress(o) for o in objs[300:])
    r, out = same_as_host(z, s, dctx=z.zstd_dctx(dict=dic))
    assert out == b"".join(objs[300:])
    same_as_host(z, s)                                                     # without the dictionary: the same result both ways


def faults_of(s, frames):
    """(name, stream) for each single structural fault of a valid stream"""
    out = []
    for cut in sorted({1, 3, 4, 5, 7, len(s) // 3, len(s) // 2, len(s) - 5, len(s) - 1} | {o + 2 for o, _, _ in frames} | {o + n - 1 for o, n, _ in frames}):
        if 0 < cut < len(s):
            out.append((f"truncated at {cut}", s[:cut]))
    for t in range(1, 5):
        out.append((f"{t} trailing bytes", s + bytes([0x28, 0xB5, 0x2F, 0xFD])[:t]))
    for o, n, dsize in frames:
        if o:
            b = bytearray(s); b[o + 3] ^= 0x40
            out.append((f"non-magic at {o}", bytes(b)))
        if struct.unpack_from("<I", s, o)[0] == 0xFD2FB528:
            fhd = s[o + 4]
            single, did, fcs = (fhd >> 5) & 1, fhd & 3, fhd >> 6
            hs = 5 + (0 if single else 1) + (0, 1, 2, 4)[did] + ((1 if single else 0) if fcs == 0 else 1 << fcs)
            b = bytearray(s); b[o + hs] |= 6
            out.append((f"block type 3 at {o}", bytes(b)))
            b = bytearray(s); b[o + 4] |= 8
            out.append((f"FHD bit 3 at {o}", bytes(b)))
            if not single:
                b = bytearray(s); b[o + 5] = 0xFF
                out.append((f"window too large at {o}", bytes(b)))
    return out


@pytest.mark.parametrize("name", ["libzstd_l3", "with_skippable", "mixed_known_unknown", "long_frame", "lookalikes"])
def test_single_faults(z, streams, name):
    s = streams[name]
    dctx = z.zstd_dctx()
    for what, t in faults_of(s, host_walk(s)):
        total = lib().ZSTD_findDecompressedSize(s, len(s))
        cap = total if total < CONTENTSIZE_ERROR else 8 * len(s) + (1 << 20)
        h, d = host_decompress(dctx, t, cap), device_decompress(dctx, t, cap)
        assert d[0] == h[0], (what, z.error_name(d[0]), z.error_name(h[0]))
        assert d[1] == h[1], what
        w = host_walk(t)
        k, fr = device_frames(dctx, t)
        if w is None:
            assert z.is_error(k), what
        else:
            assert fr == w, what


def test_checksums(z, ref):
    x = data_of("text", 200000, 1)
    f = bytearray(ref.compress(x, 3, include_checksum=True))
    s = bytes(f) + ref.compress(x[:5000], 1, include_checksum=True)
    f[-1] ^= 1
    bad = bytes(f) + ref.compress(x[:5000], 1, include_checksum=True)
    for ignore in (False, True):
        dctx = z.zstd_dctx(validate_checksum=not ignore)
        r, out = same_as_host(z, s, dctx=dctx)
        assert out == x + x[:5000]
        r, _ = same_as_host(z, bad, dctx=dctx)
        assert z.is_error(r) != ignore
        if not ignore:
            assert z.error_name(r) == z.error_name(2**64 - 22)


def test_tiny_and_empty_sources(z, ref):
    dctx = z.zstd_dctx()
    f = ref.compress(b"hello", 3)
    for t in [b""] + [f[:k] for k in range(1, 5)] + [b"\x01\x02\x03\x04", b"\x50\x2A\x4D\x18"]:
        h = host_decompress(dctx, t, 100)
        if not t:
            import torch
            out = torch.empty(8, dtype=torch.uint8, device="cuda")
            d = lib().zl_decompress_device(dctx._p, C.c_void_p(out.data_ptr()), 100, None, 0)
            assert d == h[0] == 0
            assert lib().zl_device_frames(dctx._p, None, 0, None, None, None, 0) == 0
            continue
        d = device_decompress(dctx, t, 100)
        assert d[0] == h[0], t


def test_capacity_one_short_before_a_later_fault(z, ref, streams):
    s = streams["libzstd_l3"]
    total = lib().ZSTD_findDecompressedSize(s, len(s))
    same_as_host(z, s[:-3], caps=(total - 1, total))                     # dstSize_tooSmall comes first, then the truncation


def test_device_frames_cap_zero_and_arrays(z, streams):
    s = streams["with_skippable"]
    src = to_dev(s)
    L, dctx = lib(), z.zstd_dctx()
    k = L.zl_device_frames(dctx._p, C.c_void_p(src.data_ptr()), len(s), None, None, None, 0)
    want = host_walk(s)
    assert k == len(want)
    off = (C.c_ulonglong * k)()
    assert L.zl_device_frames(dctx._p, C.c_void_p(src.data_ptr()), len(s), off, None, None, k - 1) == k      # cap too small: nothing written
    assert list(off) == [0] * k
    assert L.zl_device_frames(dctx._p, C.c_void_p(src.data_ptr()), len(s), off, None, None, k) == k
    assert list(off) == [w[0] for w in want]
    assert [f[2] for f in z.zstd_frames(src[:len(s)])] == [None if w[2] == 2**64 - 1 else w[2] for w in want]


def test_tensor_api(z, ref, streams):
    import torch
    x = data_of("rdf", 1 << 20, 2)
    t = torch.from_numpy(np.frombuffer(x, dtype=np.uint8).copy()).cuda()
    for kw in ({}, {"frame_size": 100000}, {"frame_size": 65536, "seekable": True}):
        cc = z.zstd_cctx(level=3, include_checksum=True)
        dev = z.zstd_compress(t, cctx=cc, **kw)
        host = z.zstd_compress(x, cctx=cc, **kw)
        assert dev.is_cuda and dev.cpu().numpy().tobytes() == host, kw
        assert torch.equal(z.zstd_decompress(dev, all_frames=True), t), kw
        first = z.zstd_decompress(dev)
        assert first.cpu().numpy().tobytes() == z.zstd_decompress(host), kw
    assert z.zstd_compress(t[:0]).cpu().numpy().tobytes() == z.zstd_compress(b"")
    s = streams["mixed_known_unknown"]
    src = to_dev(s)[:len(s)]
    whole = z.zstd_decompress(src, all_frames=True)
    assert whole.cpu().numpy().tobytes() == ref.decompress(s, cap=4 * len(s) + (1 << 20), all_frames=True)
    first = z.zstd_decompress(src)
    assert torch.equal(first, whole[:first.numel()])
    unk = to_dev(streams["libzstd_unknown_size"])[:len(streams["libzstd_unknown_size"])]
    assert z.zstd_decompress(unk).numel() == 50000                       # a frame without content size is decoded, not refused
    out = torch.zeros(whole.numel() + 10, dtype=torch.uint8, device="cuda")
    v = z.zstd_decompress(src, all_frames=True, out=out)
    assert v.data_ptr() == out.data_ptr() and torch.equal(v, whole)
    # a frame without content size that compresses far better than 4x, into an `out` of exactly its size
    zeros = libzstd_stream_frame(ref, bytes(1 << 20))
    zt = to_dev(zeros)[:len(zeros)]
    exact = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    for all_frames in (False, True):
        exact.fill_(7)
        v = z.zstd_decompress(zt, all_frames=all_frames, out=exact)
        assert v.numel() == 1 << 20 and int(v.max()) == 0, all_frames
    assert z.zstd_decompress(zt).numel() == 1 << 20                        # no out: the output grows to fit
    sk = to_dev(streams["with_skippable"])[:len(streams["with_skippable"])]
    assert z.zstd_decompress(sk).numel() == 0                             # a leading skippable frame: empty, like bytes
    with pytest.raises(z.ZstdError):
        z.zstd_decompress(src, type="string")


def test_4gib_of_64kib_frames(z, ref):
    """65,536 frames of 64 KiB of the benchmark's mix in device memory: the same bytes as zl_decompress_batch with the boundaries known"""
    import torch
    from zstdlite_b200 import corpus
    fb, nf = 65536, 65536
    plain, _, _ = corpus.device_mixed_slabs(nf, fb, (("text", 0.4), ("rdf", 0.4), ("lowent", 0.1), ("rand", 0.1)), index=11)
    plain = plain.reshape(-1)
    n = plain.numel()
    L, cc = lib(), z.zstd_cctx(level=3)
    cap = nf * L.ZSTD_compressBound(fb)
    dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    sizes = (C.c_size_t * nf)()
    torch.cuda.synchronize()
    r = L.zl_compress_split(cc._p, C.c_void_p(dst.data_ptr()), cap, C.c_void_p(plain.data_ptr()), n, fb, sizes, 1)
    assert not z.is_error(r), z.error_name(r)
    s = dst[:r]
    dctx = z.zstd_dctx()
    fr = z.zstd_frames(s, dctx=dctx)
    coff = np.concatenate(([0], np.cumsum(np.array(sizes[:], dtype=np.int64))))
    assert len(fr) == nf and [f[0] for f in fr[:5]] == coff[:5].tolist() and fr[-1][0] == coff[-2] and all(f[2] == fb for f in fr)
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    rr = L.zl_decompress_device(dctx._p, C.c_void_p(out.data_ptr()), n, C.c_void_p(s.data_ptr()), r)
    assert rr == n, z.error_name(rr) if z.is_error(rr) else rr
    ref_out = torch.empty(n, dtype=torch.uint8, device="cuda")
    plan = z.BatchPlan([s.data_ptr() + int(o) for o in coff[:-1]], sizes[:], [ref_out.data_ptr() + k * fb for k in range(nf)], [fb] * nf)
    res = plan.decompress(dctx)
    assert all(int(x) == fb for x in res)
    assert torch.equal(out, ref_out) and torch.equal(out, plain)
    rng = np.random.default_rng(1)
    host = s.cpu().numpy()
    for k in [int(x) for x in rng.integers(0, nf, 16)]:
        frame = host[coff[k]:coff[k + 1]].tobytes()
        assert ref.decompress(frame) == out[k * fb:(k + 1) * fb].cpu().numpy().tobytes(), k
