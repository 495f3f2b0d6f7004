"""-m gpu parity tests for the CUDA decoder: byte-exact against libzstd (oracle/ref.py)
and the C restatement, through the C ABI (zl_decompress_batch / ZSTD_decompressDCtx)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def z():
    import torch
    assert torch.cuda.is_available()
    import zstdlite_b200 as zz
    return zz


def test_kat_data_json(z):
    """reference KAT man/figures/data.json.zst <-> README.md:199-205 (committed under tests/golden)."""
    c = open(os.path.join(GOLD, "data.json.zst"), "rb").read()
    want = open(os.path.join(GOLD, "data.json"), "rb").read()
    assert z.zstd_decompress(c) == want
    assert z.zstd_info(c) == {"uncompressed_size": 172, "compressed_size": 126, "dict_id": 0, "has_checksum": True}


@pytest.mark.parametrize("family", ["text", "rdf", "lowent", "rand", "rle"])
def test_families_levels_sizes(z, ref, family):
    from zstdlite_b200 import corpus
    from tests.gpu_util import gpu_decompress_batch
    frames, want = [], []
    for size in (0, 1, 7, 100, 1000, 4096, 65536, 131072, 300000, 1 << 20):
        d = corpus.make(family, size, 11).tobytes()
        for lvl in (1, 2, 3, 5, 9, 19, -3):
            for ck in (False, True):
                frames.append(ref.compress(d, lvl, ck))
                want.append(d)
    res, outs = gpu_decompress_batch(frames, [len(w) for w in want])
    for i, (r, o, w) in enumerate(zip(res, outs, want)):
        assert not z.is_error(r), (i, z.error_name(r))
        assert r == len(w) and o == w, i
    # same frames, host pointers (staging path), arbitrary packing
    res2, outs2 = gpu_decompress_batch(frames[:40], [len(w) for w in want[:40]], device=False)
    assert outs2 == want[:40]


def test_one_shot_api_multiframe_and_skippable(z, ref):
    from zstdlite_b200 import corpus, _lib
    import ctypes as C
    a = corpus.make("text", 50000, 1).tobytes()
    b = corpus.make("rdf", 200000, 2).tobytes()
    skip = (0x184D2A53).to_bytes(4, "little") + (5).to_bytes(4, "little") + b"hello"
    blob = ref.compress(a, 3, True) + skip + ref.compress(b, 1) + ref.compress(b"", 3)
    L = _lib.lib()
    d = z.zstd_dctx()
    dst = C.create_string_buffer(len(a) + len(b))
    r = L.ZSTD_decompressDCtx(d._p, dst, len(a) + len(b), blob, len(blob))
    assert not z.is_error(r), z.error_name(r)
    assert dst.raw[:r] == a + b
    # reference semantics: zstd_decompress() only looks at the first frame (src/raw-file.c:150-189)
    assert z.zstd_decompress(blob) == a
    # too small destination
    r = L.ZSTD_decompressDCtx(d._p, dst, len(a) - 1, blob, len(blob))
    assert z.is_error(r) and z.error_name(r) == "Destination buffer is too small"


def test_checksum_behaviour(z, ref):
    """tests/testthat/test-checksums.R:2-35"""
    from zstdlite_b200 import corpus
    d = corpus.make("text", 100000, 5).tobytes()
    plain, ck = ref.compress(d, 3, False), ref.compress(d, 3, True)
    assert len(ck) == len(plain) + 4
    assert z.zstd_decompress(ck) == d
    bad = bytearray(ck)
    bad[-1] ^= 0x5A
    with pytest.raises(z.ZstdError, match="doesn't match checksum"):
        z.zstd_decompress(bytes(bad))
    assert z.zstd_decompress(bytes(bad), dctx=z.zstd_dctx(validate_checksum=False)) == d
    assert z.zstd_dctx(validate_checksum=False).settings() == {"validate_checksum": 1}     # reference quirk, src/dctx.c:233-239


def test_corrupted_inputs_never_crash(z, ref, restate):
    """every mutated frame must yield an error or output identical to what libzstd produces"""
    from zstdlite_b200 import corpus
    from tests.gpu_util import gpu_decompress_batch
    rng = np.random.default_rng(99)
    frames, caps = [], []
    for fam in ("text", "rdf", "lowent"):
        d = corpus.make(fam, 20000, 3).tobytes()
        c = bytearray(ref.compress(d, 3, True))
        for _ in range(60):
            m = bytearray(c)
            k = int(rng.integers(0, len(m)))
            m[k] ^= 1 << int(rng.integers(0, 8))
            frames.append(bytes(m)); caps.append(len(d))
        for cut in (1, 5, 10, len(c) // 2, len(c) - 1):
            frames.append(bytes(c[:cut])); caps.append(len(d))
    res, outs = gpu_decompress_batch(frames, caps)
    import oracle.ref as R
    for f, cap, r, o in zip(frames, caps, res, outs):
        try:
            want = R.DCtx().decompress(f, cap=cap, all_frames=True)
        except R.RefError:
            want = None
        if want is None:
            assert z.is_error(r), "reference rejects this frame, GPU accepted it"
        else:
            assert not z.is_error(r) and o == want


def test_dictionary_decode(z, ref):
    """config 4 shape: small objects compressed by libzstd with a trained dictionary; raw-content dict too."""
    from tests.gpu_util import gpu_decompress_batch
    rng = np.random.default_rng(4)
    names = [("country_%02d" % i).encode() for i in range(50)]
    samples = []
    for i in range(2000):
        perm = rng.permutation(50)
        samples.append(b"X\n\x00\x00\x00\x03" + b"".join(names[j] + int(rng.integers(0, 1000)).to_bytes(4, "little") for j in perm[: int(rng.integers(10, 50))]))
    d = ref.train_dict(samples[:1000], 5000)
    assert z.zstd_dict_id(d) == ref.lib().ZDICT_getDictID(d, len(d)) != 0
    for dd in (d, b"".join(samples[:20])):          # trained dict, raw-content dict
        frames = [ref.compress(s, 3, False, dict=dd) for s in samples[1000:1400]]
        res, outs = gpu_decompress_batch(frames, [len(s) for s in samples[1000:1400]], dctx=z.zstd_dctx(dict=dd))
        assert outs == samples[1000:1400]
    # wrong / missing dictionary -> error like the reference (zstd.c:41318)
    frames = [ref.compress(samples[0], 3, False, dict=d)]
    res, _ = gpu_decompress_batch(frames, [len(samples[0])])
    assert z.is_error(res[0])


def test_config2_batch_shape(z, ref):
    """configs[1] at reduced count: 512 independent 64 KiB frames, mixed families, level 3."""
    from zstdlite_b200 import corpus
    from tests.gpu_util import gpu_decompress_batch
    data, fams = corpus.mixed_frames(512, 65536, pool=16)
    cache = {}
    frames = []
    for i in range(512):
        key = data[i].tobytes()
        if key not in cache:
            cache[key] = ref.compress(key, 3)
        frames.append(cache[key])
    res, outs = gpu_decompress_batch(frames, [65536] * 512)
    for i in range(512):
        assert res[i] == 65536 and outs[i] == data[i].tobytes(), (i, fams[i])


def test_damaged_frames_without_checksum_decode_like_libzstd(z, ref):
    """Frames WITHOUT a content checksum: a damaged payload that still parses decodes to garbage in libzstd; the CUDA decoder
    must return the same bytes (or an error where libzstd reports one).  The only tolerated difference is the documented
    one: a 4-stream Huffman reader running past the start of its stream is an error here (tools/fuzz_decode.py)."""
    from zstdlite_b200 import corpus
    from tests.gpu_util import gpu_decompress_batch
    rng = np.random.default_rng(5)
    frames, caps = [], []
    for fam, size in (("text", 20000), ("rdf", 30000), ("lowent", 9000)):
        d = corpus.make(fam, size, 5).tobytes()
        c = ref.compress(d, 3, False)
        for _ in range(400):
            m = bytearray(c)
            for _k in range(int(rng.integers(1, 3))):
                m[int(rng.integers(5, len(m)))] ^= 1 << int(rng.integers(0, 8))
            frames.append(bytes(m)); caps.append(len(d))
    res, outs = gpu_decompress_batch(frames, caps)
    same = stricter = 0
    for f, cap, r, o in zip(frames, caps, res, outs):
        try:
            want = ref.DCtx().decompress(f, cap=cap, all_frames=True)
        except ref.RefError:
            want = None
        if want is None:
            assert z.is_error(r), "reference rejects this frame, GPU accepted it"
        elif z.is_error(r):
            stricter += 1
        else:
            assert o == want, "both decoders accept the damaged frame but produce different bytes"
            same += 1
    assert same > 100                      # most single-bit damage lands in the Huffman streams and decodes to garbage
    assert stricter <= len(frames) // 20


def test_large_frames_take_the_block_parallel_path(z, ref):
    """SURVEY.md 8f rank 1: one multi-megabyte frame with cross-block history (config 1's shape).  Frames of >= 1 MiB are
    executed by the block-parallel kernels (parent pointers + pointer jumping); everything must stay byte-exact: levels with
    large windows, checksums, long runs (deep copy chains), dictionaries, unknown content size, mixed batches, errors."""
    import io
    from zstdlite_b200 import corpus
    from tests.gpu_util import gpu_decompress_batch
    big = {f: corpus.make(f, 6 << 20, 31).tobytes() for f in ("text", "rdf", "rle", "lowent", "rand")}
    frames, want = [], []
    for fam, d in big.items():
        for lvl, ck in ((1, False), (3, True), (19, True)):
            if lvl == 19 and fam not in ("text", "rle"):
                continue
            frames.append(ref.compress(d, lvl, ck)); want.append(d)
    # a run of one byte (offset-1 match over megabytes: the deepest possible chain) and a two-byte period
    for d in (bytes(3 << 20), b"ab" * (1 << 20), b"x" + bytes(range(256)) * 5000):
        frames.append(ref.compress(d, 3, True)); want.append(d)
    # small frames in the same batch (warp-per-frame path) keep working next to large ones
    for i in range(40):
        d = corpus.make("text", 50000 + 1000 * i, i).tobytes()
        frames.insert(i * 2 % len(frames), ref.compress(d, 3, i % 2 == 0)); want.insert(i * 2 % len(want), d)
    res, outs = gpu_decompress_batch(frames, [len(w) for w in want])
    for i, (r, o, w) in enumerate(zip(res, outs, want)):
        assert not z.is_error(r), (i, z.error_name(r))
        assert r == len(w) and o == w, i
    # multi-threaded libzstd output (ZSTDMT jobs with overlap) is one ordinary frame
    d = big["text"] + big["rdf"]
    assert z.zstd_decompress(ref.compress(d, 3, True, num_threads=4)) == d
    # dictionary + large frame; raw-content dictionary
    tdict = ref.train_dict([corpus.make("text", 4000, 50 + i).tobytes() for i in range(300)], 30000)
    for dd in (tdict, big["text"][:70000]):
        c = ref.compress(big["text"][:3 << 20], 3, True, dict=dd)
        assert z.zstd_decompress(c, dict=dd) == big["text"][:3 << 20]
    # unknown content size (streamed by libzstd without a pledged size): decoded through the streaming entry point
    L = ref.lib()
    import ctypes as C
    cctx = L.ZSTD_createCCtx()
    src = big["rdf"][:2500000]
    outb = C.create_string_buffer(L.ZSTD_compressBound(len(src)))
    class B(C.Structure):
        _fields_ = [("p", C.c_void_p), ("size", C.c_size_t), ("pos", C.c_size_t)]
    ib = C.create_string_buffer(src, len(src))
    o, i_ = B(C.cast(outb, C.c_void_p), len(outb), 0), B(C.cast(ib, C.c_void_p), len(src), 0)
    L.ZSTD_compressStream2.restype = C.c_size_t
    L.ZSTD_compressStream2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    assert not L.ZSTD_isError(L.ZSTD_compressStream2(cctx, C.byref(o), C.byref(i_), 0)) and i_.pos == len(src)    # ZSTD_e_continue first:
    assert L.ZSTD_compressStream2(cctx, C.byref(o), C.byref(i_), 2) == 0                                          # the size is not in the header
    streamed = outb.raw[:o.pos]
    L.ZSTD_freeCCtx(cctx)
    assert z.zstd_info(streamed)["uncompressed_size"] is None
    assert z.zstd_decompress_stream(io.BytesIO(streamed).read) == src
    # errors: destination too small, damaged payloads (with checksum: every damage is an error, never a crash)
    c = ref.compress(big["text"], 3, True)
    res, _ = gpu_decompress_batch([c], [len(big["text"]) - 1])
    assert z.is_error(res[0])
    rng = np.random.default_rng(8)
    bad = []
    for _ in range(24):
        m = bytearray(c)
        k = int(rng.integers(12, len(m)))
        m[k] ^= 1 << int(rng.integers(0, 8))
        bad.append(bytes(m))
    res, _ = gpu_decompress_batch(bad, [len(big["text"])] * len(bad))
    assert all(z.is_error(r) for r in res)


def test_source_alignment_sweep(z, ref):
    """The entropy kernels fetch their bitstreams as aligned 16-byte chunks (cp.async ring): the same frames at every source
    alignment 0..15, with the last one ending on the last byte of the buffer, must decode to the same bytes."""
    import torch
    from zstdlite_b200 import corpus
    datas = [corpus.make(fam, size, 5).tobytes() for fam in ("text", "lowent", "rdf") for size in (300, 5000, 65536)]
    frames = [ref.compress(d, 3) for d in datas]
    srcs, dsts, sizes, caps, want = [], [], [], [], []
    bufs = []
    for a in range(16):
        for f, d in zip(frames, datas):
            # the frame sits `a` bytes into a 256-byte aligned block whose last byte is the frame's last byte when a == 15
            n = a + len(f)
            buf = torch.zeros((n + 255) // 256 * 256 if a != 15 else n, dtype=torch.uint8, device="cuda")
            buf[a:a + len(f)] = torch.frombuffer(bytearray(f), dtype=torch.uint8).cuda()
            out = torch.zeros(len(d) + 16, dtype=torch.uint8, device="cuda")
            bufs.append((buf, out))
            srcs.append(buf.data_ptr() + a); sizes.append(len(f)); dsts.append(out.data_ptr()); caps.append(len(d)); want.append(d)
    torch.cuda.synchronize()
    res = z.decompress_batch(z.zstd_dctx(), srcs, sizes, dsts, caps, device=True)
    for i, (r, w) in enumerate(zip(res, want)):
        assert not z.is_error(r), (i, z.error_name(r))
        assert r == len(w) and bufs[i][1][:len(w)].cpu().numpy().tobytes() == w, i


def test_pageable_host_buffers_are_staged_by_the_copy_pool(z, ref):
    """ordinary malloc'ed memory of >= 4 MiB (what the reference's C layer hands over: R vectors, src/raw-file.c:166,189) is packed into /
    unpacked from pinned staging by the host copy pool with streaming stores (zl_host.h): every source / destination alignment, frames that
    produce less than their slot, a frame that fails -- bytes identical to libzstd's, nothing written outside a frame's own bytes"""
    from zstdlite_b200 import corpus
    rng = np.random.default_rng(11)
    n, fb = 288, 65536                                          # ~7 MiB compressed, 18 MiB of slots: both directions are staged
    raws = []
    for i in range(n):
        fam = ("text", "rdf", "lowent", "rand")[i % 4]
        size = fb if i % 5 else int(rng.integers(1, fb))            # a fifth of the frames fill only part of their slot
        raws.append(corpus.make(fam, size, 100 + i).tobytes())
    frames = [ref.compress(r, 3, include_checksum=bool(i % 3 == 0)) for i, r in enumerate(raws)]
    bad = 37
    frames[bad] = frames[bad][:-9] + bytes([frames[bad][-9] ^ 0x40]) + frames[bad][-8:]            # damaged: whatever libzstd makes of it
    try:
        want_bad = ref.decompress(frames[bad], cap=fb)
    except ref.RefError:
        want_bad = None
    sizes = [len(f) for f in frames]
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    d = z.zstd_dctx()
    for shift_s, shift_d in ((0, 0), (1, 7), (13, 3)):
        src = np.zeros(int(offs[-1]) + 64, dtype=np.uint8)            # pageable: plain numpy memory
        src[shift_s:shift_s + int(offs[-1])] = np.frombuffer(b"".join(frames), dtype=np.uint8)
        dst = np.full(n * fb + 64, 0xA5, dtype=np.uint8)
        res = z.decompress_batch(d, [src.ctypes.data + shift_s + int(o) for o in offs[:-1]], sizes,
                                 [dst.ctypes.data + shift_d + i * fb for i in range(n)], [fb] * n, device=False)
        for i, r in enumerate(raws):
            got = dst[shift_d + i * fb: shift_d + (i + 1) * fb]
            if i == bad:
                assert z.is_error(res[i]) == (want_bad is None)
                if want_bad is None:
                    assert (got == 0xA5).all()
                    continue
                r = want_bad
            assert res[i] == len(r) and got[:len(r)].tobytes() == r, i
            assert (got[len(r):] == 0xA5).all(), i                   # the rest of the slot is the caller's
        assert (dst[:shift_d] == 0xA5).all() and (dst[shift_d + n * fb:] == 0xA5).all()
    # the one-shot calls on one pageable buffer (ZSTD_compress2 / ZSTD_decompressDCtx: 64 MiB pieces through the same pool)
    big = b"".join(raws)
    c = z.zstd_compress(big, level=3, include_checksum=True)
    assert ref.decompress(c) == big and z.zstd_decompress(c) == big


def test_many_small_frames_descriptors_built_on_the_device(z, ref):
    """>= 4,096 small frames in device memory: the per-frame descriptors come from zl_k_build_descs (the host only copies the caller's four
    arrays).  Same verdict and bytes as libzstd for every frame: dictionary and plain frames, empty frames, a destination that is too small,
    damaged frames, raw (incompressible) frames, checksums"""
    from zstdlite_b200 import corpus
    from tests.gpu_util import gpu_decompress_batch
    rng = np.random.default_rng(23)
    objs = corpus.small_objects(9000)
    d = ref.train_dict(objs[:3000], 4096)
    for use_dict in (True, False):
        items = list(objs)
        items[11] = b""
        items[12] = bytes(rng.integers(0, 256, 900, dtype=np.uint8))           # incompressible: a raw block
        items[13] = b"a" * 1500                                                # a run
        frames = [ref.compress(o, 3, include_checksum=bool(i % 2), dict=d if use_dict else None) for i, o in enumerate(items)]
        caps = [len(o) for o in items]
        caps[20] = max(0, caps[20] - 1)                                        # too small for its frame
        for i in (30, 31, 4000, 8999):                                         # damaged in the middle
            f = bytearray(frames[i]); f[len(f) // 2] ^= 0x10; frames[i] = bytes(f)
        dctx = z.zstd_dctx(dict=d if use_dict else None)
        res, outs = gpu_decompress_batch(frames, caps, dctx=dctx)
        rd = ref.DCtx(dict=d if use_dict else None)
        for i, (f, o, c) in enumerate(zip(frames, items, caps)):
            try:
                want = rd.decompress(f, cap=c)
            except ref.RefError:
                want = None
            if want is None:
                assert z.is_error(res[i]), i
            elif i in (30, 31, 4000, 8999) and z.is_error(res[i]):
                pass                                                           # (damaged 4-stream literals: the documented stricter case, DESIGN.md section 2)
            else:
                assert not z.is_error(res[i]) and outs[i] == want, i
        assert z.is_error(res[20]) and not z.is_error(res[21]) and outs[11] == b""
