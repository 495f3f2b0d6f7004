"""-m gpu tests of dictionary training on the GPU (SURVEY.md 8f rank 4; csrc/zl_dict_train.cuh), through the C ABI
(ZDICT_trainFromBuffer / ZDICT_optimizeTrainFromBuffer_cover) and the host mirrors zstd_train_dict_compress / _serialize.

Oracle: libzstd's own ZDICT (oracle/ref.py).  Bars: (1) the dictionary is a standard Zstandard dictionary that the
reference's libzstd loads, compresses with and decodes with; (2) at the k the reference's fastCOVER search picks, the selected
CONTENT is identical to the reference's (same dictionary ID = same XXH64 of the content, same trailing bytes); (3) held-out
objects compress within 5% of the reference pipeline (ZDICT dictionary + libzstd) when the GPU dictionary is used by the GPU
compressor (measured -2.9% .. +3.0%), and within 6% when it is used by libzstd (measured +1.0% .. +3.9%; the entropy tables are
fitted to the parser that made the statistics)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def z():
    import torch
    assert torch.cuda.is_available()
    import zstdlite_b200 as zz
    return zz


class _FastCoverParams(C.Structure):                    # ZDICT_fastCover_params_t (src/zstd/zstd.h, zdict section)
    _fields_ = [("k", C.c_uint), ("d", C.c_uint), ("f", C.c_uint), ("steps", C.c_uint), ("nbThreads", C.c_uint), ("splitPoint", C.c_double),
                ("accel", C.c_uint), ("shrinkDict", C.c_uint), ("shrinkDictMaxRegression", C.c_uint),
                ("compressionLevel", C.c_int), ("notificationLevel", C.c_uint), ("dictID", C.c_uint)]


def _reference_search(ref, train, size):
    """the search ZDICT_trainFromBuffer runs (zstd.c:50979), with the chosen parameters returned"""
    par = _FastCoverParams(); par.d = 8; par.steps = 4; par.compressionLevel = 3
    blob = b"".join(train); sizes = (C.c_size_t * len(train))(*[len(s) for s in train]); out = C.create_string_buffer(size)
    L = ref.lib()
    L.ZDICT_optimizeTrainFromBuffer_fastCover.restype = C.c_size_t
    L.ZDICT_optimizeTrainFromBuffer_fastCover.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint, C.c_void_p]
    r = L.ZDICT_optimizeTrainFromBuffer_fastCover(out, size, blob, sizes, len(train), C.byref(par))
    assert not L.ZDICT_isError(r)
    return out.raw[:r], par.k


def _quiet(fn, *a, **k):
    """the R layer warns when the samples are less than 100x the dictionary size (src/dictionaries.c:104); checked separately"""
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return fn(*a, **k)


def _gpu_total(z, objs, d):
    import torch
    cc = z.zstd_cctx(level=3, dict=d)
    src = torch.from_numpy(np.frombuffer(b"".join(objs), dtype=np.uint8).copy()).cuda()
    offs = np.concatenate([[0], np.cumsum([len(o) for o in objs])]).astype(np.int64)
    caps = [len(o) + 64 for o in objs]; coffs = np.concatenate([[0], np.cumsum(caps)]).astype(np.int64)
    dst = torch.zeros(int(coffs[-1]) + 64, dtype=torch.uint8, device="cuda")
    res = z.compress_batch(cc, [src.data_ptr() + int(o) for o in offs[:-1]], [len(o) for o in objs], [dst.data_ptr() + int(o) for o in coffs[:-1]], caps)
    assert not any(z.is_error(int(r)) for r in res)
    return sum(int(r) for r in res)


@pytest.mark.parametrize("n,size", [(4000, 5000), (12000, 20000)])
def test_trained_dictionary_is_standard_and_as_good_as_the_reference(z, ref, n, size):
    from zstdlite_b200 import corpus
    objs = corpus.small_objects(n + 1500)
    train, test = objs[:n], objs[n:]
    d = _quiet(z.zstd_train_dict_compress, train, size)
    assert 256 <= len(d) <= size and d[:4] == (0xEC30A437).to_bytes(4, "little")
    did = z.zstd_dict_id(d)
    assert 32768 <= did < 2**31 and did == ref.lib().ZDICT_getDictID(d, len(d))
    # the reference's libzstd uses it: frames carry its ID and decode only with it; our codec agrees in both directions
    rc, rd = ref.CCtx(level=3, dict=d), ref.DCtx(dict=d)
    gd = z.zstd_dctx(dict=d)
    total_ref_with_ours = 0
    for o in test[:300]:
        c = rc.compress(o)
        assert z.zstd_dict_id(c) == did and rd.decompress(c, cap=len(o)) == o and z.zstd_decompress(c, dctx=gd) == o
        g = z.zstd_compress(o, level=3, dict=d)
        assert rd.decompress(g, cap=len(o)) == o
    for o in test:
        total_ref_with_ours += len(rc.compress(o))
    # quality against the reference's trainer on the same samples
    d_ref = ref.train_dict(train, size)
    rc2 = ref.CCtx(level=3, dict=d_ref)
    total_ref = sum(len(rc2.compress(o)) for o in test)
    total_none = sum(len(ref.compress(o, 3)) for o in test)
    total_gpu = _gpu_total(z, test, d)
    assert total_ref_with_ours < 0.8 * total_none
    assert total_ref_with_ours <= 1.06 * total_ref, (total_ref_with_ours, total_ref)
    assert total_gpu <= 1.05 * total_ref, (total_gpu, total_ref)


def test_selected_content_equals_fastcover_at_the_same_k(z, ref):
    from zstdlite_b200 import corpus, _lib
    train = corpus.small_objects(6000)
    size = 8000
    d_ref, k = _reference_search(ref, train, size)
    par = _lib.CoverParams(); par.k = k; par.d = 8; par.splitPoint = 0.75
    blob = b"".join(train); sizes = (C.c_size_t * len(train))(*[len(s) for s in train]); out = C.create_string_buffer(size)
    r = _lib.lib().ZDICT_optimizeTrainFromBuffer_cover(out, size, blob, sizes, len(train), C.byref(par))
    assert not _lib.lib().ZDICT_isError(r), _lib.lib().ZDICT_getErrorName(r)
    d = out.raw[:r]
    assert (par.k, par.d) == (k, 8)
    assert z.zstd_dict_id(d) == z.zstd_dict_id(d_ref)                     # ID = XXH64 of the content (zstd.c:50752)
    # the content follows the entropy tables (a few bytes longer or shorter than the reference's): same bytes, shifted
    probe = d_ref[1000:7000]
    at = d.find(probe)
    assert at >= 0 and abs(at - 1000) < 64


def test_optimize_cover_and_serialize_mirrors(z, ref):
    from zstdlite_b200 import corpus
    train = corpus.small_objects(3000)
    d = _quiet(z.zstd_train_dict_compress, train, 4096, optim=True, optim_shrink_allow=3)
    assert ref.DCtx(dict=d).decompress(ref.CCtx(level=3, dict=d).compress(train[7]), cap=len(train[7])) == train[7]
    rng = np.random.default_rng(5)
    names = ["country_%02d" % i for i in range(50)]
    samples = [{names[j]: int(rng.integers(0, 1000)) for j in rng.permutation(50)[:int(rng.integers(10, 50))]} for _ in range(2500)]
    ds = _quiet(z.zstd_train_dict_serialize, samples, size=6000)
    with_dict = z.zstd_serialize(samples[3], level=3, dict=ds)
    assert len(with_dict) < len(z.zstd_serialize(samples[3], level=3))
    assert z.zstd_unserialize(with_dict, dict=ds) == samples[3]


def test_training_errors(z):
    from zstdlite_b200 import corpus
    objs = corpus.small_objects(50)
    with pytest.raises(z.ZstdError, match="No samples"):
        z.zstd_train_dict_compress([], 5000)
    with pytest.raises(z.ZstdError, match=">= 8 bytes"):
        z.zstd_train_dict_compress([b"short"] * 20, 5000)
    with pytest.raises(z.ZstdError, match="Training error"), pytest.warns(UserWarning, match="100x"):
        z.zstd_train_dict_compress(objs[:4], 5000)                        # fewer than 5 training samples (zstd.c:49461); src/dictionaries.c:104
    with pytest.raises(z.ZstdError, match="Training error"):
        z.zstd_train_dict_compress(objs, 100)                             # below ZDICT_DICTSIZE_MIN


def test_large_samples_are_accepted(z, ref):
    """ZDICT takes samples of any size (the d-mer selection sees every byte, only the entropy statistics clip a sample to one block,
    zstd.c:50440-50460): serialized data.frame-like objects of several hundred KiB must train, and the dictionary must be standard."""
    from zstdlite_b200 import corpus
    rng = np.random.default_rng(5)
    base = corpus.make("text", 300000, 3).tobytes()
    samples = [base[int(o):int(o) + int(n)] for o, n in zip(rng.integers(0, 100000, 24), rng.integers(140000, 200000, 24))]
    d = _quiet(z.zstd_train_dict_compress, samples, 16384)
    assert z.zstd_dict_id(d) != 0 and len(d) <= 16384
    held = base[50000:50000 + 150000]
    c = z.zstd_compress(held, level=3, dict=d)
    assert ref.DCtx(dict=d).decompress(c, cap=len(held)) == held
    assert len(ref.CCtx(level=3, dict=d).compress(held[:4000])) < len(ref.CCtx(level=3).compress(held[:4000]))
