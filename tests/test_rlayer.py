"""The reference package's C layer, restated, against the GPU library.

The package's own src/*.c cannot be compiled from this repository (its sources are not part of it), so these tests no longer run
the original C layer.  tests/rlayer_util.py restates its .Call entry points (src/init.c:46-82) with the libzstd / ZDICT calls they
make, over (a) the system's libzstd -- `cpu`, no GPU needed -- and (b) libzstdlite_gpu.so through its ZSTD_* / ZDICT_* exports --
`gpu`.  Comparison with the original rests on what it produced and is stored under tests/golden/: its known-answer frame
(man/figures/data.json.zst and the bytes README.md:199-205 prints), its dictionary (inst/sample_dict.raw, dictID 1895278874) and
the frame header README.md:102-105 prints; each is read back through both libraries.  The tests replay the package's testthat files:
  tests/testthat/test-compress-raw.R:1-33, 34-100   round trips, num_threads = 2, separate contexts, file / streaming interop
  tests/testthat/test-cctx.R:22-37                  determinism with and without a context, context re-use
  tests/testthat/test-checksums.R:1-35              + 4 bytes, "doesn't match checksum", validate_checksum = FALSE
  tests/testthat/test-train-dict.R:1-28             real dictionaries, identical when trained identically
R's serialize() is not available: the payloads are the byte strings it would hand over (corpus.r_data_frame restates its layout)."""
import os

import numpy as np
import pytest

from tests.rlayer_util import RError, RLayer

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _gold(name):
    with open(os.path.join(GOLD, name), "rb") as fh:
        return fh.read()


def _flavours():
    return [pytest.param("cpu", id="reference-libzstd"), pytest.param("gpu", id="gpu-library", marks=pytest.mark.gpu)]


@pytest.fixture(scope="module", params=_flavours())
def R(request):
    if request.param == "gpu":
        import torch
        assert torch.cuda.is_available()
    return RLayer(request.param)


def _payloads():
    from zstdlite_b200 import corpus
    rng = np.random.default_rng(11)
    return {"mtcars": corpus.r_data_frame(32)[:7000], "iris": corpus.r_data_frame(150), "sample(1e6)": rng.permutation(1_000_000).astype("<i4").tobytes(),
            "function": b"X\n\x00\x00\x00\x03\x00\x04\x04\x01\x00\x03\x05\x00" + b"function(x) {3 + 7 + x}" * 3}


def test_raw_compress_roundtrip(R):
    """test-compress-raw.R:1-33"""
    p = _payloads()
    for name, dat in p.items():
        assert R.zstd_decompress(R.zstd_compress(dat)) == dat, name
    dat = p["sample(1e6)"]
    assert R.zstd_decompress(R.zstd_compress(dat, num_threads=2)) == dat              # "Multithreading"
    cctx, dctx = R.zstd_cctx(), R.zstd_dctx()                                          # "separate context"
    assert cctx.klass == "ZSTD_CCtx" and dctx.klass == "ZSTD_DCtx"
    assert R.zstd_decompress(R.zstd_compress(p["mtcars"], cctx=cctx), dctx=dctx) == p["mtcars"]
    assert R.zstd_decompress(R.zstd_compress("a string, a string, a string"), type="string") == "a string, a string, a string"
    R.finalize(cctx); R.finalize(dctx)                                                 # finalizers run in any order, any time (src/cctx.c:191-207)
    assert R.zstd_decompress(_gold("data.json.zst"), type="string") == _gold("data.json").decode()   # the original's own frame (README.md:199-205)


def test_raw_compress_roundtrip_to_file(R, tmp_path):
    """test-compress-raw.R:34-100: one-shot and streaming writers against one-shot and streaming readers"""
    p = _payloads()
    f = str(tmp_path / "x.zst")
    with open(f, "wb") as fh:
        fh.write(_gold("data.json.zst"))                                               # the original's own file, both readers
    for rstream in (False, True):
        assert R.zstd_decompress(f, use_file_streaming=rstream) == _gold("data.json"), rstream
    for name in ("mtcars", "iris", "function"):
        assert R.zstd_compress(p[name], file=f) is None
        assert R.zstd_decompress(f) == p[name], name
    dat = p["sample(1e6)"]
    for wstream in (False, True):
        for rstream in (False, True):
            R.zstd_compress(dat, file=f, use_file_streaming=wstream, num_threads=2)
            assert R.zstd_decompress(f, use_file_streaming=rstream) == dat, (wstream, rstream)


def test_cctx_determinism(R):
    """test-cctx.R:22-37"""
    dat = _payloads()["mtcars"]
    cctx = R.zstd_cctx()
    assert R.zstd_compress(dat) == R.zstd_compress(dat, cctx=cctx)
    assert R.zstd_compress(dat) == R.zstd_compress(dat, cctx=cctx)                     # re-using a cctx
    assert R.call("get_cctx_settings_", R.zstd_cctx(level=2, num_threads=3, include_checksum=True)) == {"level": 2, "num_threads": 3, "include_checksum": True}


def test_checksums(R):
    """test-checksums.R:1-35"""
    dat = np.arange(1, 11, dtype="<i4").tobytes() * 20
    v1 = R.zstd_compress(dat)
    v2 = R.zstd_compress(dat, cctx=R.zstd_cctx(include_checksum=True))
    assert len(v1) + 4 == len(v2)
    assert R.zstd_decompress(v2) == dat
    bad = bytearray(v2); bad[-1] ^= 0xFF                                               # "manually hack the checksum"
    with pytest.raises(RError, match="doesn't match checksum"):
        R.zstd_decompress(bytes(bad))
    assert R.zstd_decompress(bytes(bad), dctx=R.zstd_dctx(validate_checksum=False)) == dat
    assert R.call("get_dctx_settings_", R.zstd_dctx(validate_checksum=False)) == {"validate_checksum": True}    # the reference's quirk (src/dctx.c:233-239)
    hdr = bytes([0x28, 0xB5, 0x2F, 0xFD, 0x60, 0xE8, 0x02, 0xC5, 0x0E, 0x00])           # the original's zstd_serialize(head(mtcars)), README.md:102-105
    assert R.zstd_info(hdr)["uncompressed_size"] == 1000 and R.zstd_info(hdr)["has_checksum"] is False
    info = R.zstd_info(v2)
    assert info["has_checksum"] is True and info["uncompressed_size"] == len(dat) and info["compressed_size"] == len(v2) and info["dict_id"] == 0


def test_train_dict(R):
    """test-train-dict.R:1-28, then the dictionary in both contexts (vignettes/dictionaries.Rmd)"""
    rng = np.random.default_rng(3)
    cars = ["Mazda RX4", "Mazda RX4 Wag", "Datsun 710", "Hornet 4 Drive", "Hornet Sportabout", "Valiant", "Duster 360", "Merc 240D", "Merc 230", "Merc 280",
            "Merc 280C", "Merc 450SE", "Merc 450SL", "Merc 450SLC", "Cadillac Fleetwood", "Lincoln Continental", "Chrysler Imperial", "Fiat 128", "Honda Civic",
            "Toyota Corolla", "Toyota Corona", "Dodge Challenger", "AMC Javelin", "Camaro Z28", "Pontiac Firebird", "Fiat X1-9", "Porsche 914-2", "Lotus Europa",
            "Ford Pantera L", "Ferrari Dino", "Maserati Bora", "Volvo 142E"]
    samples = [",".join(rng.permutation(cars)) for _ in range(1000)]
    raws = [s.encode() for s in samples]
    d1 = R.zstd_train_dict_compress(raws, size=2000)
    assert R.zstd_dict_id(d1) != 0                                                     # "is a real dictionary!"
    d2 = R.zstd_train_dict_compress(samples, size=2000)
    assert d1 == d2 and R.zstd_dict_id(d1) == R.zstd_dict_id(d2)                       # "trained identically should be identical"
    R.zstd_train_dict_compress(raws[:300], size=2000)
    assert R.warnings[0] >= 1 and "100x" in R.warnings[1]                              # src/dictionaries.c:104: less than 100x the dictionary size
    c = R.zstd_compress(raws[7], cctx=R.zstd_cctx(dict=d1))
    assert len(c) < len(R.zstd_compress(raws[7]))
    assert R.zstd_info(c)["dict_id"] == R.zstd_dict_id(d1)
    assert R.zstd_decompress(c, dctx=R.zstd_dctx(dict=d1)) == raws[7]
    sd = _gold("sample_dict.raw")                                                      # the original's inst/sample_dict.raw
    assert R.zstd_dict_id(sd) == 1895278874
    gold = np.load(os.path.join(GOLD, "frames.npz"))
    for fam in ("text", "rdf"):                                                        # frames the reference's libzstd made with it
        assert R.zstd_decompress(gold[f"{fam}_dict"].tobytes(), dctx=R.zstd_dctx(dict=sd)) == gold[f"{fam}_dict.raw"].tobytes(), fam
    with pytest.raises(RError, match="No samples"):
        R.zstd_train_dict_compress([], size=2000)


@pytest.mark.gpu
def test_gpu_and_reference_layers_interoperate():
    """the same C layer over the two libraries: every frame of one decodes with the other (both directions, with a dictionary too)"""
    import torch
    assert torch.cuda.is_available()
    G, Cc = RLayer("gpu"), RLayer("cpu")
    p = _payloads()
    for name, dat in p.items():
        for lvl in (1, 3):
            g = G.zstd_compress(dat, level=lvl, include_checksum=True)
            assert Cc.zstd_decompress(g) == dat, name
            assert G.zstd_decompress(Cc.zstd_compress(dat, level=lvl, include_checksum=True)) == dat, name
    with pytest.raises(RError, match="Bad compression level"):                         # src/cctx.c:265 <- parameter_unsupported (levels >= 4)
        G.zstd_cctx(level=9)
