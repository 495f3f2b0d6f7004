"""ctypes binding of the system's libzstd (libzstd.so.1).  TEST INFRA ONLY.

Mirrors the call sequences of the reference's C layer:
  compress    src/raw-file.c:52-83   (ZSTD_compressBound, ZSTD_compress2)
  decompress  src/raw-file.c:150-192 (findFrameCompressedSize, getFrameContentSize, decompressDCtx)
  contexts    src/cctx.c:213-315, src/dctx.c:110-197
  dictionary  src/dictionaries.c:120-208
"""
import ctypes as C
import os

# the soname of libzstd 1.x: part of every Debian / Ubuntu base system (package libzstd1), so no build step is needed
_PATH = "libzstd.so.1"
# releases the tests and the CPU baseline were checked against: the reference vendors 1.5.6; 1.5.5 differs from it in one
# decoder corner that tests/test_oracle.py pins with stored answers.  Any other release is refused rather than trusted.
ACCEPTED_VERSIONS = ("1.5.5", "1.5.6")

ZSTD_c_compressionLevel = 100
ZSTD_c_checksumFlag = 201
ZSTD_c_nbWorkers = 400
ZSTD_d_forceIgnoreChecksum = 1002
CONTENTSIZE_UNKNOWN = 2**64 - 1
CONTENTSIZE_ERROR = 2**64 - 2


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(_PATH, mode=os.RTLD_LOCAL)
        vp, sz = C.c_void_p, C.c_size_t
        L.ZSTD_createCCtx.restype = vp
        L.ZSTD_freeCCtx.argtypes = [vp]
        L.ZSTD_createDCtx.restype = vp
        L.ZSTD_freeDCtx.argtypes = [vp]
        L.ZSTD_CCtx_setParameter.argtypes = [vp, C.c_int, C.c_int]
        L.ZSTD_CCtx_setParameter.restype = sz
        L.ZSTD_DCtx_setParameter.argtypes = [vp, C.c_int, C.c_int]
        L.ZSTD_DCtx_setParameter.restype = sz
        L.ZSTD_CCtx_loadDictionary.argtypes = [vp, vp, sz]
        L.ZSTD_CCtx_loadDictionary.restype = sz
        L.ZSTD_DCtx_loadDictionary.argtypes = [vp, vp, sz]
        L.ZSTD_DCtx_loadDictionary.restype = sz
        L.ZSTD_compressBound.argtypes = [sz]
        L.ZSTD_compressBound.restype = sz
        L.ZSTD_compress2.argtypes = [vp, vp, sz, vp, sz]
        L.ZSTD_compress2.restype = sz
        L.ZSTD_decompressDCtx.argtypes = [vp, vp, sz, vp, sz]
        L.ZSTD_decompressDCtx.restype = sz
        L.ZSTD_findFrameCompressedSize.argtypes = [vp, sz]
        L.ZSTD_findDecompressedSize.argtypes = [vp, sz]
        L.ZSTD_findDecompressedSize.restype = C.c_ulonglong
        L.ZSTD_findFrameCompressedSize.restype = sz
        L.ZSTD_getFrameContentSize.argtypes = [vp, sz]
        L.ZSTD_getFrameContentSize.restype = C.c_ulonglong
        L.ZSTD_isError.argtypes = [sz]
        L.ZSTD_isError.restype = C.c_uint
        L.ZSTD_getErrorName.argtypes = [sz]
        L.ZSTD_getErrorName.restype = C.c_char_p
        L.ZSTD_versionString.restype = C.c_char_p
        L.ZSTD_getDictID_fromFrame.argtypes = [vp, sz]
        L.ZSTD_getDictID_fromFrame.restype = C.c_uint
        L.ZDICT_trainFromBuffer.argtypes = [vp, sz, vp, vp, C.c_uint]
        L.ZDICT_trainFromBuffer.restype = sz
        L.ZDICT_getDictID.argtypes = [vp, sz]
        L.ZDICT_getDictID.restype = C.c_uint
        L.ZDICT_isError.argtypes = [sz]
        L.ZDICT_isError.restype = C.c_uint
        v = L.ZSTD_versionString().decode()
        if v not in ACCEPTED_VERSIONS:
            raise RuntimeError(f"{_PATH} is libzstd {v}; the oracle accepts {', '.join(ACCEPTED_VERSIONS)}")
        _lib = L
    return _lib


class RefError(RuntimeError):
    pass


def _chk(r):
    L = lib()
    if L.ZSTD_isError(r):
        raise RefError(L.ZSTD_getErrorName(r).decode())
    return r


def _buf(b):
    return (C.c_char * max(1, len(b))).from_buffer_copy(bytes(b) if len(b) else b"\0")


class CCtx:
    """src/cctx.c:213-315 init_cctx_with_opts"""

    def __init__(self, level=3, num_threads=1, include_checksum=False, dict=None):
        L = lib()
        self.p = L.ZSTD_createCCtx()
        level = max(-5, min(22, int(level)))
        _chk(L.ZSTD_CCtx_setParameter(self.p, ZSTD_c_compressionLevel, level))
        if num_threads > 1:
            _chk(L.ZSTD_CCtx_setParameter(self.p, ZSTD_c_nbWorkers, int(num_threads)))
        _chk(L.ZSTD_CCtx_setParameter(self.p, ZSTD_c_checksumFlag, 1 if include_checksum else 0))
        if dict is not None:
            d = _buf(dict)
            _chk(L.ZSTD_CCtx_loadDictionary(self.p, d, len(dict)))

    def compress(self, data):
        L = lib()
        n = len(data)
        cap = L.ZSTD_compressBound(n)
        dst = C.create_string_buffer(cap)
        src = _buf(data)
        r = _chk(L.ZSTD_compress2(self.p, dst, cap, src, n))
        return dst.raw[:r]

    def __del__(self):
        if getattr(self, "p", None):
            lib().ZSTD_freeCCtx(self.p)
            self.p = None


class DCtx:
    """src/dctx.c:110-197 init_dctx_with_opts"""

    def __init__(self, validate_checksum=True, dict=None):
        L = lib()
        self.p = L.ZSTD_createDCtx()
        _chk(L.ZSTD_DCtx_setParameter(self.p, ZSTD_d_forceIgnoreChecksum, 0 if validate_checksum else 1))
        if dict is not None:
            d = _buf(dict)
            _chk(L.ZSTD_DCtx_loadDictionary(self.p, d, len(dict)))

    def decompress(self, data, cap=None, all_frames=False):
        """src/raw-file.c:150-192: first frame only unless all_frames."""
        L = lib()
        src = _buf(data)
        n = len(data)
        if not all_frames:
            n = _chk(L.ZSTD_findFrameCompressedSize(src, n))
        if cap is None:
            cap = L.ZSTD_getFrameContentSize(src, n)
            if cap >= CONTENTSIZE_ERROR:
                raise RefError("content size unknown")
        dst = C.create_string_buffer(max(1, cap))
        r = _chk(L.ZSTD_decompressDCtx(self.p, dst, cap, src, n))
        return dst.raw[:r]

    def __del__(self):
        if getattr(self, "p", None):
            lib().ZSTD_freeDCtx(self.p)
            self.p = None


def compress(data, level=3, include_checksum=False, dict=None, num_threads=1):
    return CCtx(level, num_threads, include_checksum, dict).compress(data)


def decompress(data, validate_checksum=True, dict=None, cap=None, all_frames=False):
    return DCtx(validate_checksum, dict).decompress(data, cap, all_frames)


def train_dict(samples, dict_size):
    """src/dictionaries.c:120-208 (ZDICT_trainFromBuffer branch)."""
    L = lib()
    blob = b"".join(samples)
    sizes = (C.c_size_t * len(samples))(*[len(s) for s in samples])
    out = C.create_string_buffer(dict_size)
    r = L.ZDICT_trainFromBuffer(out, dict_size, _buf(blob), sizes, len(samples))
    if L.ZDICT_isError(r):
        raise RefError("dict training failed")
    return out.raw[:r]


def version():
    return lib().ZSTD_versionString().decode()
