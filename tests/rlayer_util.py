"""The reference package's C layer restated over a libzstd-compatible C library (TEST INFRASTRUCTURE ONLY).

The package's src/{cctx,dctx,raw-file,raw-file-in,raw-file-out,dictionaries,zstd-info}.c are not part of this repository, so their
.Call entry points (src/init.c:46-82) are restated here with the libzstd / ZDICT calls they make (the call sites zstdlite_b200/api.py
cites) and the error and warning texts the replayed testthat files match.  One restatement runs over two libraries that export the
same symbols:
  cpu   the system's libzstd (libzstd.so.1), which pins the restatement and the replayed expectations without a GPU
  gpu   libzstdlite_gpu.so, every libzstd / ZDICT call answered by the GPU library (its canonical ZSTD_* / ZDICT_* exports)
Each flavour loads its own ctypes handle, so the signatures set here do not touch oracle.ref or zstdlite_b200._lib."""
import ctypes as C
import os

ZSTD_c_compressionLevel, ZSTD_c_checksumFlag, ZSTD_c_nbWorkers = 100, 201, 400
ZSTD_d_forceIgnoreChecksum = 1002
ZSTD_e_continue, ZSTD_e_end = 0, 2
CONTENTSIZE_UNKNOWN, CONTENTSIZE_ERROR = 2**64 - 1, 2**64 - 2
FILE_CHUNK = 1 << 17                                       # bytes handed to one streaming call (ZSTD_CStreamInSize() of 1.5.x)


class RError(RuntimeError):
    """error() raised inside the C layer"""


class _InBuffer(C.Structure):
    _fields_ = [("src", C.c_void_p), ("size", C.c_size_t), ("pos", C.c_size_t)]


class _OutBuffer(C.Structure):
    _fields_ = [("dst", C.c_void_p), ("size", C.c_size_t), ("pos", C.c_size_t)]


class _FrameHeader(C.Structure):                            # ZSTD_frameHeader, zstd.h
    _fields_ = [("frameContentSize", C.c_ulonglong), ("windowSize", C.c_ulonglong), ("blockSizeMax", C.c_uint),
                ("frameType", C.c_int), ("headerSize", C.c_uint), ("dictID", C.c_uint), ("checksumFlag", C.c_uint),
                ("_reserved1", C.c_uint), ("_reserved2", C.c_uint)]


def _library(flavour):
    if flavour == "cpu":
        return C.CDLL("libzstd.so.1", mode=os.RTLD_LOCAL)
    from zstdlite_b200 import _lib
    return C.CDLL(_lib.LIB_PATH, mode=os.RTLD_LOCAL)


class _Ptr:
    """an external pointer with its R class attribute (src/cctx.c:191-207, src/dctx.c:40-56)"""

    def __init__(self, p, klass, free):
        self.p, self.klass, self._free = p, klass, free

    def finalize(self):
        if self.p:
            self._free(self.p)
            self.p = None

    __del__ = finalize                                      # R's collector frees an unreachable context the same way


class RLayer:
    def __init__(self, flavour):
        L = _library(flavour)
        vp, sz, pint = C.c_void_p, C.c_size_t, C.POINTER(C.c_int)
        for name, res, args in (
                ("ZSTD_isError", C.c_uint, [sz]), ("ZSTD_getErrorName", C.c_char_p, [sz]),
                ("ZSTD_createCCtx", vp, []), ("ZSTD_freeCCtx", sz, [vp]), ("ZSTD_createDCtx", vp, []), ("ZSTD_freeDCtx", sz, [vp]),
                ("ZSTD_CCtx_setParameter", sz, [vp, C.c_int, C.c_int]), ("ZSTD_CCtx_getParameter", sz, [vp, C.c_int, pint]),
                ("ZSTD_DCtx_setParameter", sz, [vp, C.c_int, C.c_int]), ("ZSTD_DCtx_getParameter", sz, [vp, C.c_int, pint]),
                ("ZSTD_CCtx_loadDictionary", sz, [vp, vp, sz]), ("ZSTD_DCtx_loadDictionary", sz, [vp, vp, sz]),
                ("ZSTD_CCtx_setPledgedSrcSize", sz, [vp, C.c_ulonglong]), ("ZSTD_compressBound", sz, [sz]), ("ZSTD_compress2", sz, [vp, vp, sz, vp, sz]),
                ("ZSTD_decompressDCtx", sz, [vp, vp, sz, vp, sz]), ("ZSTD_findFrameCompressedSize", sz, [vp, sz]),
                ("ZSTD_getFrameContentSize", C.c_ulonglong, [vp, sz]), ("ZSTD_getFrameHeader", sz, [C.POINTER(_FrameHeader), vp, sz]),
                ("ZSTD_compressStream2", sz, [vp, C.POINTER(_OutBuffer), C.POINTER(_InBuffer), C.c_int]),
                ("ZSTD_decompressStream", sz, [vp, C.POINTER(_OutBuffer), C.POINTER(_InBuffer)]),
                ("ZSTD_getDictID_fromFrame", C.c_uint, [vp, sz]), ("ZDICT_getDictID", C.c_uint, [vp, sz]),
                ("ZDICT_trainFromBuffer", sz, [vp, sz, vp, C.POINTER(C.c_size_t), C.c_uint]),
                ("ZDICT_isError", C.c_uint, [sz]), ("ZDICT_getErrorName", C.c_char_p, [sz])):
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        self.L = L
        self._warnings = []

    def _err(self, where, r):
        raise RError(f"{where}: {self.L.ZSTD_getErrorName(r).decode()}")

    @property
    def warnings(self):
        """(warnings raised by the last call, the last one's text), as R would report them"""
        return len(self._warnings), self._warnings[-1] if self._warnings else ""

    def finalize(self, ptr):
        """run the external pointer's finalizer, as R's collector would"""
        ptr.finalize()

    def call(self, name, *args):
        """the settings entry points (src/cctx.c:343-369, src/dctx.c:228-245), by their .Call names"""
        self._warnings = []
        ctx = args[0]
        if name == "get_cctx_settings_":
            out = {}
            for key, par in (("level", ZSTD_c_compressionLevel), ("num_threads", ZSTD_c_nbWorkers), ("include_checksum", ZSTD_c_checksumFlag)):
                v = C.c_int(0)
                self.L.ZSTD_CCtx_getParameter(ctx.p, par, C.byref(v))
                out[key] = bool(v.value) if key == "include_checksum" else v.value
            return out
        if name == "get_dctx_settings_":
            v = C.c_int(0)
            self.L.ZSTD_DCtx_getParameter(ctx.p, ZSTD_d_forceIgnoreChecksum, C.byref(v))
            return {"validate_checksum": bool(v.value)}          # the reference's quirk: it reports forceIgnoreChecksum
        raise KeyError(name)

    # ---- init_cctx_ / init_dctx_ (src/cctx.c:213-315, src/dctx.c:110-197)
    def zstd_cctx(self, level=3, num_threads=1, include_checksum=False, dict=None):
        L = self.L
        p = L.ZSTD_createCCtx()
        if not p:
            raise RError("init_cctx(): Couldn't initialse memory for 'cctx'")
        cctx = _Ptr(p, "ZSTD_CCtx", L.ZSTD_freeCCtx)
        if L.ZSTD_isError(L.ZSTD_CCtx_setParameter(p, ZSTD_c_compressionLevel, max(-5, min(22, int(level))))):
            raise RError("init_cctx(): Bad compression level")
        if int(num_threads) > 1:
            r = L.ZSTD_CCtx_setParameter(p, ZSTD_c_nbWorkers, int(num_threads))
            if L.ZSTD_isError(r):
                self._err("init_cctx(): Bad num_threads", r)
        L.ZSTD_CCtx_setParameter(p, ZSTD_c_checksumFlag, 1 if include_checksum else 0)
        if dict is not None:
            r = L.ZSTD_CCtx_loadDictionary(p, bytes(dict), len(dict))
            if L.ZSTD_isError(r):
                self._err("init_cctx(): Error initialising dict", r)
        return cctx

    def zstd_dctx(self, validate_checksum=True, dict=None):
        L = self.L
        p = L.ZSTD_createDCtx()
        if not p:
            raise RError("init_dctx(): Couldn't initialse memory for 'dctx'")
        dctx = _Ptr(p, "ZSTD_DCtx", L.ZSTD_freeDCtx)
        L.ZSTD_DCtx_setParameter(p, ZSTD_d_forceIgnoreChecksum, 0 if validate_checksum else 1)
        if dict is not None:
            r = L.ZSTD_DCtx_loadDictionary(p, bytes(dict), len(dict))
            if L.ZSTD_isError(r):
                self._err("init_dctx(): Error initialising dict", r)
        return dctx

    # ---- zstd_compress_ (src/raw-file.c:52-83, src/raw-file-out.c)
    def zstd_compress(self, src, file=None, cctx=None, use_file_streaming=False, **opts):
        self._warnings = []
        L = self.L
        if cctx is None:
            cctx = self.zstd_cctx(**opts)
        data = src.encode() if isinstance(src, str) else bytes(src)
        if file is not None and use_file_streaming:
            r = L.ZSTD_CCtx_setPledgedSrcSize(cctx.p, len(data))       # the whole input is known: its size goes in the frame header
            if L.ZSTD_isError(r):
                self._err("zstd_compress_stream_file_()", r)
            with open(file, "wb") as fh:
                out = C.create_string_buffer(FILE_CHUNK + 1024)
                for pos in range(0, len(data) + 1, FILE_CHUNK):
                    chunk = data[pos:pos + FILE_CHUNK]
                    last = pos + FILE_CHUNK >= len(data)
                    ib = _InBuffer(C.cast(C.c_char_p(chunk), C.c_void_p), len(chunk), 0)
                    while True:
                        ob = _OutBuffer(C.cast(out, C.c_void_p), len(out), 0)
                        r = L.ZSTD_compressStream2(cctx.p, C.byref(ob), C.byref(ib), ZSTD_e_end if last else ZSTD_e_continue)
                        if L.ZSTD_isError(r):
                            self._err("zstd_compress_stream_file_()", r)
                        fh.write(out.raw[:ob.pos])
                        if (r == 0) if last else (ib.pos == ib.size):
                            break
                    if last:
                        break
            return None
        cap = L.ZSTD_compressBound(len(data))
        dst = C.create_string_buffer(max(1, cap))
        r = L.ZSTD_compress2(cctx.p, dst, cap, data, len(data))
        if L.ZSTD_isError(r):
            self._err("zstd_compress()", r)
        if file is not None:
            with open(file, "wb") as fh:
                fh.write(dst.raw[:r])
            return None
        return dst.raw[:r]

    # ---- zstd_decompress_ (src/raw-file.c:150-192, src/raw-file-in.c)
    def zstd_decompress(self, src, type="raw", dctx=None, use_file_streaming=False, **opts):
        self._warnings = []
        L = self.L
        if dctx is None:
            dctx = self.zstd_dctx(**opts)
        if isinstance(src, str) and use_file_streaming:
            parts = []
            out = C.create_string_buffer(FILE_CHUNK)
            r = 1
            with open(src, "rb") as fh:
                while True:
                    chunk = fh.read(FILE_CHUNK)
                    if not chunk:
                        break
                    ib = _InBuffer(C.cast(C.c_char_p(chunk), C.c_void_p), len(chunk), 0)
                    while ib.pos < ib.size or r != 0:
                        ob = _OutBuffer(C.cast(out, C.c_void_p), len(out), 0)
                        r = L.ZSTD_decompressStream(dctx.p, C.byref(ob), C.byref(ib))
                        if L.ZSTD_isError(r):
                            self._err("zstd_decompress_stream_file_()", r)
                        parts.append(out.raw[:ob.pos])
                        if ob.pos < ob.size and ib.pos == ib.size:
                            break
            if r != 0:
                raise RError("zstd_decompress_stream_file_(): truncated input")
            data = b"".join(parts)
        else:
            if isinstance(src, str):
                with open(src, "rb") as fh:
                    src = fh.read()
            src = bytes(src)
            n = L.ZSTD_findFrameCompressedSize(src, len(src))
            if L.ZSTD_isError(n):
                self._err("zstd_decompress()", n)
            cap = L.ZSTD_getFrameContentSize(src, n)
            if cap >= CONTENTSIZE_ERROR:
                raise RError("zstd_decompress(): Frame content size unknown")
            dst = C.create_string_buffer(max(1, cap))
            r = L.ZSTD_decompressDCtx(dctx.p, dst, cap, src, n)
            if L.ZSTD_isError(r):
                self._err("zstd_decompress(): De-compression error", r)
            data = dst.raw[:r]
        return data.decode() if type == "string" else data

    # ---- zstd_train_dictionary_ / zstd_dict_id_ (src/dictionaries.c:23-208)
    def zstd_train_dict_compress(self, samples, size=100000, optim=False, optim_shrink_allow=0):
        self._warnings = []
        L = self.L
        if len(samples) == 0:
            raise RError("zstd_train_dictionary(): No samples provided")
        bufs = [s.encode() if isinstance(s, str) else bytes(s) for s in samples]
        total = sum(len(b) for b in bufs)
        if total < 100 * size:
            self._warnings.append("zstd_train_dictionary() ZSTD documentation recommends training data size 100x dictionary size.\n"
                                  "Only supplied with %.1fx" % (total / max(size, 1)))
        sizes = (C.c_size_t * len(bufs))(*[len(b) for b in bufs])
        dst = C.create_string_buffer(max(1, size))
        r = L.ZDICT_trainFromBuffer(dst, size, b"".join(bufs), sizes, len(bufs))
        if L.ZDICT_isError(r):
            raise RError("zstd_train_dictionary() Training error %s" % L.ZDICT_getErrorName(r).decode())
        return dst.raw[:r]

    def zstd_dict_id(self, d):
        d = bytes(d)
        did = self.L.ZDICT_getDictID(d, len(d))
        return int(did or self.L.ZSTD_getDictID_fromFrame(d, len(d)))

    # ---- zstd_info_ (src/zstd-info.c:60-87)
    def zstd_info(self, src):
        L = self.L
        src = bytes(src)
        fh = _FrameHeader()
        if L.ZSTD_getFrameHeader(C.byref(fh), src, min(len(src), 18)) != 0:
            raise RError("zstd_info(): Couldn't read frame header")
        csize = L.ZSTD_findFrameCompressedSize(src, len(src))
        return {"uncompressed_size": None if fh.frameContentSize == CONTENTSIZE_UNKNOWN else int(fh.frameContentSize),
                "compressed_size": None if L.ZSTD_isError(csize) else int(csize),
                "dict_id": int(fh.dictID), "has_checksum": bool(fh.checksumFlag)}
