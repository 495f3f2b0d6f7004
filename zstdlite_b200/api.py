"""Host-side mirror of zstdlite's R API for the one-shot path, over the C ABI.

Names, argument meaning and error behaviour follow the reference:
  zstd_cctx / zstd_dctx          R/cctx.R:38-48,72-80  -> src/cctx.c:213-315, src/dctx.c:110-197
  zstd_compress / zstd_decompress R/serialize.R:128-156 -> src/raw-file.c:25-118,125-210
  zstd_info                      R/zstd-info.R:19      -> src/zstd-info.c:60-87
  zstd_dict_id                   R/dictionaries.R:27   -> src/dictionaries.c:23-58
plus the batch entry points the benchmark shapes need (SURVEY.md 8b).
Everything computes on the GPU through libzstdlite_gpu.so; there is no CPU path here.
"""
import ctypes as C
import warnings

from . import _lib
from ._lib import CONTENTSIZE_ERROR, CONTENTSIZE_UNKNOWN


class ZstdError(RuntimeError):
    pass


def _check(r, what):
    L = _lib.lib()
    if L.ZSTD_isError(r):
        raise ZstdError(f"{what}: {L.ZSTD_getErrorName(r).decode()}")
    return r


def _as_buffer(x):
    """bytes-like -> (pointer for the C ABI, length, object that keeps the memory alive).  No copy: the library reads the caller's own
    memory, read-only or not, like the reference reads RAW(src) (src/raw-file.c:41-46; str is UTF-8 encoded as there)."""
    if isinstance(x, str):
        x = x.encode("utf-8")
    mv = memoryview(x).cast("B")
    n = mv.nbytes
    if n == 0:
        return C.c_char_p(b""), 0, mv
    import numpy as np
    arr = np.frombuffer(mv, dtype=np.uint8)
    return C.c_void_p(arr.ctypes.data), n, (arr, mv)


# One-shot outputs: a bytes object of the final size that the library writes into directly (PyBytes_FromStringAndSize(NULL, n) is the C API's
# way to make one) -- a ctypes buffer would be zero-filled first and copied twice on the way out, which for a 64 MiB result cost more than
# the decode.  Compressed output, whose size is only known afterwards, goes through an uninitialised numpy array and one copy of the result.
_py = C.pythonapi
_py.PyBytes_FromStringAndSize.restype = C.py_object
_py.PyBytes_FromStringAndSize.argtypes = [C.c_void_p, C.c_ssize_t]
_py.PyBytes_AsString.restype = C.c_void_p
_py.PyBytes_AsString.argtypes = [C.py_object]


def _new_bytes(n):
    """(bytes object of n uninitialised bytes, its address)"""
    b = _py.PyBytes_FromStringAndSize(None, n)
    return b, _py.PyBytes_AsString(b)


def _scratch(n):
    """(uninitialised numpy byte array of n bytes, its address)"""
    import numpy as np
    a = np.empty(max(1, n), dtype=np.uint8)
    return a, a.ctypes.data


class zstd_dctx:
    """zstd_dctx(validate_checksum = TRUE, dict = NULL)  (R/cctx.R:72-80, src/dctx.c:110-197)."""

    def __init__(self, validate_checksum=True, dict=None, num_gpus=0, **unknown):
        """num_gpus (extension): GPUs a batch of HOST buffers is spread over, one contiguous frame range per device (0: the
        ZSTDLITE_GPUS environment variable, default 1).  zstd_cctx takes the reference's own knob for this: num_threads."""
        for k in unknown:
            warnings.warn(f"init_dctx(): Unknown option '{k}'")          # src/dctx.c:171
        L = _lib.lib()
        self._p = L.ZSTD_createDCtx()
        if not self._p:
            raise ZstdError("init_dctx(): Couldn't initialse memory for 'dctx'")
        self.validate_checksum = bool(validate_checksum)
        _check(L.ZSTD_DCtx_setParameter(self._p, _lib.ZSTD_d_forceIgnoreChecksum, 0 if validate_checksum else 1), "init_dctx()")
        if num_gpus:
            _check(L.zl_dctx_set_gpus(self._p, int(num_gpus)), "init_dctx() num_gpus")
        if dict is not None:
            if isinstance(dict, str):
                with open(dict, "rb") as fh:                              # filename form, src/dctx.c:183-190
                    dict = fh.read()
            buf, n, _ = _as_buffer(dict)
            _check(L.ZSTD_DCtx_loadDictionary(self._p, buf, n), "init_dctx() dictionary")

    def settings(self):
        """get_dctx_settings_ (src/dctx.c:228-245; reports forceIgnoreChecksum under the name validate_checksum)."""
        v = C.c_int(0)
        _lib.lib().ZSTD_DCtx_getParameter(self._p, _lib.ZSTD_d_forceIgnoreChecksum, C.byref(v))
        return {"validate_checksum": v.value}

    def set_stream(self, cuda_stream):
        _lib.lib().zl_dctx_set_stream(self._p, C.c_void_p(cuda_stream))

    def set_profile(self, on):
        """True: single-slice, single-stream batches with per-kernel timings; False (default): slice pipeline."""
        _lib.lib().zl_dctx_set_profile(self._p, 1 if on else 0)

    @property
    def launch_count(self):
        return _lib.lib().zl_dctx_launch_count(self._p)

    @property
    def last_kernel_ms(self):
        return _lib.lib().zl_dctx_last_kernel_ms(self._p)

    def __del__(self):
        p = getattr(self, "_p", None)
        if p:
            try:
                _lib.lib().ZSTD_freeDCtx(p)
            except Exception:
                pass
            self._p = None


class zstd_cctx:
    """zstd_cctx(level = 3, num_threads = 1, include_checksum = FALSE, dict = NULL)  (R/cctx.R:38-48, src/cctx.c:213-315)."""

    def __init__(self, level=3, num_threads=1, include_checksum=False, dict=None, level_fallback=False, **unknown):
        """Levels 4 and 5 run the level-3 engine (within 3 % of libzstd at those levels, DESIGN.md section 1).
        level_fallback (extension): levels 6..22 are not implemented on the GPU and are refused ("init_cctx(): Bad compression level",
        src/cctx.c:265) unless this is True (or ZSTDLITE_GPU_LEVEL_FALLBACK=1): then they run the level-3 engine."""
        for k in unknown:
            warnings.warn(f"init_cctx(): Unknown option '{k}'")          # src/cctx.c:288
        L = _lib.lib()
        self._p = L.ZSTD_createCCtx()
        if not self._p:
            raise ZstdError("init_cctx(): Couldn't initialse memory for 'cctx'")
        level = max(-5, min(22, int(level)))                              # src/cctx.c:261-268
        if level_fallback:
            L.zl_cctx_allow_level_fallback(self._p, 1)
        if is_error(L.ZSTD_CCtx_setParameter(self._p, _lib.ZSTD_c_compressionLevel, level)):
            raise ZstdError("init_cctx(): Bad compression level")        # src/cctx.c:265 (levels >= 6: see level_fallback)
        if int(num_threads) > 1:                                          # src/cctx.c:269-277
            _check(L.ZSTD_CCtx_setParameter(self._p, _lib.ZSTD_c_nbWorkers, int(num_threads)), "init_cctx() num_threads")
        _check(L.ZSTD_CCtx_setParameter(self._p, _lib.ZSTD_c_checksumFlag, 1 if include_checksum else 0), "init_cctx() checksum")
        if dict is not None:
            if isinstance(dict, str):
                with open(dict, "rb") as fh:
                    dict = fh.read()
            buf, n, _ = _as_buffer(dict)
            _check(L.ZSTD_CCtx_loadDictionary(self._p, buf, n), "init_cctx() dictionary")

    def settings(self):
        """get_cctx_settings_ (src/cctx.c:343-369)."""
        L = _lib.lib()
        out = {}
        for name, par in (("level", _lib.ZSTD_c_compressionLevel), ("num_threads", _lib.ZSTD_c_nbWorkers),
                          ("include_checksum", _lib.ZSTD_c_checksumFlag)):
            v = C.c_int(0)
            L.ZSTD_CCtx_getParameter(self._p, par, C.byref(v))
            out[name] = v.value
        return out

    def set_stream(self, cuda_stream):
        _lib.lib().zl_cctx_set_stream(self._p, C.c_void_p(cuda_stream))

    @property
    def launch_count(self):
        return _lib.lib().zl_cctx_launch_count(self._p)

    @property
    def last_kernel_ms(self):
        return _lib.lib().zl_cctx_last_kernel_ms(self._p)

    def __del__(self):
        p = getattr(self, "_p", None)
        if p:
            try:
                _lib.lib().ZSTD_freeCCtx(p)
            except Exception:
                pass
            self._p = None


def zstd_compress(src, cctx=None, frame_size=None, seekable=False, **opts):
    """zstd_compress(src, ..., cctx)  (src/raw-file.c:25-118): raw vector or string -> one zstd frame.

    frame_size=N (extension, SURVEY.md 8b): the input is cut into independent frames of N content bytes, returned as one
    standard concatenated stream (zl_compress_split); zstd_decompress(all_frames=True) or any zstd reader decodes it.
    seekable=True (with frame_size): the same frames followed by a seek table in Zstandard's seekable format
    (zl_compress_seekable), so that zstd_decompress_range can decode any byte range without decoding the rest.
    A 1-D contiguous torch.uint8 CUDA tensor `src` gives a CUDA uint8 tensor holding the same bytes as for the data in host memory."""
    L = _lib.lib()
    if cctx is None:
        cctx = zstd_cctx(**opts)
    if getattr(src, "is_cuda", False):
        return _compress_device(L, src, cctx, frame_size, seekable)
    buf, n, _keep = _as_buffer(src)
    L.ZSTD_CCtx_setParameter(cctx._p, _lib.ZSTD_c_stableInBuffer, 1)      # src/cctx.c:70-96
    L.ZSTD_CCtx_setParameter(cctx._p, _lib.ZSTD_c_stableOutBuffer, 1)
    if seekable:
        if not frame_size:
            raise ZstdError("zstd_compress(): seekable=True needs frame_size")
        v = C.c_int(0)
        L.ZSTD_CCtx_getParameter(cctx._p, _lib.ZSTD_c_checksumFlag, C.byref(v))
        cap = _check(L.zl_compress_seekable_bound(n, int(frame_size), v.value), "zstd_compress(): frame_size")
        dst, dptr = _scratch(cap)
        r = L.zl_compress_seekable(cctx._p, dptr, cap, buf, n, int(frame_size), 0)
        _check(r, "zstd_compress(): Compression error")
        return dst[:r].tobytes()
    if frame_size:
        frame_size = int(frame_size)
        nfr = max(1, -(-n // frame_size))
        cap = nfr * L.ZSTD_compressBound(min(n, frame_size))
        dst, dptr = _scratch(cap)
        r = L.zl_compress_split(cctx._p, dptr, cap, buf, n, frame_size, None, 0)
        _check(r, "zstd_compress(): Compression error")
        return dst[:r].tobytes()
    cap = L.ZSTD_compressBound(n)
    dst, dptr = _scratch(cap)
    r = L.ZSTD_compress2(cctx._p, dptr, cap, buf, n)
    _check(r, "zstd_compress(): Compression error")
    return dst[:r].tobytes()


def zstd_decompress(src, type="raw", dctx=None, all_frames=False, out=None, **opts):
    """zstd_decompress(src, type, ..., dctx)  (src/raw-file.c:125-210): first frame only, like the reference.

    all_frames=True is SURVEY.md 8f rank 2: the output is sized with ZSTD_findDecompressedSize (zstd.c:41244) over EVERY
    frame of `src` and the whole stream goes through one ZSTD_decompressDCtx call, which decodes the frames as one GPU
    batch -- so the multi-frame output of zstd_compress(frame_size=...) / zl_compress_split round-trips through this API.

    A 1-D contiguous torch.uint8 CUDA tensor `src` is decoded on its device without leaving it: the frames are found on the device
    (zl_device_frames) and the result is a CUDA uint8 tensor, or a view of `out` (a 1-D contiguous CUDA uint8 tensor) written in place.
    all_frames=True decodes the whole stream (zl_decompress_device); otherwise frame 0 only (a leading skippable frame gives an empty
    result).  Frames without a recorded content size are decoded too; given `out`, its whole size is the capacity.  Unlike the bytes
    path, which looks at frame 0 alone, a tensor source is indexed whole even for frame 0: a structural error anywhere in it (trailing
    padding or garbage included) raises, so pass exactly the stream's bytes."""
    L = _lib.lib()
    if dctx is None:
        dctx = zstd_dctx(**opts)
    if getattr(src, "is_cuda", False):
        return _decompress_device(L, src, type, dctx, all_frames, out)
    if out is not None:
        raise ZstdError("zstd_decompress(): out is only taken for a CUDA source")
    buf, n, _keep = _as_buffer(src)
    if all_frames:
        csize = n
        usize = L.ZSTD_findDecompressedSize(buf, n)
    else:
        csize = L.ZSTD_findFrameCompressedSize(buf, n)
        _check(csize, "zstd_decompress(): Error finding compressed size")
        usize = L.ZSTD_getFrameContentSize(buf, csize)
    if usize >= CONTENTSIZE_ERROR:
        # the reference does not check this (SURVEY.md 3.2) and would try a 2^64 allocation; we raise instead
        raise ZstdError("zstd_decompress(): frame does not record its content size")
    out, optr = _new_bytes(usize)
    L.ZSTD_DCtx_setParameter(dctx._p, _lib.ZSTD_d_stableOutBuffer, 1)     # src/dctx.c:98-103
    r = L.ZSTD_decompressDCtx(dctx._p, optr, usize, buf, csize)
    _check(r, "zstd_decompress(): De-compression error")
    if r != usize:
        out = out[:r]
    return out.decode("utf-8") if type == "string" else out


_DST_TOO_SMALL = 2**64 - 70


def _tensor_out(out, n, like, what):
    import torch
    if out is None:
        return torch.empty(max(1, n), dtype=torch.uint8, device=like.device)
    if not getattr(out, "is_cuda", False) or out.dim() != 1 or not out.is_contiguous() or out.dtype != torch.uint8:
        raise ZstdError(f"{what}: out must be a 1-D contiguous torch.uint8 CUDA tensor")
    torch.cuda.current_stream(out.device).synchronize()
    return out


def _device_frames(L, dctx, buf, n):
    """zl_device_frames into arrays sized by a guess, so that one index build usually answers (a frame takes at least 9 bytes)"""
    import numpy as np
    guess = max(1, min(n // 9 + 1, 1 << 16))
    while True:
        arr = [np.empty(guess, dtype=np.uint64) for _ in range(3)]
        p = C.POINTER(C.c_ulonglong)
        k = _check(L.zl_device_frames(dctx._p, buf, n, *[a.ctypes.data_as(p) for a in arr], guess), "zstd_frames()")
        if k <= guess:
            return [(int(o), int(c), None if d == CONTENTSIZE_UNKNOWN else int(d)) for o, c, d in zip(arr[0][:k], arr[1][:k], arr[2][:k])]
        guess = k


def zstd_frames(src, dctx=None):
    """Every frame of a Zstandard stream in a 1-D contiguous torch.uint8 CUDA tensor, found on its device (zl_device_frames):
    a list of (offset, compressed_size, content_size or None), one per frame; skippable frames are listed with content size 0."""
    import torch
    buf, n, _keep, dev = _source(src)
    if not dev:
        raise ZstdError("zstd_frames(): src must be a CUDA tensor")
    if dctx is None:
        dctx = zstd_dctx()
    torch.cuda.current_stream(src.device).synchronize()                   # the library reads on its own stream
    return _device_frames(_lib.lib(), dctx, buf, n)


def _decompress_device(L, src, type, dctx, all_frames, out):
    import torch
    if type == "string":
        raise ZstdError("zstd_decompress(): type='string' needs a bytes-like source")
    buf, n, _keep, _ = _source(src)
    torch.cuda.current_stream(src.device).synchronize()                   # the library reads on its own stream
    if all_frames and out is not None:                                    # the caller sized the output: one call, one index
        out = _tensor_out(out, 0, src, "zstd_decompress()")
        r = L.zl_decompress_device(dctx._p, C.c_void_p(out.data_ptr()), out.numel(), buf, n)
        _check(r, "zstd_decompress(): De-compression error")
        return out[:r]
    fr = _device_frames(L, dctx, buf, n)
    csize = n
    if not all_frames:                                                    # frame 0 only, like the bytes path
        fr = fr[:1]
        csize = fr[0][1] if fr else 0
    if out is not None:
        out = _tensor_out(out, 0, src, "zstd_decompress()")
        r = L.zl_decompress_device(dctx._p, C.c_void_p(out.data_ptr()), out.numel(), buf, csize)
        _check(r, "zstd_decompress(): De-compression error")
        return out[:r]
    known = sum(f[2] for f in fr if f[2] is not None)
    unknown = [f[1] for f in fr if f[2] is None]
    # a frame without a recorded size regenerates at most 128 KiB per block of >= 3 bytes: start from a smaller guess and grow
    bound = known + sum((c // 3 + 1) << 17 for c in unknown)
    cap = min(bound, known + sum(4 * c + (64 << 10) for c in unknown))
    while True:
        out = _tensor_out(None, cap, src, "zstd_decompress()")
        r = L.zl_decompress_device(dctx._p, C.c_void_p(out.data_ptr()), cap, buf, csize)
        if not unknown or cap >= bound or r != _DST_TOO_SMALL:
            break
        cap = min(bound, 4 * cap)
    _check(r, "zstd_decompress(): De-compression error")
    return out[:r]


def _compress_device(L, src, cctx, frame_size, seekable):
    import torch
    buf, n, _keep, _ = _source(src)
    if n == 0:
        src = torch.zeros(1, dtype=torch.uint8, device=src.device)      # the engine wants a device address even for no bytes
        buf = C.c_void_p(src.data_ptr())
    torch.cuda.current_stream(src.device).synchronize()                   # the library reads on its own stream
    if seekable:
        if not frame_size:
            raise ZstdError("zstd_compress(): seekable=True needs frame_size")
        v = C.c_int(0)
        L.ZSTD_CCtx_getParameter(cctx._p, _lib.ZSTD_c_checksumFlag, C.byref(v))
        cap = _check(L.zl_compress_seekable_bound(n, int(frame_size), v.value), "zstd_compress(): frame_size")
        dst = torch.empty(cap, dtype=torch.uint8, device=src.device)
        r = L.zl_compress_seekable(cctx._p, C.c_void_p(dst.data_ptr()), cap, buf, n, int(frame_size), 1)
    elif frame_size:
        frame_size = int(frame_size)
        cap = max(1, -(-n // frame_size)) * L.ZSTD_compressBound(min(n, frame_size))
        dst = torch.empty(cap, dtype=torch.uint8, device=src.device)
        r = L.zl_compress_split(cctx._p, C.c_void_p(dst.data_ptr()), cap, buf, n, frame_size, None, 1)
    else:
        cap = L.ZSTD_compressBound(n)
        dst = torch.empty(cap, dtype=torch.uint8, device=src.device)
        sp, ss = (C.c_void_p * 1)(buf.value), (C.c_size_t * 1)(n)
        dp, dc, res = (C.c_void_p * 1)(dst.data_ptr()), (C.c_size_t * 1)(cap), (C.c_size_t * 1)(0)
        _check(L.zl_compress_batch(cctx._p, sp, ss, dp, dc, res, 1, 1), "zstd_compress(): Compression error")
        r = res[0]
    _check(r, "zstd_compress(): Compression error")
    return dst[:r]


def _source(src):
    """bytes-like, or a 1-D contiguous torch.uint8 CUDA tensor (duck-typed: torch is not imported for it) ->
    (pointer, length, object that keeps the memory alive, is_device)"""
    if getattr(src, "is_cuda", False):
        if src.dim() != 1 or not src.is_contiguous() or str(src.dtype) != "torch.uint8":
            raise ZstdError("a device source must be a 1-D contiguous torch.uint8 CUDA tensor")
        return C.c_void_p(src.data_ptr() or None), src.numel(), src, True
    buf, n, keep = _as_buffer(src)
    return buf, n, keep, False


def _seek_table(buf, n, dev):
    L = _lib.lib()
    k = _check(L.zl_seekable_frames(buf, n, 1 if dev else 0, None, None, None, 0, None), "zstd_seek_table()")
    cs, ds, ck, has = (C.c_uint * max(1, k))(), (C.c_uint * max(1, k))(), (C.c_uint * max(1, k))(), C.c_int(0)
    _check(L.zl_seekable_frames(buf, n, 1 if dev else 0, cs, ds, ck, k, C.byref(has)), "zstd_seek_table()")
    return [(cs[i], ds[i], ck[i] if has.value else None) for i in range(k)]


def zstd_seek_table(src):
    """The seek table of a seekable stream (zstd_compress(..., seekable=True), or any writer of Zstandard's seekable format):
    a list of (compressed_size, decompressed_size, checksum or None), one per frame.  `src` is bytes-like or a CUDA tensor."""
    buf, n, _keep, dev = _source(src)
    if dev:
        import torch
        torch.cuda.current_stream(src.device).synchronize()
    return _seek_table(buf, n, dev)


def zstd_decompress_range(src, offset, length, dctx=None, type="raw", out=None, **opts):
    """Bytes [offset, offset + length) of a seekable stream's content, clamped to its end; only the frames the range touches are decoded
    (zl_decompress_range).  A bytes-like `src` gives bytes (str with type="string"); a CUDA tensor gives a CUDA uint8 tensor, or the
    first bytes of `out` (a CUDA uint8 tensor) written in place.  The table's checksums are verified unless validate_checksum=False."""
    L = _lib.lib()
    if dctx is None:
        dctx = zstd_dctx(**opts)
    buf, n, _keep, dev = _source(src)
    offset, length = int(offset), int(length)
    if offset < 0 or length < 0:
        raise ZstdError("zstd_decompress_range(): offset and length must be >= 0")
    if dev:
        import torch
        torch.cuda.current_stream(src.device).synchronize()               # the library reads on its own stream
    total = sum(d for _, d, _ in _seek_table(buf, n, dev))
    want = max(0, min(length, total - offset))
    if dev:
        if out is None:
            out = torch.empty(max(1, want), dtype=torch.uint8, device=src.device)
        elif not getattr(out, "is_cuda", False) or out.dim() != 1 or not out.is_contiguous() or out.dtype != torch.uint8:
            raise ZstdError("zstd_decompress_range(): out must be a 1-D contiguous torch.uint8 CUDA tensor")
        else:
            torch.cuda.current_stream(out.device).synchronize()
        r = L.zl_decompress_range(dctx._p, C.c_void_p(out.data_ptr()), out.numel(), buf, n, offset, length, 1)
        _check(r, "zstd_decompress_range(): De-compression error")
        return out[:r]
    if out is not None:
        raise ZstdError("zstd_decompress_range(): out is only taken for a CUDA source")
    res, rptr = _new_bytes(want)
    r = L.zl_decompress_range(dctx._p, rptr, want, buf, n, offset, length, 0)
    _check(r, "zstd_decompress_range(): De-compression error")
    return res.decode("utf-8") if type == "string" else res


def zstd_decompress_ranges(src, ranges, dctx=None, type="raw", out=None, **opts):
    """Many byte ranges of one seekable stream in one call (zl_decompress_ranges): `ranges` is a sequence of (offset, length) pairs, each
    clamped to the stream's end like zstd_decompress_range.  The table is read once and every touched frame is decoded once, however many
    ranges share it.  A bytes-like `src` gives a list of bytes (str with type="string"); a CUDA tensor gives a list of CUDA uint8 tensors,
    views into one tensor that holds the ranges back to back in request order -- `out` (a 1-D contiguous CUDA uint8 tensor) when given.
    A failed range raises ZstdError naming the first failing range's index.  The table's checksums are verified unless
    validate_checksum=False."""
    import numpy as np
    L = _lib.lib()
    if dctx is None:
        dctx = zstd_dctx(**opts)
    buf, n, _keep, dev = _source(src)
    rg = np.asarray(ranges, dtype=np.int64).reshape(-1, 2) if len(ranges) else np.zeros((0, 2), dtype=np.int64)
    if (rg < 0).any():
        raise ZstdError("zstd_decompress_ranges(): offsets and lengths must be >= 0")
    k = len(rg)
    if dev:
        import torch
        torch.cuda.current_stream(src.device).synchronize()               # the library reads on its own stream
    try:
        total = sum(d for _, d, _ in _seek_table(buf, n, dev))
    except ZstdError:
        total = 0                                                         # the call reports the table's error for every range
    offs, lens = rg[:, 0].astype(np.uint64), rg[:, 1].astype(np.uint64)
    want = np.clip(np.minimum(rg[:, 1], total - rg[:, 0]), 0, None).astype(np.uint64)
    at = np.concatenate(([0], np.cumsum(want))).astype(np.uint64)          # each range's place in the packed output
    if dev:
        if out is None:
            out = torch.empty(max(1, int(at[-1])), dtype=torch.uint8, device=src.device)
        elif not getattr(out, "is_cuda", False) or out.dim() != 1 or not out.is_contiguous() or out.dtype != torch.uint8:
            raise ZstdError("zstd_decompress_ranges(): out must be a 1-D contiguous torch.uint8 CUDA tensor")
        else:
            torch.cuda.current_stream(out.device).synchronize()
        base = out.data_ptr()
        caps = np.clip(np.minimum(want.astype(np.int64), out.numel() - at[:-1].astype(np.int64)), 0, None).astype(np.uint64)
        dsts = base + at[:-1]
        keep = None
    else:
        if out is not None:
            raise ZstdError("zstd_decompress_ranges(): out is only taken for a CUDA source")
        keep = [_new_bytes(int(w)) for w in want]
        dsts = np.array([p for _, p in keep], dtype=np.uint64)
        caps = want
    srcs = np.full(k, C.cast(buf, C.c_void_p).value or 0, dtype=np.uint64)
    sizes = np.full(k, n, dtype=np.uint64)
    res = np.zeros(k, dtype=np.uint64)
    pp, psz = C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)
    _check(L.zl_decompress_ranges(dctx._p, srcs.ctypes.data_as(pp), sizes.ctypes.data_as(psz), offs.ctypes.data_as(psz),
                                  lens.ctypes.data_as(psz), dsts.ctypes.data_as(pp), caps.ctypes.data_as(psz), res.ctypes.data_as(psz),
                                  k, 1 if dev else 0), "zstd_decompress_ranges()")
    failed = np.flatnonzero(res > np.uint64(2**64 - 121))                 # error codes are the last 120 values of size_t
    if len(failed):
        i = int(failed[0])
        raise ZstdError(f"zstd_decompress_ranges(): range {i}: {L.ZSTD_getErrorName(int(res[i])).decode()}")
    if dev:
        return list(torch.split(out[:int(at[-1])], want.tolist()))
    return [b.decode("utf-8") if type == "string" else b for b, _ in keep]


def zstd_serialize(obj, cctx=None, frame_size=None, **opts):
    """zstd_serialize(robj, ..., cctx)  (R/serialize.R:56, src/serialize.c:41-118): serialize the object to bytes, compress them
    as one frame.  The reference serializes with R_Serialize (version 3, binary); R is not in this image, so this host mirror
    uses Python's own binary serialization (pickle protocol 5) -- the codec path behind it is the same ZSTD_compress2 call."""
    import pickle
    return zstd_compress(pickle.dumps(obj, protocol=5), cctx=cctx, frame_size=frame_size, **opts)


def zstd_unserialize(src, dctx=None, **opts):
    """zstd_unserialize(src, ..., dctx)  (R/serialize.R:74, src/serialize.c:141-215): decompress, then unserialize.
    Like the reference this reads content sizes from the frame headers; every frame of `src` is decoded (8f rank 2).

    WARNING: pickle stands in for R's unserialize() in this mirror, and unpickling runs code named by the payload.  Only the
    plain-data types zstd_serialize() is used with in the tests are accepted (a restricted Unpickler); anything else raises
    pickle.UnpicklingError -- never feed this frames from an untrusted source expecting more than that."""
    import io
    return _SafeUnpickler(io.BytesIO(zstd_decompress(src, dctx=dctx, all_frames=True, **opts))).load()


import pickle as _pickle


class _SafeUnpickler(_pickle.Unpickler):
    """Plain data only: builtins' containers / scalars and numpy arrays (what a data.frame-like payload needs)."""
    _ALLOWED = {("builtins", n) for n in ("list", "dict", "tuple", "set", "frozenset", "bytes", "bytearray", "str", "int", "float", "complex", "bool", "slice", "range")} | {
        ("numpy.core.multiarray", "_reconstruct"), ("numpy._core.multiarray", "_reconstruct"), ("numpy", "ndarray"), ("numpy", "dtype"),
        ("numpy.core.multiarray", "scalar"), ("numpy._core.multiarray", "scalar"), ("numpy._core.numeric", "_frombuffer"), ("numpy.core.numeric", "_frombuffer"),
        ("collections", "OrderedDict")}

    def find_class(self, module, name):
        if (module, name) in self._ALLOWED:
            return super().find_class(module, name)
        raise _pickle.UnpicklingError(f"zstd_unserialize: {module}.{name} is not plain data; refusing to unpickle it")


_OUTSIZE, _INSIZE = 131591, 131072          # static buffer sizes of the reference's streaming writers (src/raw-file-out.c:23-24)


def zstd_compress_stream(src, write, cctx=None, **opts):
    """The reference's streaming writer loop (src/raw-file-out.c:74-118, use_file_streaming=TRUE): pledge the size, feed
    ZSTD_compressStream2 in 128 KiB chunks with ZSTD_e_continue, finish with ZSTD_e_end; `write(bytes)` receives the output."""
    L = _lib.lib()
    if cctx is None:
        cctx = zstd_cctx(**opts)
    if isinstance(src, str):
        src = src.encode("utf-8")
    data = bytes(memoryview(src).cast("B"))
    n = len(data)
    _check(L.ZSTD_CCtx_setPledgedSrcSize(cctx._p, n), "zstd_compress_stream(): pledged size")
    obuf = C.create_string_buffer(_OUTSIZE)
    pos = 0
    while True:
        chunk = data[pos:pos + _INSIZE]
        pos += len(chunk)
        last = pos >= n
        ib = C.create_string_buffer(chunk, max(1, len(chunk)))
        inb = _lib.InBuffer(C.cast(ib, C.c_void_p), len(chunk), 0)
        while True:
            outb = _lib.OutBuffer(C.cast(obuf, C.c_void_p), _OUTSIZE, 0)
            rem = L.ZSTD_compressStream2(cctx._p, C.byref(outb), C.byref(inb), _lib.ZSTD_e_end if last else _lib.ZSTD_e_continue)
            _check(rem, "zstd_compress_stream(): Compression error")
            if outb.pos:
                write(obuf.raw[:outb.pos])
            if (rem == 0) if last else (inb.pos == inb.size):
                break
        if last:
            return


def zstd_decompress_stream(read, dctx=None, out_chunk=131702, **opts):
    """The reference's streaming reader loop (src/raw-file-in.c:94-104): `read(n)` supplies compressed bytes (b"" at the end);
    ZSTD_decompressStream is called until the input is consumed and the decoder holds no more output."""
    L = _lib.lib()
    if dctx is None:
        dctx = zstd_dctx(**opts)
    out = bytearray()
    obuf = C.create_string_buffer(out_chunk)
    status = 0
    while True:
        chunk = read(_INSIZE)
        if not chunk:
            break
        ib = C.create_string_buffer(chunk, len(chunk))
        inb = _lib.InBuffer(C.cast(ib, C.c_void_p), len(chunk), 0)
        while True:
            outb = _lib.OutBuffer(C.cast(obuf, C.c_void_p), out_chunk, 0)
            status = L.ZSTD_decompressStream(dctx._p, C.byref(outb), C.byref(inb))
            _check(status, "zstd_decompress_stream(): De-compression error")
            out += obuf.raw[:outb.pos]
            if inb.pos == inb.size and outb.pos < out_chunk:
                break
    if status != 0:
        raise ZstdError("zstd_decompress_stream(): input ends inside a frame")
    return bytes(out)


def zstd_info(src):
    """zstd_info(src)  (src/zstd-info.c:60-87)."""
    L = _lib.lib()
    if isinstance(src, str):
        with open(src, "rb") as fh:
            src = fh.read(18)
    buf, n, _keep = _as_buffer(src)
    fh = _lib.FrameHeader()
    r = L.ZSTD_getFrameHeader(C.byref(fh), buf, min(n, 18))
    if r != 0:
        raise ZstdError("zstd_info(): Couldn't read frame header")
    whole, m, _k = _as_buffer(src)
    csize = L.ZSTD_findFrameCompressedSize(whole, m)
    return {"uncompressed_size": None if fh.frameContentSize == CONTENTSIZE_UNKNOWN else int(fh.frameContentSize),
            "compressed_size": None if L.ZSTD_isError(csize) else int(csize),
            "dict_id": int(fh.dictID), "has_checksum": bool(fh.checksumFlag)}


def zstd_dict_id(x):
    """zstd_dict_id(dict | compressed frame)  (src/dictionaries.c:23-58)."""
    L = _lib.lib()
    buf, n, _keep = _as_buffer(x)
    did = L.ZDICT_getDictID(buf, n)
    if did == 0:
        did = L.ZSTD_getDictID_fromFrame(buf, n)
    return int(did)


def zstd_train_dict_compress(samples, size=100000, optim=False, optim_shrink_allow=0):
    """zstd_train_dict_compress(samples, size, optim, optim_shrink_allow)  (R/dictionaries.R:65, src/dictionaries.c:75-208):
    `samples` is a list of bytes-like objects (each >= 8 bytes) or strings; returns a Zstandard dictionary of at most `size`
    bytes, trained on the GPU (csrc/zl_dict_train.cuh)."""
    L = _lib.lib()
    if not isinstance(samples, (list, tuple)):
        raise ZstdError("zstd_train_dictionary(): samples must be provided as a list of raw vectors or character strings")
    if len(samples) == 0:
        raise ZstdError("zstd_train_dictionary(): No samples provided")
    bufs = []
    for s in samples:
        if isinstance(s, str):
            s = s.encode("utf-8")
        else:
            s = bytes(memoryview(s).cast("B"))
            if len(s) < 8:
                raise ZstdError("zstd_train_dictionary(): When samples are raw vectors, all vector lengths must be >= 8 bytes")
        bufs.append(s)
    total = sum(len(b) for b in bufs)
    size = int(size)
    if total < 100 * size:                                               # src/dictionaries.c:104-106
        warnings.warn("zstd_train_dictionary() ZSTD documentation recommends training data size 100x dictionary size.\n"
                      "Only supplied with %.1fx" % (total / max(size, 1)))
    blob = b"".join(bufs)
    sizes = (C.c_size_t * len(bufs))(*[len(b) for b in bufs])
    dst = C.create_string_buffer(max(1, size))
    if not optim:
        r = L.ZDICT_trainFromBuffer(dst, size, blob, sizes, len(bufs))
    else:
        par = _lib.CoverParams()
        if int(optim_shrink_allow) > 0:
            par.shrinkDict, par.shrinkDictMaxRegression = 1, int(optim_shrink_allow)
        r = L.ZDICT_optimizeTrainFromBuffer_cover(dst, size, blob, sizes, len(bufs), C.byref(par))
    if L.ZDICT_isError(r):
        raise ZstdError("zstd_train_dictionary() Training error %s" % L.ZDICT_getErrorName(r).decode())
    return dst.raw[:r]


def zstd_train_dict_serialize(samples, size=100000, optim=False, optim_shrink_allow=0):
    """zstd_train_dict_serialize(samples, ...)  (R/dictionaries.R:87-93): every sample object is serialized first (pickle here,
    R's serialize() in the reference), for use with zstd_serialize() / zstd_unserialize()."""
    import pickle
    if not isinstance(samples, (list, tuple)):
        raise ZstdError("zstd_train_dict_serialize(): samples must be a list")
    return zstd_train_dict_compress([pickle.dumps(x, protocol=5) for x in samples], size, optim, optim_shrink_allow)


def zstd_version():
    return _lib.lib().ZSTD_versionString().decode()


# ---- batch extension ---------------------------------------------------------------------------------
def _ptr_arrays(ptrs, sizes):
    n = len(ptrs)
    return (C.c_void_p * n)(*ptrs), (C.c_size_t * n)(*sizes)


def decompress_batch(dctx, src_ptrs, src_sizes, dst_ptrs, dst_caps, device=True):
    """zl_decompress_batch: lists of raw addresses (device pointers when device=True). Returns list of sizes/error codes."""
    L = _lib.lib()
    n = len(src_ptrs)
    sp, ss = _ptr_arrays(src_ptrs, src_sizes)
    dp, ds = _ptr_arrays(dst_ptrs, dst_caps)
    res = (C.c_size_t * n)()
    r = L.zl_decompress_batch(dctx._p, sp, ss, dp, ds, res, n, 1 if device else 0)
    _check(r, "zl_decompress_batch()")
    return list(res)


def compress_batch(cctx, src_ptrs, src_sizes, dst_ptrs, dst_caps, device=True):
    L = _lib.lib()
    n = len(src_ptrs)
    sp, ss = _ptr_arrays(src_ptrs, src_sizes)
    dp, ds = _ptr_arrays(dst_ptrs, dst_caps)
    res = (C.c_size_t * n)()
    r = L.zl_compress_batch(cctx._p, sp, ss, dp, ds, res, n, 1 if device else 0)
    _check(r, "zl_compress_batch()")
    return list(res)


class BatchPlan:
    """Pre-built ctypes argument arrays for repeated batch calls on the same buffers (bench loop)."""

    def __init__(self, src_ptrs, src_sizes, dst_ptrs, dst_caps):
        self.n = len(src_ptrs)
        self.sp, self.ss = _ptr_arrays(src_ptrs, src_sizes)
        self.dp, self.ds = _ptr_arrays(dst_ptrs, dst_caps)
        self.res = (C.c_size_t * self.n)()

    def decompress(self, dctx, device=True):
        r = _lib.lib().zl_decompress_batch(dctx._p, self.sp, self.ss, self.dp, self.ds, self.res, self.n, 1 if device else 0)
        _check(r, "zl_decompress_batch()")
        return self.res

    def compress(self, cctx, device=True):
        r = _lib.lib().zl_compress_batch(cctx._p, self.sp, self.ss, self.dp, self.ds, self.res, self.n, 1 if device else 0)
        _check(r, "zl_compress_batch()")
        return self.res


def is_error(code):
    return bool(_lib.lib().ZSTD_isError(code))


def error_name(code):
    return _lib.lib().ZSTD_getErrorName(code).decode()
