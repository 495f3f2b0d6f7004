"""ctypes binding of libzstdlite_gpu.so (C ABI: include/zstdlite_gpu.h).

The library is the product: if it is missing this module raises -- there is no CPU fallback.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ZSTDLITE_GPU_LIB") or os.path.join(_HERE, "libzstdlite_gpu.so")      # (override: development A/B builds)

CONTENTSIZE_UNKNOWN = 2**64 - 1
CONTENTSIZE_ERROR = 2**64 - 2
ZSTD_c_compressionLevel, ZSTD_c_checksumFlag, ZSTD_c_nbWorkers = 100, 201, 400
ZSTD_c_windowLog = 101
ZSTD_c_stableInBuffer, ZSTD_c_stableOutBuffer = 1006, 1007
ZSTD_d_stableOutBuffer, ZSTD_d_forceIgnoreChecksum = 1001, 1002


class InBuffer(C.Structure):
    _fields_ = [("src", C.c_void_p), ("size", C.c_size_t), ("pos", C.c_size_t)]


class OutBuffer(C.Structure):
    _fields_ = [("dst", C.c_void_p), ("size", C.c_size_t), ("pos", C.c_size_t)]


ZSTD_e_continue, ZSTD_e_flush, ZSTD_e_end = 0, 1, 2


class ZdictParams(C.Structure):
    _fields_ = [("compressionLevel", C.c_int), ("notificationLevel", C.c_uint), ("dictID", C.c_uint)]


class CoverParams(C.Structure):
    _fields_ = [("k", C.c_uint), ("d", C.c_uint), ("steps", C.c_uint), ("nbThreads", C.c_uint), ("splitPoint", C.c_double),
                ("shrinkDict", C.c_uint), ("shrinkDictMaxRegression", C.c_uint), ("zParams", ZdictParams)]


class FrameHeader(C.Structure):
    _fields_ = [("frameContentSize", C.c_ulonglong), ("windowSize", C.c_ulonglong), ("blockSizeMax", C.c_uint),
                ("frameType", C.c_int), ("headerSize", C.c_uint), ("dictID", C.c_uint), ("checksumFlag", C.c_uint),
                ("_reserved1", C.c_uint), ("_reserved2", C.c_uint)]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or make -C zstdlite_b200/csrc). zstdlite_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH, mode=os.RTLD_LOCAL)
    vp, sz, pp, psz = C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)
    sig = {
        "ZSTD_isError": (C.c_uint, [sz]), "ZSTD_getErrorName": (C.c_char_p, [sz]), "ZSTD_versionString": (C.c_char_p, []),
        "zl_backend_string": (C.c_char_p, []),
        "ZSTD_createDCtx": (vp, []), "ZSTD_freeDCtx": (sz, [vp]), "ZSTD_DCtx_reset": (sz, [vp, C.c_int]),
        "ZSTD_DCtx_setParameter": (sz, [vp, C.c_int, C.c_int]), "ZSTD_DCtx_getParameter": (sz, [vp, C.c_int, C.POINTER(C.c_int)]),
        "ZSTD_DCtx_loadDictionary": (sz, [vp, vp, sz]),
        "ZSTD_findFrameCompressedSize": (sz, [vp, sz]), "ZSTD_getFrameContentSize": (C.c_ulonglong, [vp, sz]),
        "ZSTD_findDecompressedSize": (C.c_ulonglong, [vp, sz]),
        "ZSTD_decompressDCtx": (sz, [vp, vp, sz, vp, sz]),
        "ZSTD_getFrameHeader": (sz, [C.POINTER(FrameHeader), vp, sz]), "ZSTD_getDictID_fromFrame": (C.c_uint, [vp, sz]),
        "ZSTD_getDictID_fromDict": (C.c_uint, [vp, sz]), "ZDICT_getDictID": (C.c_uint, [vp, sz]),
        "zl_decompress_batch": (sz, [vp, pp, psz, pp, psz, psz, sz, C.c_int]),
        "zl_dctx_set_stream": (sz, [vp, vp]), "zl_dctx_set_profile": (sz, [vp, C.c_int]), "zl_dctx_launch_count": (C.c_ulonglong, [vp]), "zl_dctx_last_kernel_ms": (C.c_double, [vp]),
        "zl_dctx_last_stage_ms": (C.c_double, [vp, C.c_int]), "zl_dctx_set_gpus": (sz, [vp, C.c_int]),
        # compression half
        "ZSTD_createCCtx": (vp, []), "ZSTD_freeCCtx": (sz, [vp]), "ZSTD_CCtx_reset": (sz, [vp, C.c_int]),
        "ZSTD_CCtx_setParameter": (sz, [vp, C.c_int, C.c_int]), "ZSTD_CCtx_getParameter": (sz, [vp, C.c_int, C.POINTER(C.c_int)]),
        "ZSTD_CCtx_loadDictionary": (sz, [vp, vp, sz]), "ZSTD_CCtx_setPledgedSrcSize": (sz, [vp, C.c_ulonglong]),
        "ZSTD_compressBound": (sz, [sz]), "ZSTD_compress2": (sz, [vp, vp, sz, vp, sz]),
        "zl_compress_batch": (sz, [vp, pp, psz, pp, psz, psz, sz, C.c_int]),
        "zl_compress_split": (sz, [vp, vp, sz, vp, sz, sz, psz, C.c_int]),
        # seekable streams
        "zl_compress_seekable": (sz, [vp, vp, sz, vp, sz, sz, C.c_int]), "zl_compress_seekable_bound": (sz, [sz, sz, C.c_int]),
        "zl_seekable_frames": (sz, [vp, sz, C.c_int, C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.POINTER(C.c_uint), sz, C.POINTER(C.c_int)]),
        "zl_decompress_range": (sz, [vp, vp, sz, vp, sz, sz, sz, C.c_int]),
        "zl_decompress_ranges": (sz, [vp, pp, psz, psz, psz, pp, psz, psz, sz, C.c_int]),
        # streams in device memory
        "zl_device_frames": (sz, [vp, vp, sz, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong), sz]),
        "zl_decompress_device": (sz, [vp, vp, sz, vp, sz]),
        "zl_cctx_set_stream": (sz, [vp, vp]), "zl_cctx_launch_count": (C.c_ulonglong, [vp]), "zl_cctx_last_kernel_ms": (C.c_double, [vp]),
        "zl_cctx_last_stage_ms": (C.c_double, [vp, C.c_int]),
        "zl_cctx_allow_level_fallback": (sz, [vp, C.c_int]), "zl_cctx_engine_level": (C.c_int, [vp]),
        # dictionary training
        "ZDICT_trainFromBuffer": (sz, [vp, sz, vp, psz, C.c_uint]),
        "ZDICT_optimizeTrainFromBuffer_cover": (sz, [vp, sz, vp, psz, C.c_uint, C.POINTER(CoverParams)]),
        "ZDICT_isError": (C.c_uint, [sz]), "ZDICT_getErrorName": (C.c_char_p, [sz]),
        # streaming entry points (whole-frame buffering over the same engine)
        "ZSTD_compressStream2": (sz, [vp, C.POINTER(OutBuffer), C.POINTER(InBuffer), C.c_int]),
        "ZSTD_decompressStream": (sz, [vp, C.POINTER(OutBuffer), C.POINTER(InBuffer)]),
    }
    missing = []
    for name, (res, args) in sig.items():
        try:
            fn = getattr(L, name)
        except AttributeError:
            missing.append(name)
            continue
        fn.restype = res
        fn.argtypes = args
    L._missing = missing
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "ZSTD_isError", "ZSTD_getErrorName", "ZSTD_versionString", "ZSTD_createCCtx", "ZSTD_freeCCtx", "ZSTD_CCtx_reset",
    "ZSTD_CCtx_setParameter", "ZSTD_CCtx_getParameter", "ZSTD_CCtx_loadDictionary", "ZSTD_CCtx_setPledgedSrcSize",
    "ZSTD_compressBound", "ZSTD_compress2", "ZSTD_createDCtx", "ZSTD_freeDCtx", "ZSTD_DCtx_reset", "ZSTD_DCtx_setParameter",
    "ZSTD_DCtx_getParameter", "ZSTD_DCtx_loadDictionary", "ZSTD_findFrameCompressedSize", "ZSTD_getFrameContentSize", "ZSTD_findDecompressedSize",
    "ZSTD_decompressDCtx", "ZSTD_compressStream2", "ZSTD_decompressStream", "ZSTD_getFrameHeader", "ZSTD_getDictID_fromFrame", "ZSTD_getDictID_fromDict", "ZDICT_getDictID",
    "ZDICT_trainFromBuffer", "ZDICT_optimizeTrainFromBuffer_cover", "ZDICT_isError", "ZDICT_getErrorName",
    "zl_decompress_batch", "zl_compress_batch", "zl_compress_split", "zl_dctx_set_stream", "zl_dctx_set_profile", "zl_cctx_set_stream",
    "zl_dctx_launch_count", "zl_cctx_launch_count", "zl_dctx_last_kernel_ms", "zl_cctx_last_kernel_ms", "zl_dctx_last_stage_ms", "zl_cctx_last_stage_ms", "zl_backend_string",
    "zl_cctx_allow_level_fallback", "zl_cctx_engine_level", "zl_dctx_set_gpus",
    "zl_compress_seekable", "zl_compress_seekable_bound", "zl_seekable_frames", "zl_decompress_range", "zl_decompress_ranges",
    "zl_device_frames", "zl_decompress_device",
]
