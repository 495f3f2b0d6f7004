/* zstdlite_gpu_map.h -- the reference-side binding of INTEGRATION.md section 2 as a header: force-include it
 * (cc -include zstdlite_gpu_map.h) in front of zstdlite's package C files and every libzstd / ZDICT symbol they call
 * (SURVEY.md 8b; call sites under /root/reference/src: cctx.c:72-92,205,222,265-304,352-354; dctx.c:54,99,119,163,181,186,234;
 * raw-file.c:52,74,150,155,189; raw-file-in.c:66,102; raw-file-out.c:89-118; dictionaries.c:52,54,155,198-207; zstd-info.c:61)
 * resolves to the zlg_-prefixed export of libzstdlite_gpu.so -- declarations in zstd.h / zdict.h are renamed with the calls, so the
 * sources stay unmodified and the vendored libzstd can stay linked beside it without a symbol clash.
 * The package's sources are not part of this repository, so no build here compiles them through this header. */
#ifndef ZSTDLITE_GPU_MAP_H
#define ZSTDLITE_GPU_MAP_H
#define ZSTD_isError                          zlg_ZSTD_isError
#define ZSTD_getErrorName                     zlg_ZSTD_getErrorName
#define ZSTD_versionString                    zlg_ZSTD_versionString
#define ZSTD_createCCtx                       zlg_ZSTD_createCCtx
#define ZSTD_freeCCtx                         zlg_ZSTD_freeCCtx
#define ZSTD_CCtx_reset                       zlg_ZSTD_CCtx_reset
#define ZSTD_CCtx_setParameter                zlg_ZSTD_CCtx_setParameter
#define ZSTD_CCtx_getParameter                zlg_ZSTD_CCtx_getParameter
#define ZSTD_CCtx_loadDictionary              zlg_ZSTD_CCtx_loadDictionary
#define ZSTD_CCtx_setPledgedSrcSize           zlg_ZSTD_CCtx_setPledgedSrcSize
#define ZSTD_compressBound                    zlg_ZSTD_compressBound
#define ZSTD_compress2                        zlg_ZSTD_compress2
#define ZSTD_compressStream2                  zlg_ZSTD_compressStream2
#define ZSTD_createDCtx                       zlg_ZSTD_createDCtx
#define ZSTD_freeDCtx                         zlg_ZSTD_freeDCtx
#define ZSTD_DCtx_reset                       zlg_ZSTD_DCtx_reset
#define ZSTD_DCtx_setParameter                zlg_ZSTD_DCtx_setParameter
#define ZSTD_DCtx_getParameter                zlg_ZSTD_DCtx_getParameter
#define ZSTD_DCtx_loadDictionary              zlg_ZSTD_DCtx_loadDictionary
#define ZSTD_findFrameCompressedSize          zlg_ZSTD_findFrameCompressedSize
#define ZSTD_getFrameContentSize              zlg_ZSTD_getFrameContentSize
#define ZSTD_findDecompressedSize             zlg_ZSTD_findDecompressedSize
#define ZSTD_decompressDCtx                   zlg_ZSTD_decompressDCtx
#define ZSTD_decompressStream                 zlg_ZSTD_decompressStream
#define ZSTD_getFrameHeader                   zlg_ZSTD_getFrameHeader
#define ZSTD_getDictID_fromFrame              zlg_ZSTD_getDictID_fromFrame
#define ZSTD_getDictID_fromDict               zlg_ZSTD_getDictID_fromDict
#define ZDICT_getDictID                       zlg_ZDICT_getDictID
#define ZDICT_trainFromBuffer                 zlg_ZDICT_trainFromBuffer
#define ZDICT_optimizeTrainFromBuffer_cover   zlg_ZDICT_optimizeTrainFromBuffer_cover
#define ZDICT_isError                         zlg_ZDICT_isError
#define ZDICT_getErrorName                    zlg_ZDICT_getErrorName
#endif
