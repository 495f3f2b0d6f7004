/*
 * zstdlite_gpu.h -- C ABI of libzstdlite_gpu.so, the B200-native Zstandard engine that stands in
 * for the vendored libzstd on zstdlite's ONE-SHOT path.
 *
 * Every ZSTD_* entry point below has the exact signature of the libzstd 1.5.6 symbol that the
 * reference's C layer calls (citations: file:line under /root/reference).  The library exports each
 * of them twice: under the canonical name and under a `zlg_` prefix (zlg_ZSTD_compress2, ...) so a
 * package that keeps the vendored libzstd for its streaming/ZDICT code can bind the one-shot path
 * explicitly (see INTEGRATION.md).  There is no CPU fallback: when no CUDA device is usable the
 * compute entry points return a libzstd-style error code (ZSTD_isError() is true).
 *
 * Plain C: pointers and sizes only.
 */
#ifndef ZSTDLITE_GPU_H
#define ZSTDLITE_GPU_H
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ZSTD_CCtx_s ZSTD_CCtx;
typedef struct ZSTD_DCtx_s ZSTD_DCtx;

/* src/zstd/zstd.h:566-568 */
typedef enum { ZSTD_reset_session_only = 1, ZSTD_reset_parameters = 2, ZSTD_reset_session_and_parameters = 3 } ZSTD_ResetDirective;
/* the parameters zstdlite sets: src/zstd/zstd.h:333,440,449,507-508,2083,2103 and 638-639,2422,2433 */
typedef enum {
    ZSTD_c_compressionLevel = 100, ZSTD_c_windowLog = 101, ZSTD_c_checksumFlag = 201, ZSTD_c_nbWorkers = 400,
    ZSTD_c_stableInBuffer = 1006, ZSTD_c_stableOutBuffer = 1007
} ZSTD_cParameter;
typedef enum { ZSTD_d_windowLogMax = 100, ZSTD_d_stableOutBuffer = 1001, ZSTD_d_forceIgnoreChecksum = 1002 } ZSTD_dParameter;
typedef enum { ZSTD_frame = 0, ZSTD_skippableFrame = 1 } ZSTD_frameType_e;
/* src/zstd/zstd.h:1472-1482 */
typedef struct {
    unsigned long long frameContentSize;
    unsigned long long windowSize;
    unsigned blockSizeMax;
    ZSTD_frameType_e frameType;
    unsigned headerSize;
    unsigned dictID;
    unsigned checksumFlag;
    unsigned _reserved1;
    unsigned _reserved2;
} ZSTD_frameHeader;

#define ZSTD_CONTENTSIZE_UNKNOWN (0ULL - 1)   /* src/zstd/zstd.h:190 */
#define ZSTD_CONTENTSIZE_ERROR   (0ULL - 2)   /* src/zstd/zstd.h:191 */

/* ---- errors / version: src/cctx.c, src/dctx.c, src/raw-file.c, src/serialize.c (43 + 27 call sites) ---- */
unsigned    ZSTD_isError(size_t code);                       /* zstd.c:15758 */
const char* ZSTD_getErrorName(size_t code);                  /* zstd.c:15762, strings zstd.c:3590-3630 */
const char* ZSTD_versionString(void);                        /* zstd.c:15748; src/serialize.c:27 */

/* ---- compression context: src/cctx.c:205,222,72-92,265-304,352-354 ---- */
ZSTD_CCtx* ZSTD_createCCtx(void);                                                   /* zstd.c:22610 */
size_t     ZSTD_freeCCtx(ZSTD_CCtx* cctx);                                          /* zstd.c:22693 */
size_t     ZSTD_CCtx_reset(ZSTD_CCtx* cctx, ZSTD_ResetDirective reset);             /* zstd.c:23872 */
size_t     ZSTD_CCtx_setParameter(ZSTD_CCtx* cctx, ZSTD_cParameter param, int v);   /* zstd.c:23223 */
size_t     ZSTD_CCtx_getParameter(const ZSTD_CCtx* cctx, ZSTD_cParameter param, int* v); /* zstd.c:23531 */
size_t     ZSTD_CCtx_loadDictionary(ZSTD_CCtx* cctx, const void* dict, size_t dictSize); /* zstd.c:23826 (copies) */
size_t     ZSTD_CCtx_setPledgedSrcSize(ZSTD_CCtx* cctx, unsigned long long pledged); /* zstd.c:23735 */

/* ---- one-shot compression: src/raw-file.c:52,74; src/serialize.c:73,91 ---- */
size_t ZSTD_compressBound(size_t srcSize);                                          /* zstd.c:22583 */
size_t ZSTD_compress2(ZSTD_CCtx* cctx, void* dst, size_t dstCapacity, const void* src, size_t srcSize); /* zstd.c:28949 */

/* ---- decompression context: src/dctx.c:54,99,119,163,181,186,234 ---- */
ZSTD_DCtx* ZSTD_createDCtx(void);                                                   /* zstd.c:40913 */
size_t     ZSTD_freeDCtx(ZSTD_DCtx* dctx);                                          /* zstd.c:40927 */
size_t     ZSTD_DCtx_reset(ZSTD_DCtx* dctx, ZSTD_ResetDirective reset);             /* zstd.c:42548 */
size_t     ZSTD_DCtx_setParameter(ZSTD_DCtx* dctx, ZSTD_dParameter param, int v);   /* zstd.c:42507 */
size_t     ZSTD_DCtx_getParameter(ZSTD_DCtx* dctx, ZSTD_dParameter param, int* v);  /* zstd.c:42478 */
size_t     ZSTD_DCtx_loadDictionary(ZSTD_DCtx* dctx, const void* dict, size_t dictSize); /* zstd.c:42321 (copies) */

/* ---- one-shot decompression: src/raw-file.c:150,155,189; src/serialize.c:171,177,197 ---- */
size_t             ZSTD_findFrameCompressedSize(const void* src, size_t srcSize);   /* zstd.c:41410 */
unsigned long long ZSTD_getFrameContentSize(const void* src, size_t srcSize);       /* zstd.c:41170 */
unsigned long long ZSTD_findDecompressedSize(const void* src, size_t srcSize);      /* zstd.c:41244; sums every frame of a stream (SURVEY.md 8f rank 2) */
size_t ZSTD_decompressDCtx(ZSTD_DCtx* dctx, void* dst, size_t dstCapacity, const void* src, size_t srcSize); /* zstd.c:41798 */

/* ---- streaming entry points (SURVEY.md 8f rank 3): src/raw-file-out.c:95,113; src/raw-file-in.c:102; src/serialize-*-out.c,
 *      src/serialize-*-in.c; src/zstdfile.c:238,362,475,511.  Implemented over the same GPU engine by buffering whole frames on
 *      the host: input is accumulated until ZSTD_e_end (compress) / until a complete frame has arrived (decompress), then the
 *      one-shot kernels run and the result is handed out in the caller's chunk sizes.  Output is one standard frame whose
 *      header records the content size, interchangeable with the one-shot path (tests/testthat/test-compress-raw.R:61-89). ---- */
typedef struct { const void* src; size_t size; size_t pos; } ZSTD_inBuffer;        /* src/zstd/zstd.h:705-709 */
typedef struct { void* dst; size_t size; size_t pos; } ZSTD_outBuffer;             /* src/zstd/zstd.h:711-715 */
typedef enum { ZSTD_e_continue = 0, ZSTD_e_flush = 1, ZSTD_e_end = 2 } ZSTD_EndDirective;   /* src/zstd/zstd.h:775-790 */
size_t ZSTD_compressStream2(ZSTD_CCtx* cctx, ZSTD_outBuffer* output, ZSTD_inBuffer* input, ZSTD_EndDirective endOp); /* zstd.c:28828 */
size_t ZSTD_decompressStream(ZSTD_DCtx* dctx, ZSTD_outBuffer* output, ZSTD_inBuffer* input);                          /* zstd.c:42687 */

/* ---- introspection: src/zstd-info.c:61; src/dictionaries.c:52,54 ---- */
size_t   ZSTD_getFrameHeader(ZSTD_frameHeader* zfhPtr, const void* src, size_t srcSize); /* zstd.c:41160 */
unsigned ZSTD_getDictID_fromFrame(const void* src, size_t srcSize);                 /* zstd.c:42245 */
unsigned ZSTD_getDictID_fromDict(const void* dict, size_t dictSize);                /* zstd.c:42225 */
unsigned ZDICT_getDictID(const void* dict, size_t dictSize);                        /* zstd.c:49974 */

/* ---- dictionary training on the GPU (SURVEY.md 8f rank 4): src/dictionaries.c:161 (ZDICT_trainFromBuffer), :199 (optim = TRUE),
 *      :202-205 (error reporting).  fastCOVER's method with its default parameters (d = 8, f = 20, 4 values of k in [50, 2000],
 *      75/25 split); every candidate is finished with entropy tables and scored by compressing the test samples on the GPU.
 *      The dictionary is a standard Zstandard dictionary (magic, ID, Huffman + FSE tables, repeat offsets, content). ---- */
typedef struct { int compressionLevel; unsigned notificationLevel; unsigned dictID; } ZDICT_params_t;           /* src/zstd/zstd.h (zdict section) */
typedef struct {
    unsigned k, d, steps, nbThreads;
    double splitPoint;
    unsigned shrinkDict, shrinkDictMaxRegression;
    ZDICT_params_t zParams;
} ZDICT_cover_params_t;
size_t ZDICT_trainFromBuffer(void* dictBuffer, size_t dictBufferCapacity, const void* samplesBuffer,
                             const size_t* samplesSizes, unsigned nbSamples);                                  /* zstd.c:50979 */
size_t ZDICT_optimizeTrainFromBuffer_cover(void* dictBuffer, size_t dictBufferCapacity, const void* samplesBuffer,
                                           const size_t* samplesSizes, unsigned nbSamples, ZDICT_cover_params_t* parameters); /* zstd.c:46957 */
unsigned    ZDICT_isError(size_t code);                      /* zstd.c:50101 */
const char* ZDICT_getErrorName(size_t code);                 /* zstd.c:50103 */

/* ---- batch extension (SURVEY.md 8b; needed because src/raw-file.c:150-189 decodes one frame per call and
 *      R's length() is 32-bit).  Arrays live in HOST memory; when ptrs_are_device != 0 the src[i] / dst[i]
 *      pointers themselves are DEVICE pointers (inputs/outputs already resident in HBM).  Each item is
 *      exactly one Zstandard frame.  result[i] receives the produced size or a libzstd error code.
 *      Returns 0, or an error code if the batch as a whole could not run. ---- */
size_t zl_decompress_batch(ZSTD_DCtx* dctx, const void* const* src, const size_t* srcSize,
                           void* const* dst, const size_t* dstCapacity, size_t* result,
                           size_t n, int ptrs_are_device);
size_t zl_compress_batch(ZSTD_CCtx* cctx, const void* const* src, const size_t* srcSize,
                         void* const* dst, const size_t* dstCapacity, size_t* result,
                         size_t n, int ptrs_are_device);
/* one buffer -> concatenated independent frames of `frameSize` content bytes each (a standard multi-frame
 * zstd stream); frameSizes[k] (optional, may be NULL, capacity ceil(srcSize/frameSize)) receives the compressed
 * size of frame k.  Returns total compressed size or an error code. */
size_t zl_compress_split(ZSTD_CCtx* cctx, void* dst, size_t dstCapacity, const void* src, size_t srcSize,
                         size_t frameSize, size_t* frameSizes, int ptrs_are_device);

/* ---- seekable streams (Zstandard's seekable format, zstd's contrib/seekable_format) ----
 * A seekable stream is N >= 1 independent frames followed by a skippable frame holding the seek table:
 *   magic 0x184D2A5E, Frame_Size u32, N entries {Compressed_Size u32, Decompressed_Size u32[, Checksum u32]},
 *   then a 9-byte footer: Number_Of_Frames u32, Seek_Table_Descriptor u8 (bit 7: entries carry a checksum; bits 6-2: 0),
 *   Seekable_Magic_Number u32 = 0x8F92EAB1.  All little-endian; Checksum is the low 32 bits of the XXH64 (seed 0) of the frame's content.
 * Every Zstandard reader, ZSTD_decompressDCtx included, still decodes the whole stream: the table is a skippable frame.  A table is valid
 * when Frame_Size = 8N + 9 (12N + 9 with checksums), the reserved bits are 0, N <= 0x8000000 and the Compressed_Size values plus the
 * table frame add up to the stream's length; anything else is corruption_detected.  A stream that does not end in the seekable magic
 * gives prefix_unknown.
 *
 * zl_compress_seekable: zl_compress_split's frames, byte for byte, then their seek table (with checksums when the context has
 * ZSTD_c_checksumFlag: the frames' own trailers).  frameSize must be 1 .. 0x40000000 (parameter_outOfBound otherwise).  With
 * ptrs_are_device the table is written to device memory after the frames.  Returns the stream's size or an error code.
 * zl_compress_seekable_bound: a dstCapacity that is always enough for zl_compress_seekable (or an error code for a bad frameSize). */
size_t zl_compress_seekable(ZSTD_CCtx* cctx, void* dst, size_t dstCapacity, const void* src, size_t srcSize, size_t frameSize,
                            int ptrs_are_device);
size_t zl_compress_seekable_bound(size_t srcSize, size_t frameSize, int checksum);
/* The seek table of a stream: returns N, or an error code.  When cap >= N, cSizes / dSizes / checksums (each optional, N entries)
 * receive the table's fields; call with cap = 0 to learn N first.  *hasChecksums (optional) says whether the table has checksums.
 * With ptrs_are_device the footer and then the entries are copied from device memory on the current device (no GPU is needed otherwise). */
size_t zl_seekable_frames(const void* src, size_t srcSize, int ptrs_are_device, unsigned* cSizes, unsigned* dSizes,
                          unsigned* checksums, size_t cap, int* hasChecksums);
/* Bytes [offset, offset + length) of a seekable stream's content into dst; a range past the end is clamped, like pread.  Returns the
 * bytes written, min(length, total - offset).  Only the frames the range touches are decoded, in one batch on the context's device, with
 * its dictionary; every frame must produce exactly its table size (corruption_detected otherwise) and, unless ZSTD_d_forceIgnoreChecksum
 * is set, match the table's checksum as well as its own trailer (checksum_wrong).  offset > total: parameter_outOfBound; dstCapacity
 * below the result: dstSize_tooSmall.  ptrs_are_device: src and dst are device memory. */
size_t zl_decompress_range(ZSTD_DCtx* dctx, void* dst, size_t dstCapacity, const void* src, size_t srcSize, size_t offset,
                           size_t length, int ptrs_are_device);
/* Many ranges in one call: item i is bytes [offset[i], offset[i] + length[i]) of the seekable stream (src[i], srcSize[i]) into
 * (dst[i], dstCapacity[i]).  result[i] receives what zl_decompress_range would return for that item alone -- the byte count, or the
 * same error, checked in the same order: the table (prefix_unknown, corruption_detected), parameter_outOfBound, dstSize_tooSmall,
 * dstBuffer_null, then the frames -- and dst[i] the same bytes; a failed item leaves its dst[i] unspecified.  Items with the same
 * (src, srcSize) share one table read, and a frame touched by several items is decoded once; a frame that fails fails every item that
 * touches it (an item touching several failing frames gets the error of the first in stream order), and the other items still get their
 * bytes.  The arrays are host memory; with ptrs_are_device every src[i] and dst[i] is device memory on the context's device.  The
 * destinations must not overlap each other or any source.  The whole call runs on the context's device, with its dictionary and
 * ZSTD_d_forceIgnoreChecksum.  Returns 0 (also for n = 0), or an error for the whole call: null arguments, no device,
 * memory_allocation (the scratch for the frames that are shared or only partly wanted), a failed launch. */
size_t zl_decompress_ranges(ZSTD_DCtx* dctx, const void* const* src, const size_t* srcSize, const size_t* offset, const size_t* length,
                            void* const* dst, const size_t* dstCapacity, size_t* result, size_t n, int ptrs_are_device);

/* ---- streams in device memory (any Zstandard stream: no seek table needed) ----
 * zl_device_frames: every frame of a Zstandard stream in DEVICE memory on the context's device (concatenated frames, skippable frames
 * included), found on the device.  Returns the number of frames N, or an error: the same code ZSTD_decompressDCtx would return for the
 * stream's structure -- prefix_unknown at offset 0; srcSize_wrong for a non-magic at a later frame boundary, a truncated header or
 * block, or 1-4 trailing bytes; corruption_detected for block type 3; frameParameter_unsupported; frameParameter_windowTooLarge.
 * When cap >= N: cOff[k] / cSize[k] receive frame k's offset and compressed size in src, dSize[k] its header's content size:
 * ZSTD_CONTENTSIZE_UNKNOWN when the header has none, 0 for a skippable frame (ZSTD_getFrameContentSize's convention).  Each array is
 * optional.  Call with cap = 0 first to learn N.  srcSize = 0 gives 0. */
size_t zl_device_frames(ZSTD_DCtx* dctx, const void* src, size_t srcSize, unsigned long long* cOff,
                        unsigned long long* cSize, unsigned long long* dSize, size_t cap);
/* ZSTD_decompressDCtx for src and dst in device memory on the context's device: every frame, with the context's dictionary and
 * ZSTD_d_forceIgnoreChecksum.  Returns the bytes written or an error code: the same value, and on success the same bytes, as
 * ZSTD_decompressDCtx on host copies, with the structural errors above and dstSize_tooSmall when the content sizes overflow
 * dstCapacity.  One difference of order: every frame is found before any is decoded, whereas ZSTD_decompressDCtx decodes a frame
 * without a content size as soon as it reaches it -- so for a stream with a decode error at or before such a frame AND a structural
 * error after it, this call reports the structural error.  Frames without a content size are decoded into scratch of
 * min(blocks x blockSizeMax, dstCapacity) bytes each (at most 2 GiB per frame: memory_allocation beyond) and then moved into place,
 * so this call decodes such a frame where ZSTD_decompressDCtx, which offers it all the capacity left, refuses more than 2 GiB.
 * Neither call spreads over several GPUs. */
size_t zl_decompress_device(ZSTD_DCtx* dctx, void* dst, size_t dstCapacity, const void* src, size_t srcSize);

/* Several GPUs from ONE process (frames are independent: SURVEY.md 8e).  Batches of HOST buffers (zl_decompress_batch / zl_compress_batch, and
 * ZSTD_decompressDCtx on a multi-frame stream) are cut into contiguous frame ranges of about equal bytes, one per device, each handled by a helper
 * context on its own host thread; no collective, no peer traffic.  How many GPUs: zl_dctx_set_gpus(n) for a DCtx; num_threads (ZSTD_c_nbWorkers) >= 2 for
 * a CCtx -- the reference's knob for "more hardware" (src/cctx.c:269-277); 0 / unset: the ZSTDLITE_GPUS environment variable ("all" or a number;
 * default 1).  Never more than the visible devices; a context's own device is the one current at its first use. */
size_t zl_dctx_set_gpus(ZSTD_DCtx* dctx, int n);

/* Compression levels: 1, 2, 3 are native (negative "fast" levels run the level-1 engine, 0 means 3).  Levels 4 and 5 run the level-3
 * engine, whose output is within 3 % of libzstd's at those levels (measured per family, 4 KB - 8 MiB, with and without a dictionary).
 * Levels 6..22 -- the lazy / optimal parsers of zstd.c:31546-33746 -- are not implemented: ZSTD_CCtx_setParameter(ZSTD_c_compressionLevel,
 * >= 6) returns parameter_unsupported, unless the context (this call) or the process (ZSTDLITE_GPU_LEVEL_FALLBACK=1) opted into running
 * them on the level-3 engine, which is announced once on stderr.  zl_cctx_engine_level: the engine a context's level runs (1..3). */
size_t zl_cctx_allow_level_fallback(ZSTD_CCtx* cctx, int on);
int zl_cctx_engine_level(const ZSTD_CCtx* cctx);
/* ZSTD_c_windowLog (src/zstd/zstd.h:347): blocks are 128 KiB and searched on their own with offsets up to 64 KiB; frames of more than
 * one block additionally look every position up in per-region tables of earlier occurrences ("far candidates", offsets below 2^24)
 * and declare a window that covers them, at most 2^24.  0 (default) and 24..31: that; 18..23: far offsets stay below 2^windowLog;
 * 17: no far candidates (the fastest setting for one large buffer, about 12 % larger output on text); below 17:
 * parameter_outOfBound, a window smaller than a block cannot be honoured. */

/* CUDA stream (cudaStream_t passed as void*) the context launches on; default: a private non-blocking stream */
size_t zl_dctx_set_stream(ZSTD_DCtx* dctx, void* cuda_stream);
size_t zl_cctx_set_stream(ZSTD_CCtx* cctx, void* cuda_stream);
/* 1: run the next batches as one slice on one stream with per-kernel events (zl_dctx_last_stage_ms); 0 (default): slice
 * pipeline over internal streams, per-kernel times are then reported as -1 */
size_t zl_dctx_set_profile(ZSTD_DCtx* dctx, int on);
/* number of kernel launches issued by the context since creation (bench.py's gpu_launches) */
unsigned long long zl_dctx_launch_count(const ZSTD_DCtx* dctx);
unsigned long long zl_cctx_launch_count(const ZSTD_CCtx* cctx);
/* milliseconds spent on-device by the kernels of the most recent batch call (CUDA events on the context's stream) */
double zl_dctx_last_kernel_ms(const ZSTD_DCtx* dctx);
double zl_cctx_last_kernel_ms(const ZSTD_CCtx* cctx);
/* per-kernel split of the above; decode stages: 0 literals, 1 sequences, 2 execute, 3 checksum; returns -1 for an unknown stage */
double zl_dctx_last_stage_ms(const ZSTD_DCtx* dctx, int stage);
double zl_cctx_last_stage_ms(const ZSTD_CCtx* cctx, int stage);
const char* zl_backend_string(void);

#ifdef __cplusplus
}
#endif
#endif
