// zl_launch.h -- host-visible launcher interface between zl_api.cu and the kernel translation units.
#pragma once
#include <cuda_runtime.h>
#include "zl_common.cuh"

#define ZL_QUADS_PER_WARP 8
#define ZL_EXEC_WARPS 4
#ifndef ZL_EXEC_MIN_CTAS
#define ZL_EXEC_MIN_CTAS 7          // 72 registers: 9 CTAs (56 registers, spills) measured 1.76 ms per 8,192 frames, 8: 1.73, 7: 1.55
#endif
#define ZL_DEC_STAGES 4      // (index +) literals, sequences, execute, checksum
#define ZL_NORM_SLOTS 16384  // resident quads of one sequence-kernel launch the normalized-count scratch has room for
#define ZL_DEC_LANES 8                       // internal streams of the decode slice pipeline
#define ZL_DEC_MAX_SLICES 8                  // one slice per lane: concurrency between streams is what pays, not queueing
#define ZL_DEC_SLICE_BYTES (64ull << 20)     // aim for >= 64 MiB of content ...
#define ZL_DEC_SLICE_MIN_FRAMES 512          // ... and >= 512 frames per slice (host buffers)
#define ZL_DEC_SLICE_DEV_FRAMES 2048         // device buffers: slices of >= 2,048 frames (kernels of different slices run concurrently:
                                             // the execute kernel is issue-bound and uses no shared memory, the entropy kernels are
                                             // latency-bound and limited by shared memory, so they fill each other's idle resources)

// digested dictionary in device memory (zstd.c:42053-42159, ZSTD_DDict): entropy tables in the packed
// cell formats of zl_dec_entropy.cuh plus the raw content that acts as history before the frame.
struct ZlDictDev {
    u16 fseLL[512];
    u16 fseML[512];
    u16 fseOF[256];
    u16 huf[2048];
    u32 hufLog;
    u32 tlog[3];
    u32 rep[3];
    u32 hasEntropy;
    u32 dictID;
    u32 contentSize;
    const u8* content;     // device pointer
};

// ---- large frames (zl_dec_large.cuh) ----
#define ZL_LARGE_FRAME_BYTES (1u << 20)      // frames that may regenerate this much take the block-parallel execute path
#define ZL_PAR_DONE 0xFFFFFF00u
#define ZL_LJUMP_MAX_PASSES 40
struct ZlSymSlot { u32 kind, val; };         // symbolic history slot: kind 0..2 = incoming slot minus val, kind 3 = the constant val
struct ZlLBlock {                            // per block of a large frame (64 B)
    u32 regen;                               // bytes the block regenerates (L2b)
    u32 outOff;                              // frame-relative output offset (L2b)
    u32 err;
    u32 sumL, sumO;                          // sums over its chunks (L2a)
    ZlSymSlot t[3];                          // the block's transform of the repeat-offset history = its chunks' composed (L2a)
    u32 h[3];                                // history before the block (L2b)
    u32 pad[2];
};
// The records of a block are handled in CHUNKS of ZL_LCHUNK_RECS (a warp each in L1 and L3): a 128 KiB block has ~12 of them.
#define ZL_LCHUNK_LOG 10
#define ZL_LCHUNK_RECS (1u << ZL_LCHUNK_LOG)
#define ZL_LCHUNK_MAX ((ZL_BLOCKSIZE_MAX / 3 + ZL_LCHUNK_RECS) >> ZL_LCHUNK_LOG)     // chunks of one block: <= 128 KiB / 3 records + spares
struct ZlLChunk {                            // per chunk (56 B)
    u32 sumL, sumO;                          // literal bytes / output bytes of its records (L1)
    ZlSymSlot t[3];                          // its transform of the repeat-offset history (L1)
    u32 outOff, litOff;                      // frame-relative output offset, block-relative literal offset (L2)
    u32 h[3];                                // history before the chunk (L2)
    u32 pad;
};
// chunks of a block with nrec records (at least one: it carries the block's last literals / the raw or RLE body)
static inline __host__ __device__ u32 zl_lchunks(u32 nrec) { return nrec ? (nrec + ZL_LCHUNK_RECS - 1) >> ZL_LCHUNK_LOG : 1u; }
// index of a block's first chunk inside its frame's share of the chunk arena: blocks are told apart by their record offset
// (a block owns >= nrec + 8 record slots) plus their number
static inline __host__ __device__ u32 zl_lchunk_index(u32 recOff, u32 block) { return (recOff >> ZL_LCHUNK_LOG) + block; }

struct ZlDecodeLaunch {          // one slice of a batch: frames [frameBase, frameBase + nframes)
    const ZlFrameDesc* descs;    // this slice's descriptors / infos / results ...
    ZlFrameInfo* infos;
    u64* results;
    const ZlFrameDesc* descsAll; // ... and the arrays of the whole batch (the block units carry global frame numbers)
    ZlFrameInfo* infosAll;
    u32 frameBase;
    ZlBlockHdr* hdrArena;
    u64* recArena;
    u8* litArena;
    i16* normArena;              // 3 x 64 i16 per resident quad of the sequence kernel: normalized counts while FSE tables are built
    u32 normSlots;               // quads the scratch has room for
    ZlUnit* units;               // this slice's block-unit list (compressed blocks), capacity unitCap
    u32 unitCap;
    u32* counters;               // this slice's {unit count, literal cursor, sequence cursor}
    u32 nframes;
    int verifyChecksum;
    const u32* expect = nullptr; // optional, per frame of the slice: a checksum from a seek table the output must also match (zl_seek.h)
    // large frames of this slice (zl_dec_large.cuh); nLarge == 0: none
    const u32* largeIdx;         // device: indices (relative to the slice) of the large frames
    u32 nLarge, largeMaxBlocks;  // count; largest hdrCap among them (grid bound for the warp-per-block kernels)
    u64 largeMaxBytes;           // largest dstCap among them (grid bound for the pointer-jumping passes)
    ZlLBlock* lbArena;    // per-block scratch, indexed like hdrArena
    ZlLChunk* lcArena;           // per-chunk scratch: frame share starts at (recBase >> ZL_LCHUNK_LOG) + hdrBase
    u32* parentArena;            // one u32 per output byte of the large frames
    u32* remain;                 // device: open bytes after every pass
    u32* remainHost;             // pinned host word for the convergence check
    const ZlDictDev* dict;       // device pointer or null
    cudaEvent_t* stageEv;        // null, or ZL_DEC_STAGES + 1 events recorded around each kernel (per-kernel timing for bench.py)
    // optional: the sequence kernel of the slice runs on `side`, next to the literal kernel (both only depend on the index kernel)
    cudaStream_t side = nullptr; cudaEvent_t sideFork = nullptr, sideJoin = nullptr;
    unsigned long long* launched = nullptr;      // += kernels launched (bench.py's gpu_launches)
};

size_t zl_literals_smem_bytes();
size_t zl_sequences_smem_bytes();
cudaError_t zl_launch_decode(const ZlDecodeLaunch& L, cudaStream_t st);
// descriptors of a slice of small frames from the caller's arrays (raw = [src | dst | srcSize | dstCap], cnt u64 each), zl_dec_kernels.cu
cudaError_t zl_launch_build_descs(const u64* raw, u32 cnt, ZlFrameDesc* descs, u64 lit0, u64 rec0, u64 hdr0, bool worst, cudaStream_t st);
cudaError_t zl_launch_xxh64(const u8* const* ptrs, const u32* sizes, u64* out, u32 n, cudaStream_t st, bool anyLarge = false);
// copy-out of zl_decompress_ranges: one warp per item (device memory, n of them), each at most ZL_SCATTER_BYTES
#define ZL_SCATTER_BYTES (64u << 10)
struct ZlScatterItem { const u8* src; u8* dst; u32 bytes; };
cudaError_t zl_launch_range_scatter(const ZlScatterItem* items, u32 n, cudaStream_t st);
// frame index of a stream in device memory (zl_dec_index.cuh, zl_stream_index.h)
struct ZlStreamFrame { u64 cOff, cSize, dSize; u32 nblocks, bsm; };      // bsm: blockSizeMax, ZL_FRAME_SKIP for a skippable frame
#define ZL_FRAME_SKIP 0xFFFFFFFFu
struct ZlIdxStatus { u64 first; u32 tail, link, err, pad; };            // first candidate's offset; the chain's last candidate
// I1: cand null: per-tile counts and their prefix sums (tileOff, tiles + 1 entries); else the candidates' offsets into cand
cudaError_t zl_launch_idx_candidates(const u8* src, u64 srcSize, u32 tiles, u32* tileCount, u64* tileOff, u64* cand, cudaStream_t st);
cudaError_t zl_launch_idx_extent(const u8* src, u64 srcSize, const u64* cand, u32 n, u32 cap, u32* link, u32* errc, u32* nblk, u32* mark, cudaStream_t st);
cudaError_t zl_launch_idx_jump(u32 n, u32* j0, u32* j1, u32* mark, u32* open, u32 pass0, u32 passes, cudaStream_t st);
cudaError_t zl_launch_idx_frontier(const u8* src, u64 srcSize, const u64* cand, u32 n, u32* link, u32* errc, u32* nblk, u32* mark,
                                   const ZlIdxStatus* status, bool serial, cudaStream_t st);
// I4: frames null: per-tile counts of marked candidates, their prefix sums and *status; else the frame records
cudaError_t zl_launch_idx_frames(const u8* src, u64 srcSize, const u64* cand, u32 n, const u32* link, const u32* errc, const u32* nblk,
                                 const u32* mark, u32 tiles, u32* tileCount, u64* tileOff, ZlIdxStatus* status, ZlStreamFrame* frames, cudaStream_t st);

// ---- compression --------------------------------------------------------------------------------------------------
#include "zl_enc_entropy.cuh"
#include "zl_enc_match.cuh"

#ifndef ZL_MATCH_WARPS
#define ZL_MATCH_WARPS 15     // named barriers 1..15 carry the table token (0 is __syncthreads); more than 15 warps share them (zl_k_match)
#endif
#define ZL_PARSE_WARPS (ZL_BLOCKSIZE_MAX / ZL_PARSE_SEG)     // one warp per segment of a block
#define ZL_ASM_WARPS 4
#define ZL_ENT_WARPS 4       // warps (= blocks) per CTA in the two entropy kernels
#define ZL_ENC_STAGES 5      // match, parse, literals, sequences, plan+assemble
#define ZL_ENC_PARTS 4       // a wave of very many one-block frames is described and launched in this many parts (zl_enc_wave)
#define ZL_BLK_FIRST 1u
#define ZL_BLK_LAST 2u

struct ZlEncBlock {          // one per block of <= 128 KiB (24 B)
    const u8* src;           // device pointer
    u32 srcSize;
    u32 frame;               // index into the frame array
    u32 flags;               // ZL_BLK_FIRST / ZL_BLK_LAST within its frame
    u32 pad;                 // offset of the block inside its frame (far candidates)
};
struct ZlEncFrame {          // one per frame (64 B)
    u8* dst;                 // device pointer to the frame's output
    u64 dstCap;
    u32 firstBlock, nblocks;
    u32 hdrSize, checksumFlag;
    u8 hdr[24];              // frame header bytes, prepared on the host (zl_write_frame_header)
    u64 pad;                 // far-candidate table: offset in the far arena (u32 units, low 56 bits) | log2 entries << 56; 0 = none
};
struct ZlEncBlockMeta { u32 nseq, nlit; };
struct ZlEncBlockPlan { u64 dstOff; u32 type, size; };     // offset inside the frame's output, block type, payload size

struct ZlEncodeLaunch {
    const ZlEncBlock* blocks; u32 nblocks;
    const ZlEncFrame* frames; u32 nframes;
    ZlEncParams params;
    u32* M; u32 slotM;                 // words per block slot (>= max block size); reused for streams + sequence bits
    u64* recs; u32 slotRec;
    u8* lit; u32 slotLit;
    u32* hist;
    ZlEncBlockMeta* metas;
    ZlEncBlockOut* outs;
    ZlEncBlockPlan* plans;
    u32 streamCapWords, streamWordsPerBlock, seqCapWords;
    u64* results;
    const u64* xxh;                    // per-frame XXH64 of the content (only read when the frame carries a checksum)
    const ZlEncDictDev* dict;          // device pointer to the digested dictionary, or null
    cudaEvent_t* stageEv;              // null or ZL_ENC_STAGES + 1 events
    cudaStream_t side = nullptr; cudaEvent_t sideFork = nullptr, sideJoin = nullptr;   // optional: sequence coding next to literal coding
    u32 maxBlock = ZL_BLOCKSIZE_MAX;   // largest block of the wave (the parse kernel walks blocks of more than one segment with a CTA each)
    u32* stats = nullptr;              // dictionary training: sum literal / code statistics here after the parse and stop (zl_dict_train.cuh)
    u32 nSmall = 0;                    // blocks of at most ZL_SMALL_BLOCK bytes (> 0, non-empty) in the wave: zl_k_match_small takes those
    u32* far = nullptr;                // far-candidate tables of the wave's multi-block frames (zl_enc_match.cuh), preset to 0xFF; null: none
};
cudaError_t zl_enc_upload_const();
size_t zl_enc_match_smem(const ZlEncParams& P);
cudaError_t zl_launch_encode(const ZlEncodeLaunch& L, cudaStream_t st);
cudaError_t zl_launch_results_out(const u64* src, u64* hostDst, u32 n, cudaStream_t st);      // hostDst: pinned host memory (device-mapped under UVA)
cudaError_t zl_launch_gather(const u8* const* srcs, const u64* sizes, const u64* offs, u8* dst, u32 n, cudaStream_t st);
