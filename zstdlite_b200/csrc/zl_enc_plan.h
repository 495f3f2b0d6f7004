// zl_enc_plan.h -- host-side plan of a compress batch (zl_api_compress.cu): wave and part cuts, slot sizes, descriptors with their far
// tables and frame headers, the placement and staged upload of host buffers, the gather table, and the frames and chunks of
// zl_compress_split.  No CUDA call: tests/host/enc_plan_check.cpp checks it on the CPU.
#pragma once
#include "zl_batch_plan.h"      // ZlRun, zl_build_runs (and zl_host.h, zl_launch.h)

#define ZL_WAVE_BLOCKS 8192u          // blocks per launch wave (bounds the scratch arenas: ~0.9 MB per 128 KiB block)

// blocks of a frame of s bytes (an empty frame has one empty block)
static inline size_t zl_enc_nblocks(size_t s) { return s ? (s + ZL_BLOCKSIZE_MAX - 1) / ZL_BLOCKSIZE_MAX : 1; }

// Development switches of the compress planning (DESIGN.md §3.7), read once from the environment by zl_api_compress.cu:
// ZL_ENC_HLOG=s,l (sets hlog), ZL_ENC_NOFAR, ZL_ENC_SIDE=0|1|2, ZL_ENC_PARTS=n
struct ZlEncTuning { bool hlog = false; u32 hlogS = 0, hlogL = 0; bool noFar = false; int side = 2, parts = ZL_ENC_PARTS; };

// The engine parameters of a call: table sizes from ZL_ENC_HLOG (not with a dictionary, whose tables were built for the level's sizes),
// and the far-offset bound from ZSTD_c_windowLog (17: no far candidates, >= 24: the most M[p] can hold)
static inline void zl_enc_tune_params(ZlEncParams& P, bool dict, int windowLog, const ZlEncTuning& t)
{
    if (t.hlog && !dict) { P.hlogS = t.hlogS; if (P.hlogL) P.hlogL = t.hlogL; }
    if (windowLog) P.farMaxOff = windowLog <= 17 ? 0u : (windowLog >= 24 ? ZL_FAR_MAX_OFF : (1u << windowLog));
}

// Blocks per wave: the scratch of a block scales with the largest block of the batch, so batches of small inputs run in far fewer
// waves (config 4's 1e5 objects: one wave instead of 13, each of which ended in a host sync).  Returns srcSize_wrong for an input of
// >= 0xFFFFFFF0 bytes, else 0.
static inline size_t zl_enc_wave_blocks(const size_t* srcSize, size_t n, size_t* waveBlocks)
{
    size_t maxSrc = 512;
    for (size_t i = 0; i < n; i++) { if (srcSize[i] >= 0xFFFFFFF0ull) return ZL_ERROR(srcSize_wrong); maxSrc = std::max(maxSrc, srcSize[i]); }
    maxSrc = std::min<size_t>(maxSrc, ZL_BLOCKSIZE_MAX);
    *waveBlocks = std::min((size_t)ZL_WAVE_BLOCKS * (ZL_BLOCKSIZE_MAX / ((maxSrc + 255) & ~(size_t)255)), (size_t)1 << 20);
    return 0;
}
// the end of the wave that starts at frame f0: as many frames as fit waveBlocks, and at least one
static inline size_t zl_enc_wave_end(const size_t* srcSize, size_t n, size_t f0, size_t waveBlocks)
{
    size_t f1 = f0;
    for (size_t nb = 0; f1 < n && (f1 == f0 || nb + zl_enc_nblocks(srcSize[f1]) <= waveBlocks); f1++) nb += zl_enc_nblocks(srcSize[f1]);
    return f1;
}

// One wave: frames [f0, f0 + nf) of the call's arrays (device addresses), their block slots in the scratch arenas and their parts.
struct ZlEncWave {
    const u8* const* src; const size_t* srcSize; u8* const* dst; const size_t* dstCap;
    size_t f0 = 0, nf = 0, nb = 0, parts = 1, partCut[ZL_ENC_PARTS + 1];       // part p = frames [partCut[p], partCut[p + 1]) of the wave
    u32 maxBlock = 0, S, slotM, slotRec, slotLit, streamCapWords, streamWordsPerBlock, seqCapWords;
    u32 farMaxOff = 0;                     // far-offset bound of the frames, 0 = no far tables
    size_t nextBlock = 0, farEntries = 0;  // descriptor fill: the first block of the next part, far-table entries handed out so far
};
// Lays out the wave of frames [f0, f1) for engine parameters P.  stats: the dictionary trainer's statistics pass.  Returns memory_allocation
// for more than 0x3FFFFFFF blocks, else 0.
static inline size_t zl_enc_wave_layout(ZlEncWave& w, const u8* const* src, const size_t* srcSize, u8* const* dst, const size_t* dstCap,
                                        size_t f0, size_t f1, bool stats, const ZlEncParams& P, const ZlEncTuning& t)
{
    w = ZlEncWave(); w.src = src; w.srcSize = srcSize; w.dst = dst; w.dstCap = dstCap;
    w.f0 = f0; w.nf = f1 - f0; w.farMaxOff = t.noFar ? 0u : P.farMaxOff;
    for (size_t i = f0; i < f1; i++) { w.nb += zl_enc_nblocks(srcSize[i]); w.maxBlock = std::max(w.maxBlock, (u32)std::min<size_t>(srcSize[i], ZL_BLOCKSIZE_MAX)); }
    if (w.nb > 0x3FFFFFFFull) return ZL_ERROR(memory_allocation);
    w.S = ((w.maxBlock < 512 ? 512 : w.maxBlock) + 255) & ~255u;      // slot layout below needs S >= 264
    w.slotM = w.S; w.slotRec = w.S / 5 + 32; w.slotLit = w.S + 16;    // records: ZL_PARSE_WARPS segments of <= ZL_PARSE_SEG_RECS (zl_enc_match.cuh)
    w.streamCapWords = (((w.S / 4 + 1) * 11) / 8 + 16 + 3) / 4; w.streamWordsPerBlock = 4 * w.streamCapWords; w.seqCapWords = w.S / 4;
    // A wave of very many one-block frames (configs[3]: 1e5 small objects) is described, uploaded and launched in ZL_ENC_PARTS parts: writing
    // 1e5 frame and block descriptors takes the host about a millisecond, a quarter of what the device then needs for them -- this way the
    // device starts after the first part.  The parts use disjoint ranges of every host and device array; stream order keeps them apart.
    if (w.nb == w.nf && w.nf >= 16384 && !stats && t.parts > 1) w.parts = (size_t)std::min(t.parts, ZL_ENC_PARTS);
    for (size_t p = 0; p <= w.parts; p++) w.partCut[p] = w.nf * p / w.parts;
    return 0;
}

struct ZlEncPart { size_t fa, fb, b0, nb; u32 nSmall; bool anyLarge; };
// Descriptors of part `part` (called in part order): frames hf[fa, fb) and blocks hb[b0, b0 + nb), with `frame` and `firstBlock` relative
// to the part; with hp / hs, each frame's source and size for its XXH64.  A frame of several blocks and < 0xFFFFFF00 bytes gets a
// far-candidate table while the wave's tables fit 2^30 entries, first come first served.
static inline ZlEncPart zl_enc_fill_part(ZlEncWave& w, size_t part, u32 dictID, u32 checksumFlag, ZlEncFrame* hf, ZlEncBlock* hb,
                                         const u8** hp, u32* hs)
{
    ZlEncPart q = {w.partCut[part], w.partCut[part + 1], w.nextBlock, 0, 0, false};
    size_t bi = q.b0;
    for (size_t r = q.fa; r < q.fb; r++) {
        const size_t i = w.f0 + r, s = w.srcSize[i], nblk = zl_enc_nblocks(s);
        ZlEncFrame& f = hf[r] = ZlEncFrame();
        f.dst = w.dst[i]; f.dstCap = w.dstCap[i]; f.firstBlock = (u32)(bi - q.b0); f.nblocks = (u32)nblk; f.checksumFlag = checksumFlag;
        bool far = false;
        if (nblk > 1 && s < 0xFFFFFF00ull && w.farMaxOff) {
            const size_t fe = (size_t)zl_far_entries(s);                 // one table per 8 MiB region
            if (w.farEntries + fe <= ((size_t)1 << 30)) { f.pad = (u64)w.farEntries | ((u64)zl_far_log(s) << 56); w.farEntries += fe; far = true; }
        }
        f.hdrSize = zl_write_frame_header(f.hdr, s, dictID, checksumFlag, far ? w.farMaxOff : 0u);
        for (size_t k = 0; k < nblk; k++) {
            ZlEncBlock& b = hb[bi++];
            b.src = w.src[i] + k * ZL_BLOCKSIZE_MAX; b.srcSize = (u32)std::min<size_t>(s - k * ZL_BLOCKSIZE_MAX, ZL_BLOCKSIZE_MAX); b.frame = (u32)(r - q.fa);
            b.flags = (k == 0 ? ZL_BLK_FIRST : 0u) | (k + 1 == nblk ? ZL_BLK_LAST : 0u); b.pad = (u32)(k * ZL_BLOCKSIZE_MAX);
            if (b.srcSize && b.srcSize <= ZL_SMALL_BLOCK) q.nSmall++;
        }
        if (hp) { hp[r] = w.src[i]; hs[r] = (u32)s; q.anyLarge |= s >= ZL_LARGE_FRAME_BYTES; }
    }
    q.nb = bi - q.b0; w.nextBlock = bi;
    return q;
}
// sequence coding of a part on the side stream, next to literal coding (measured +3..4% on 4,096 blocks, +13% on 128)
static inline bool zl_enc_side(const ZlEncTuning& t, size_t partBlocks) { return t.side == 2 || (t.side == 1 && partBlocks <= 1024); }

// A batch of host buffers in the device arenas: the sources as contiguous copy runs (256-aligned in dSrc), the destinations as 16-aligned
// slots of dstCap bytes (dDst)
struct ZlEncPlace { std::vector<ZlRun> runs; std::vector<u32> runOf; size_t srcTotal = 0, dstTotal = 0; };
static inline void zl_enc_place(ZlEncPlace& p, const void* const* src, const size_t* srcSize, const size_t* dstCap, size_t n)
{
    const size_t cut[2] = {0, n};
    size_t runCut[2];
    p = ZlEncPlace(); p.runOf.resize(n);
    zl_build_runs(p.runs, p.runOf.data(), runCut, src, srcSize, cut, 1);
    p.srcTotal = p.runs.back().devOff + p.runs.back().bytes;
    for (size_t i = 0; i < n; i++) p.dstTotal += (dstCap[i] + 15) & ~(size_t)15;
}
// each frame's device source and destination, with the arenas at dSrc / dDst
static inline void zl_enc_place_ptrs(const ZlEncPlace& p, const void* const* src, const size_t* dstCap, size_t n, const u8* dSrc, u8* dDst,
                                     const u8** dsrc, u8** ddst)
{
    for (size_t i = 0, doff = 0; i < n; doff += (dstCap[i] + 15) & ~(size_t)15, i++) {
        const ZlRun& r = p.runs[p.runOf[i]];
        dsrc[i] = dSrc + r.devOff + ((const u8*)src[i] - r.hbase); ddst[i] = dDst + doff;
    }
}
// Scattered inputs (a list of separately allocated objects) are packed by the host into pinned staging and go in with ONE copy; the
// frames are then gathered on the device, copied back with ONE copy and unpacked by the host (a cudaMemcpyAsync per object costs ~2.5 us).
// So are PAGEABLE inputs of a few MiB and more (what the reference's C layer passes to ZSTD_compress2: an R vector, src/raw-file.c:74):
// the host copy pool packs them into staging faster than the driver's own pageable path (one thread, ~8 GB/s).  pageable() is only
// asked for inputs of >= 4 MiB.
template <class Pageable> static inline bool zl_enc_staged(const ZlEncPlace& p, size_t n, Pageable pageable)
{
    return p.runs.size() > 64 || n > 256 || (p.srcTotal >= (4u << 20) && pageable());
}
// The staged upload in pieces of 64 MiB: the host copy pool packs `segs` into the staging buffer hs, then staging [from, to) is copied to
// the device -- while the pool packs the next piece
struct ZlUpload { std::vector<ZlCopySeg> segs; size_t from, to; };
static inline std::vector<ZlUpload> zl_enc_stage_uploads(const ZlEncPlace& p, u8* hs)
{
    const size_t piece = (size_t)64 << 20;
    std::vector<ZlUpload> ups; std::vector<ZlCopySeg> segs;
    size_t sent = 0;
    auto flush = [&](size_t upTo) { if (upTo > sent) { ups.push_back({std::move(segs), sent, upTo}); segs.clear(); sent = upTo; } };
    for (const ZlRun& r : p.runs)
        for (size_t o = 0; o < r.bytes; o += piece) {
            const size_t len = std::min(r.bytes - o, piece);
            segs.push_back({hs + r.devOff + o, r.hbase + o, len});
            if (r.devOff + o + len - sent >= piece) flush(r.devOff + o + len);
        }
    flush(p.srcTotal);
    return ups;
}

// The gather table of n frames in t (3n words): sizes, their exclusive prefix sums (the frames' offsets in the gathered output) and
// the frames' device addresses.  A failed frame counts 0 bytes.  Returns the total.
static inline size_t zl_enc_gather_table(u64* t, const u64* results, u8* const* ddst, size_t n)
{
    size_t total = 0;
    for (size_t i = 0; i < n; total += t[i], i++) { t[i] = zl_is_error((size_t)results[i]) ? 0 : results[i]; t[n + i] = total; reinterpret_cast<const u8**>(t + 2 * n)[i] = ddst[i]; }
    return total;
}

// zl_compress_split: frames [0, cnt) of `bytes` at src, cut every frameSize bytes (the last one short), each with a slot of `slot` bytes at dst
static inline void zl_enc_split_frames(const u8* src, size_t bytes, size_t frameSize, u8* dst, size_t slot, size_t cnt,
                                       const u8** dsrc, size_t* ssz, u8** ddst)
{
    for (size_t i = 0; i < cnt; i++) { dsrc[i] = src + i * frameSize; ssz[i] = std::min(bytes - i * frameSize, frameSize); ddst[i] = dst + i * slot; }
}
// zl_compress_split of srcSize bytes as frames of frameSize: host buffers of >= 2 chunks of at most ZL_WAVE_BLOCKS blocks and 1 GiB, of
// >= 64 MiB each, go through the pipelined path.  Its chunk sizes grow 1/8, 1/4, 1/2, 1, 1, ... of a full chunk: the first staging copy,
// which nothing can overlap, is short (shrinking them again towards the end, for a short last copy back, was measured: the same 143 ms per
// 4 GiB -- small chunks compress less efficiently, which eats what the shorter tail saves).
struct ZlSplitPlan { size_t nf, chunkFrames; bool pipelined; std::vector<size_t> cstart; };    // chunk k = frames [cstart[k], cstart[k + 1])
static inline ZlSplitPlan zl_enc_split_plan(size_t srcSize, size_t frameSize, bool dev)
{
    ZlSplitPlan p;
    p.nf = srcSize ? (srcSize + frameSize - 1) / frameSize : 1;
    p.chunkFrames = std::min<size_t>(ZL_WAVE_BLOCKS / zl_enc_nblocks(frameSize), ((size_t)1 << 30) / frameSize);
    p.pipelined = !dev && p.chunkFrames >= 1 && p.nf >= 2 * p.chunkFrames && p.chunkFrames * frameSize >= ((size_t)64 << 20);
    if (p.pipelined) {
        for (size_t f = 0, sz = std::max<size_t>(p.chunkFrames / 8, 1); f < p.nf; f += sz, sz = std::min(sz * 2, p.chunkFrames)) p.cstart.push_back(f);
        p.cstart.push_back(p.nf);
    }
    return p;
}
