// zl_stream_index.h -- the frame index of a Zstandard stream in device memory (zl_device_frames, zl_decompress_device) and the decode
// plan built on it.  No CUDA call: the per-thread bodies of the index kernels (zl_dec_index.cuh) are ZL_HD functions here, and
// tests/host/stream_index_check.cpp runs them in host loops against the serial walk.
//
// Frames are byte-aligned and carry no index, and following the chain from offset 0 costs one dependent load per block on one thread.
// The index is built speculatively instead:
//   I1 scan     every offset whose 4 bytes read as a frame or skippable magic is a candidate; compacted in stream order
//   I2 extent   a thread per candidate walks its frame with at most ZL_IDX_W block steps: its end is a candidate (link = that index),
//               the stream's end (END), an error (BAD: its own; STRAY: it ends where no frame starts), or the cap was reached (LONG)
//   I3 mark     pointer jumping over the links marks every candidate reachable from candidate 0 -- only reachability separates the real
//               chain from a run of valid frames stored inside a raw block, which may end exactly on a true frame start
//   frontier    the chain may end in a LONG candidate: one thread finishes that walk without a cap, marking resumes from its end; after
//               ZL_IDX_R such rounds one thread walks the rest of the chain serially
//   I4 compact  the marked candidates in order are the frames; the chain's last one says END or the error
// Work: I2 at most W block steps per candidate; at most R + 2 rounds of at most ceil(log2 n) + 1 marking passes over n candidates (R
// rounds that end in a frontier walk, one that ends in the serial walk, one final); and the frontier walks' block steps, bounded by
// the stream's own blocks -- never quadratic in look-alikes.
#pragma once
#include <algorithm>
#include "zl_host.h"              // (and <vector>)

#define ZL_IDX_W 1024u                   // block steps of one I2 walk
#define ZL_IDX_R 8u                      // single-candidate frontier rounds before the serial walk
#define ZL_IDX_TILE_THREADS 256u
#define ZL_IDX_TILE_CHUNKS 16u           // I1: 16-byte chunks per thread of a tile (a tile is 64 KiB of the stream)
#define ZL_IDX_TILE_NODES 4096u          // I4: candidates per tile
#define ZL_IDX_MAX_PASSES 40u            // marking passes of one round: ceil(log2 2^32) + 1 is enough

// link values above the candidate indices
#define ZL_LINK_END 0xFFFFFFFFu          // the frame ends exactly at the end of the stream
#define ZL_LINK_BAD 0xFFFFFFFEu          // the frame itself is malformed: errc holds the code
#define ZL_LINK_STRAY 0xFFFFFFFDu        // the frame is well formed but ends where no frame starts: srcSize_wrong
#define ZL_LINK_LONG 0xFFFFFFFCu         // the walk reached its step cap
#define ZL_LINK_NODES 0xFFFFFFF0u        // links below this are candidate indices (so are candidate counts)

ZL_HD bool zl_idx_magic(u32 w) { return w == ZL_MAGIC || (w & 0xFFFFFFF0u) == ZL_MAGIC_SKIP; }

// The frame header (zstd.c:41050-41152) at ip with srcSize bytes left: 0, an error code, or the bytes a complete header needs.
ZL_HD size_t zl_frame_head(ZlHostFrameHeader* h, const u8* ip, u64 srcSize)
{
    *h = ZlHostFrameHeader{};
    if (srcSize < 5) {                               // zstd.c:41061-41077: a too-short prefix must still look like a magic number
        if (srcSize > 0) {
            const u8 m[4] = {0x28, 0xB5, 0x2F, 0xFD};
            const u8 sk[4] = {0x50, 0x2A, 0x4D, 0x18};
            bool a = true, b = true;
            for (u32 i = 0; i < srcSize && i < 4; i++) { if (ip[i] != m[i]) a = false; if (i > 0 && ip[i] != sk[i]) b = false; if (i == 0 && (ip[i] & 0xF0) != 0x50) b = false; }
            if (!a && !b) return ZL_ERROR(prefix_unknown);
        }
        return 5;
    }
    const u32 magic = zl_rd32(ip);
    if ((magic & 0xFFFFFFF0u) == ZL_MAGIC_SKIP) {
        if (srcSize < 8) return 8;
        h->skippable = 1; h->contentSize = zl_rd32(ip + 4); h->headerSize = 8;
        return 0;
    }
    if (magic != ZL_MAGIC) return ZL_ERROR(prefix_unknown);
    const u32 fhd = ip[4], didCode = fhd & 3, single = (fhd >> 5) & 1, fcsID = fhd >> 6;
    const u32 didSz = didCode == 3 ? 4 : didCode, fcsSz = fcsID == 0 ? (single ? 1u : 0u) : (1u << fcsID);
    const u32 hs = 5 + (single ? 0 : 1) + didSz + fcsSz;
    if (srcSize < hs) return hs;
    h->headerSize = hs;
    if (fhd & 8) return ZL_ERROR(frameParameter_unsupported);
    u32 p = 5; u64 window = 0;
    if (!single) {
        const u32 wl = ip[p++], wlog = (wl >> 3) + 10;
        if (wlog > 31) return ZL_ERROR(frameParameter_windowTooLarge);
        window = 1ull << wlog; window += (window >> 3) * (wl & 7);
    }
    u32 did = 0;
    if (didSz == 1) did = ip[p]; else if (didSz == 2) did = zl_rd16(ip + p); else if (didSz == 4) did = zl_rd32(ip + p);
    p += didSz;
    u64 fcs = ~0ull;                                 // ZSTD_CONTENTSIZE_UNKNOWN
    if (fcsID == 0) { if (single) fcs = ip[p]; } else if (fcsID == 1) fcs = zl_rd16(ip + p) + 256; else if (fcsID == 2) fcs = zl_rd32(ip + p); else fcs = zl_rd64(ip + p);
    if (single) window = fcs;
    h->contentSize = fcs; h->windowSize = window;
    h->blockSizeMax = (unsigned)(window < ZL_BLOCKSIZE_MAX ? window : ZL_BLOCKSIZE_MAX);
    h->dictID = did; h->checksumFlag = (fhd >> 2) & 1;
    return 0;
}

// The one frame-extent rule of the host walk (zl_host_find_frame_size) and the device index: the frame or skippable frame at ip with
// `left` bytes to the end of the stream.  state 0: it ends at `end`; 1: `err` (the host walk's code); 2: `cap` block steps (> 0) were
// taken and the frame goes on (cap 0: no cap).
struct ZlExtent { u64 end; size_t err; u32 nblocks, state; };
ZL_HD ZlExtent zl_frame_extent(const u8* ip, u64 left, u32 cap)
{
    ZlExtent x = {0, 0, 0, 1};
    if (left >= 8 && (zl_rd32(ip) & 0xFFFFFFF0u) == ZL_MAGIC_SKIP) {                // zstd.c:41188
        const u64 sz = (u64)zl_rd32(ip + 4) + 8;
        if (sz > left) { x.err = ZL_ERROR(srcSize_wrong); return x; }
        x.end = sz; x.state = 0;
        return x;
    }
    ZlHostFrameHeader h;
    const size_t r = zl_frame_head(&h, ip, left);
    if (r > (size_t)0 - (size_t)ZL_E_maxCode) { x.err = r; return x; }                   // (zl_is_error is host code)
    if (r > 0) { x.err = ZL_ERROR(srcSize_wrong); return x; }
    u64 pos = h.headerSize; u32 nb = 0;
    for (;;) {                                                                       // zstd.c:41370-41384
        if (cap && nb == cap) { x.end = pos; x.nblocks = nb; x.state = 2; return x; }
        if (left - pos < 3) { x.err = ZL_ERROR(srcSize_wrong); return x; }
        const u32 bh = zl_rd24(ip + pos), last = bh & 1, type = (bh >> 1) & 3;
        u32 cs = bh >> 3;
        if (type == 3) { x.err = ZL_ERROR(corruption_detected); return x; }
        if (type == 1) cs = 1;
        if (3 + (u64)cs > left - pos) { x.err = ZL_ERROR(srcSize_wrong); return x; }
        pos += 3 + cs; nb++;
        if (last) break;
    }
    if (h.checksumFlag) { if (left - pos < 4) { x.err = ZL_ERROR(srcSize_wrong); return x; } pos += 4; }
    x.end = pos; x.nblocks = nb; x.state = 0;
    return x;
}

// ---- the per-thread bodies of the index kernels ---------------------------------------------------------------------------------
// I1: candidates among the 16 offsets of a 16-byte chunk; w[0..3] are the chunk's bytes as little-endian words, w[4..7] the next
// chunk's (any value where it lies past the stream's last 16-byte chunk).  Offsets q with lo <= q <= hi are inside the stream with
// 4 bytes to read.  Bit q of the result: offset q is a candidate.
ZL_HD u32 zl_idx_chunk_mask(const u32 w[8], int lo, int hi)
{
    u32 m = 0;
#pragma unroll
    for (int q = 0; q < 16; q++) {
        const u32 a = w[q >> 2], b = w[(q >> 2) + 1], s = (u32)(q & 3) * 8;
        const u32 v = s ? (a >> s) | (b << (32 - s)) : a;
        if (q >= lo && q <= hi && zl_idx_magic(v)) m |= 1u << q;
    }
    return m;
}

// I2 (and the frontier, cap 0): the extent of candidate i at offset cand[i] of a stream of srcSize bytes; the n candidates are sorted.
ZL_HD u32 zl_idx_find(const u64* cand, u32 n, u64 pos)
{
    u32 a = 0, b = n;
    while (a < b) { const u32 m = a + (b - a) / 2; if (cand[m] < pos) a = m + 1; else b = m; }
    return a < n && cand[a] == pos ? a : ZL_LINK_NODES;
}
ZL_HD void zl_idx_extent(const u8* src, u64 srcSize, const u64* cand, u32 n, u32 i, u32 cap, u32* link, u32* errc, u32* nblk)
{
    const u64 p = cand[i];
    const ZlExtent x = zl_frame_extent(src + p, srcSize - p, cap);
    nblk[i] = x.nblocks; errc[i] = 0;
    if (x.state == 2) { link[i] = ZL_LINK_LONG; return; }
    if (x.state == 1) { link[i] = ZL_LINK_BAD; errc[i] = (u32)((size_t)0 - x.err); return; }
    const u64 end = p + x.end;
    if (end == srcSize) { link[i] = ZL_LINK_END; return; }
    const u32 j = zl_idx_find(cand, n, end);
    if (j == ZL_LINK_NODES) { link[i] = ZL_LINK_STRAY; errc[i] = ZL_E_srcSize_wrong; return; }
    link[i] = j;
}

// I3: one pointer-jumping pass for candidate v.  jin[v] is its 2^r-th successor (or a link value: it has fewer); marks every node that
// a marked node reaches in 2^r steps, and writes the 2^(r+1)-th successor to jout[v].  Returns 1 when v is marked and jin[v] is a node
// (the chain from a marked node is not yet covered); a round is done after a pass in which no node returned 1.
ZL_HD u32 zl_idx_jump(u32 v, const u32* jin, u32* jout, u32* mark)
{
    const u32 j = jin[v];
    if (j >= ZL_LINK_NODES) { jout[v] = j; return 0; }
    jout[v] = jin[j];
    if (!mark[v]) return 0;
    mark[j] = 1;
    return 1;
}

// I4: a marked candidate is a frame unless it is the chain's last one and malformed itself
ZL_HD bool zl_idx_is_frame(const u32* mark, const u32* link, u32 v) { return mark[v] && link[v] != ZL_LINK_BAD; }
// the record of a frame (a marked candidate v, ZlStreamFrame in zl_launch.h).  A skippable frame reports content size 0
// (ZSTD_getFrameContentSize's convention) and bsm ZL_FRAME_SKIP; the chain's last frame has cSize 0 when it ends where no frame starts.
ZL_HD ZlStreamFrame zl_idx_record(const u8* src, u64 srcSize, const u64* cand, const u32* link, const u32* nblk, u32 v)
{
    const u64 p = cand[v];
    ZlHostFrameHeader h;
    zl_frame_head(&h, src + p, srcSize - p);
    ZlStreamFrame f;
    f.cOff = p; f.nblocks = nblk[v];
    f.cSize = link[v] == ZL_LINK_END ? srcSize - p : (link[v] < ZL_LINK_NODES ? cand[link[v]] - p : 0);
    f.dSize = h.skippable ? 0 : h.contentSize;
    f.bsm = h.skippable ? ZL_FRAME_SKIP : h.blockSizeMax;
    return f;
}
// The status of the chain from offset 0 for a stream of srcSize >= 5 bytes: 0 (it ends exactly at the end), or the code
// ZSTD_decompressDCtx gives for the stream's structure at the chain's end.  first: the first candidate's offset (none: n == 0).
static inline size_t zl_idx_tail_error(u64 n, u64 first, u32 link, u32 err)
{
    if (!n || first != 0) return ZL_ERROR(prefix_unknown);
    if (link == ZL_LINK_END) return 0;
    return (size_t)0 - (size_t)err;
}

// The serial walk the index must reproduce: zl_host_find_frame_size frame after frame from offset 0 with ZSTD_decompressDCtx's rules
// (zstd.c:41681-41766).  frames receives every complete frame (the last one included when only what follows it is wrong); returns the
// status as zl_idx_tail_error does, and 0 for srcSize 0.
static inline size_t zl_stream_walk(const u8* src, u64 srcSize, std::vector<ZlStreamFrame>& frames)
{
    frames.clear();
    u64 pos = 0;
    while (srcSize - pos >= 5) {
        const ZlExtent x = zl_frame_extent(src + pos, srcSize - pos, 0);
        if (x.state) {
            if (pos && x.err == ZL_ERROR(prefix_unknown)) return ZL_ERROR(srcSize_wrong);      // zstd.c:41724-41729
            return x.err;
        }
        ZlHostFrameHeader h;
        zl_frame_head(&h, src + pos, srcSize - pos);
        frames.push_back({pos, x.end, h.skippable ? 0 : h.contentSize, x.nblocks, h.skippable ? ZL_FRAME_SKIP : h.blockSizeMax});
        pos += x.end;
    }
    return pos == srcSize ? 0 : ZL_ERROR(srcSize_wrong);
}

// ---- the decode plan of zl_decompress_device ------------------------------------------------------------------------------------
// Frames with a content size decode straight into dst at the prefix sum of the sizes before them.  Frames without one decode first into
// scratch (min(nblocks * blockSizeMax, dstCapacity) each, at 16-byte-aligned places); their results fix every place, and each is then
// moved into dst by zl_k_range_scatter in pieces of at most ZL_SCATTER_BYTES.  The checks follow ZSTD_decompressDCtx frame by frame:
// a frame whose content does not fit in what is left of dstCapacity is dstSize_tooSmall, and nothing after it is decoded.
struct ZlDevDecode { u32 frame; u64 place, cap; };      // place: in dst, or in scratch for a frame without content size
struct ZlDevPiece { u64 from, to, bytes; };             // scratch -> dst
struct ZlDevPlan {
    std::vector<ZlDevDecode> unknown, known;            // in stream order
    u64 scratchBytes = 0;
    u32 stop = ~0u;                                     // the first frame that is not decoded (~0u: none); stopErr its error
    size_t stopErr = 0;
    std::vector<ZlDevPiece> pieces;
    u64 total = 0;
};
// Step 1, before any decode: the status of the index, then dstSize_tooSmall when the frames with a content size alone overflow
// dstCapacity at some frame (which ZSTD_decompressDCtx reports at that frame, whatever the frames without one produce); then the
// scratch of the frames without content size.  Returns 0 or the error of the whole call.
static inline size_t zl_dev_plan_unknown(ZlDevPlan& p, const std::vector<ZlStreamFrame>& f, size_t status, u64 dstCap)
{
    p = ZlDevPlan();
    u64 known = 0;
    for (size_t k = 0; k < f.size(); k++) {
        if (f[k].bsm == ZL_FRAME_SKIP || f[k].dSize == ~0ull) continue;
        if (f[k].dSize > dstCap - known) return ZL_ERROR(dstSize_tooSmall);
        known += f[k].dSize;
    }
    if (zl_is_error(status)) return status;
    for (size_t k = 0; k < f.size(); k++) {
        if (f[k].bsm == ZL_FRAME_SKIP || f[k].dSize != ~0ull) continue;
        const u64 cap = std::min<u64>((u64)f[k].nblocks * f[k].bsm, dstCap);
        p.unknown.push_back({(u32)k, p.scratchBytes, cap});
        p.scratchBytes += (cap + 15) & ~15ull;
    }
    return 0;
}
// Step 2, with the results of the frames without content size (unknownRes[j] for p.unknown[j]): every frame's place, where decoding
// stops and why, the frames with content size to decode into dst and the pieces to move.
static inline void zl_dev_plan_places(ZlDevPlan& p, const std::vector<ZlStreamFrame>& f, const size_t* unknownRes, u64 dstCap)
{
    u64 op = 0; size_t j = 0;
    p.known.clear(); p.pieces.clear(); p.stop = ~0u; p.stopErr = 0;
    for (size_t k = 0; k < f.size(); k++) {
        if (f[k].bsm == ZL_FRAME_SKIP) continue;
        u64 size = f[k].dSize;
        if (size == ~0ull) {
            const ZlDevDecode& u = p.unknown[j];
            const size_t r = unknownRes[j++];
            if (zl_is_error(r)) { p.stop = (u32)k; p.stopErr = r; break; }
            size = r;
            if (size > dstCap - op) { p.stop = (u32)k; p.stopErr = ZL_ERROR(dstSize_tooSmall); break; }
            for (u64 o = 0; o < size; o += ZL_SCATTER_BYTES) p.pieces.push_back({u.place + o, op + o, std::min<u64>(size - o, ZL_SCATTER_BYTES)});
        } else {
            if (size > dstCap - op) { p.stop = (u32)k; p.stopErr = ZL_ERROR(dstSize_tooSmall); break; }
            p.known.push_back({(u32)k, op, size});
        }
        op += size;
    }
    p.total = op;
}
// The call's result: the first frame in stream order that failed -- a decode with content size whose result is an error or not its
// content size (corruption_detected), or the frame decoding stopped at -- else the total.
static inline size_t zl_dev_plan_result(const ZlDevPlan& p, const size_t* knownRes)
{
    for (size_t i = 0; i < p.known.size(); i++) {
        if (zl_is_error(knownRes[i])) return knownRes[i];
        if (knownRes[i] != p.known[i].cap) return ZL_ERROR(corruption_detected);
    }
    return p.stop != ~0u ? p.stopErr : (size_t)p.total;
}
