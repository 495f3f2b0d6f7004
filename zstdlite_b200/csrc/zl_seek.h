// zl_seek.h -- the seek table of Zstandard's seekable format (zstd's contrib/seekable_format) and the range plan built on it: which
// frames a byte range of the decompressed stream touches, where each is decoded and what is copied out of the edge frames -- and the plan
// of many ranges in one batch.  No CUDA call: tests/host/seek_check.cpp and tests/host/ranges_check.cpp check it on the CPU.
//
// A seekable stream is N independent Zstandard frames followed by one skippable frame, the seek table:
//   magic 0x184D2A5E | Frame_Size u32 | N entries {Compressed_Size u32, Decompressed_Size u32[, Checksum u32]} |
//   Number_Of_Frames u32 | Seek_Table_Descriptor u8 | Seekable_Magic_Number u32 = 0x8F92EAB1        (all little-endian)
// Checksum is the low 32 bits of the XXH64 (seed 0) of the frame's content; descriptor bit 7 says whether entries carry one, bits 6-2
// are reserved and must be 0.
#pragma once
#include <algorithm>
#include <map>
#include "zl_host.h"              // (and <vector>)

#define ZL_SEEK_TABLE_MAGIC 0x184D2A5Eu
#define ZL_SEEK_MAGIC 0x8F92EAB1u
#define ZL_SEEK_FOOTER 9u
#define ZL_SEEK_MAX_FRAMES 0x8000000u
#define ZL_SEEK_MAX_FRAME_SIZE 0x40000000u      // the reference writer's largest frame content

// bytes of the table frame of n entries, skippable header and footer included
static inline size_t zl_seek_table_size(size_t n, bool checksums) { return 8 + n * (checksums ? 12 : 8) + ZL_SEEK_FOOTER; }

static inline void zl_seek_wr32(u8* p, u32 v) { p[0] = (u8)v; p[1] = (u8)(v >> 8); p[2] = (u8)(v >> 16); p[3] = (u8)(v >> 24); }

// the table frame of n frames into out[0, zl_seek_table_size(n, checksums != nullptr))
static inline void zl_seek_write(u8* out, size_t n, const u32* cSize, const u32* dSize, const u32* checksums)
{
    const size_t entry = checksums ? 12 : 8, total = zl_seek_table_size(n, checksums != nullptr);
    zl_seek_wr32(out, ZL_SEEK_TABLE_MAGIC);
    zl_seek_wr32(out + 4, (u32)(total - 8));
    for (size_t i = 0; i < n; i++) {
        u8* e = out + 8 + i * entry;
        zl_seek_wr32(e, cSize[i]); zl_seek_wr32(e + 4, dSize[i]);
        if (checksums) zl_seek_wr32(e + 8, checksums[i]);
    }
    u8* f = out + total - ZL_SEEK_FOOTER;
    zl_seek_wr32(f, (u32)n); f[4] = checksums ? 0x80 : 0; zl_seek_wr32(f + 5, ZL_SEEK_MAGIC);
}

// The footer: the last min(srcSize, 9) bytes of a stream of srcSize bytes.  Returns the size of the whole table frame (its bytes are the
// stream's last ones), prefix_unknown when the stream does not end in the seekable magic, or corruption_detected.
static inline size_t zl_seek_footer(const u8* tail, size_t srcSize, u32* nOut, bool* checksums)
{
    if (srcSize < ZL_SEEK_FOOTER) {
        if (srcSize >= 4 && zl_rd32(tail + srcSize - 4) == ZL_SEEK_MAGIC) return ZL_ERROR(corruption_detected);
        return ZL_ERROR(prefix_unknown);
    }
    if (zl_rd32(tail + 5) != ZL_SEEK_MAGIC) return ZL_ERROR(prefix_unknown);
    const u32 n = zl_rd32(tail), desc = tail[4];
    if ((desc & 0x7C) || n > ZL_SEEK_MAX_FRAMES) return ZL_ERROR(corruption_detected);
    const size_t size = zl_seek_table_size(n, (desc & 0x80) != 0);
    if (size > srcSize) return ZL_ERROR(corruption_detected);
    *nOut = n; *checksums = (desc & 0x80) != 0;
    return size;
}

struct ZlSeekTable {
    size_t n = 0;
    bool checksums = false;
    std::vector<u32> cSize, dSize, checksum;       // per frame (checksum: only with checksums)
    std::vector<u64> cOff, dOff;                   // prefix sums, n + 1 entries: frame i is [cOff[i], cOff[i + 1]) of the stream
};
// The table frame (`table`, `size` bytes as returned by zl_seek_footer) of a stream of srcSize bytes.  Returns 0 or corruption_detected.
static inline size_t zl_seek_parse(ZlSeekTable& t, const u8* table, size_t size, size_t srcSize)
{
    if (size < zl_seek_table_size(0, false)) return ZL_ERROR(corruption_detected);
    u32 n = 0; bool ck = false;
    const size_t fs = zl_seek_footer(table + size - ZL_SEEK_FOOTER, size, &n, &ck);
    if (zl_is_error(fs)) return fs;
    if (fs != size || zl_rd32(table) != ZL_SEEK_TABLE_MAGIC || zl_rd32(table + 4) != size - 8) return ZL_ERROR(corruption_detected);
    t = ZlSeekTable(); t.n = n; t.checksums = ck;
    t.cSize.resize(n); t.dSize.resize(n); t.cOff.resize(n + 1); t.dOff.resize(n + 1);
    if (ck) t.checksum.resize(n);
    const size_t entry = ck ? 12 : 8;
    t.cOff[0] = t.dOff[0] = 0;
    for (size_t i = 0; i < n; i++) {
        const u8* e = table + 8 + i * entry;
        t.cSize[i] = zl_rd32(e); t.dSize[i] = zl_rd32(e + 4);
        if (ck) t.checksum[i] = zl_rd32(e + 8);
        t.cOff[i + 1] = t.cOff[i] + t.cSize[i]; t.dOff[i + 1] = t.dOff[i] + t.dSize[i];
    }
    if (t.cOff[n] + size != srcSize) return ZL_ERROR(corruption_detected);      // (n <= 2^27 sizes of < 2^32: no overflow)
    return 0;
}

// One of the at most two frames a range starts or ends inside: decoded whole into scratch at scratchOff, then bytes [skip, skip + take)
// of it go to outOff of the caller's buffer.
struct ZlSeekEdge { size_t frame; u64 scratchOff, skip, take, outOff; };
struct ZlSeekPlan {
    u64 bytes = 0;                   // what the call returns: min(length, total - offset)
    size_t first = 0, last = 0;      // frames [first, last) are decoded (none when bytes == 0)
    std::vector<u64> place;          // frame first + j is decoded at place[j]: of the caller's buffer, or of the scratch for an edge frame
    std::vector<u8> edge;            // 1: frame first + j is an edge frame
    ZlSeekEdge edges[2] = {};
    size_t nEdges = 0;
    u64 scratchBytes = 0;
};
// Bytes [offset, offset + length) of the decompressed stream, clamped to its end like pread.  Frames of zero size count as touched only
// between the first and the last frame that hold a byte of the range.  Returns 0, or parameter_outOfBound when offset > total.
static inline size_t zl_seek_plan_range(ZlSeekPlan& p, const ZlSeekTable& t, u64 offset, u64 length)
{
    p = ZlSeekPlan();
    const u64 total = t.dOff[t.n];
    if (offset > total) return ZL_ERROR(parameter_outOfBound);
    p.bytes = std::min(length, total - offset);
    if (!p.bytes) return 0;
    const u64 end = offset + p.bytes;
    // first: dOff[first] <= offset < dOff[first + 1]; last: the first frame that starts at or after the end
    p.first = (size_t)(std::upper_bound(t.dOff.begin(), t.dOff.end(), offset) - t.dOff.begin()) - 1;
    p.last = (size_t)(std::lower_bound(t.dOff.begin(), t.dOff.end(), end) - t.dOff.begin());
    for (size_t f = p.first; f < p.last; f++) {
        const u64 a = std::max(offset, t.dOff[f]), b = std::min(end, t.dOff[f + 1]);
        const bool isEdge = t.dSize[f] && b - a != t.dSize[f];
        if (isEdge) {
            p.edges[p.nEdges++] = {f, p.scratchBytes, a - t.dOff[f], b - a, a - offset};
            p.place.push_back(p.scratchBytes);
            p.scratchBytes += (t.dSize[f] + 15) & ~(u64)15;
        } else p.place.push_back(t.dOff[f] - offset);
        p.edge.push_back(isEdge ? 1 : 0);
    }
    return 0;
}

// ---- many ranges (zl_decompress_ranges) ------------------------------------------------------------------------------------------
// Item i asks for bytes [offset[i], offset[i] + length[i]) of stream streamOf[i].  Every (stream, frame) an item touches is decoded once:
// straight into dst[item] when exactly one item touches it and covers it whole, else whole into scratch, from which each item that
// touches it gets a piece.
#define ZL_RANGE_SCRATCH (~(size_t)0)
struct ZlRangeDecode { size_t stream, frame, item; u64 place; u32 size; };   // item == ZL_RANGE_SCRATCH: place is in the scratch
struct ZlRangePiece { size_t item; u64 from, bytes, outOff; };             // scratch [from, from + bytes) -> dst[item] + outOff
struct ZlRangesPlan {
    std::vector<size_t> result;             // per item: its pre-decode error, or the bytes it returns if all its frames decode
    std::vector<ZlRangeDecode> decodes;     // by stream, then frame
    std::vector<size_t> touchStart, touch;  // item i touches decodes touch[touchStart[i] .. touchStart[i + 1]), in stream order
    std::vector<ZlRangePiece> pieces;       // none of 0 bytes
    u64 scratchBytes = 0;                   // every scratch frame at a 16-byte-aligned place
};

// Groups items by (src, srcSize): streamOf[i] = its stream, numbered in order of first appearance; firstItem[s] = an item of stream s.
static inline size_t zl_ranges_streams(const void* const* src, const size_t* srcSize, size_t n, size_t* streamOf, std::vector<size_t>& firstItem)
{
    std::map<std::pair<const void*, size_t>, size_t> seen;
    firstItem.clear();
    for (size_t i = 0; i < n; i++) {
        auto it = seen.emplace(std::make_pair(src[i], srcSize[i]), firstItem.size());
        if (it.second) firstItem.push_back(i);
        streamOf[i] = it.first->second;
    }
    return firstItem.size();
}

// tables[s] / tableErr[s]: stream s's table, or the error reading it.  Each item is checked as zl_decompress_range checks a range, in the
// same order: table error, parameter_outOfBound, dstSize_tooSmall, (0 bytes: 0), dstBuffer_null.  A rejected item adds no frames.
static inline void zl_ranges_plan(ZlRangesPlan& p, const std::vector<ZlSeekTable>& tables, const std::vector<size_t>& tableErr,
                                  const size_t* streamOf, const size_t* offset, const size_t* length, void* const* dst, const size_t* dstCap,
                                  size_t n)
{
    p = ZlRangesPlan();
    p.result.assign(n, 0);
    const size_t ns = tables.size();
    std::vector<size_t> first(n, 0), last(n, 0);
    std::vector<size_t> lo(ns, ~(size_t)0), hi(ns, 0);                       // per stream: the frames any accepted item touches
    for (size_t i = 0; i < n; i++) {
        const size_t s = streamOf[i];
        if (zl_is_error(tableErr[s])) { p.result[i] = tableErr[s]; continue; }
        ZlSeekPlan sp;
        if (const size_t r = zl_seek_plan_range(sp, tables[s], offset[i], length[i])) { p.result[i] = r; continue; }
        if (sp.bytes > dstCap[i]) { p.result[i] = ZL_ERROR(dstSize_tooSmall); continue; }
        if (!sp.bytes) continue;
        if (!dst[i]) { p.result[i] = ZL_ERROR(dstBuffer_null); continue; }
        p.result[i] = sp.bytes; first[i] = sp.first; last[i] = sp.last;
        lo[s] = std::min(lo[s], sp.first); hi[s] = std::max(hi[s], sp.last);
    }
    // mark[s][f - lo[s]]: 0 untouched, i + 1 touched by item i alone, SHARED by several; then the decode's index
    const size_t SHARED = ~(size_t)0;
    std::vector<std::vector<size_t>> mark(ns);
    for (size_t s = 0; s < ns; s++) if (lo[s] < hi[s]) mark[s].assign(hi[s] - lo[s], 0);
    for (size_t i = 0; i < n; i++) {
        std::vector<size_t>& m = mark[streamOf[i]];
        for (size_t f = first[i]; f < last[i]; f++) { size_t& k = m[f - lo[streamOf[i]]]; k = k ? SHARED : i + 1; }
    }
    for (size_t s = 0; s < ns; s++) {
        const ZlSeekTable& t = tables[s];
        for (size_t f = lo[s]; f < hi[s]; f++) {
            size_t& k = mark[s][f - lo[s]];
            if (!k) continue;
            ZlRangeDecode d{s, f, ZL_RANGE_SCRATCH, 0, t.dSize[f]};
            const size_t i = k - 1;
            if (k != SHARED && t.dOff[f] >= offset[i] && t.dOff[f + 1] <= offset[i] + p.result[i]) { d.item = i; d.place = t.dOff[f] - offset[i]; }
            else { d.place = p.scratchBytes; p.scratchBytes += (t.dSize[f] + 15) & ~(u64)15; }
            k = p.decodes.size();
            p.decodes.push_back(d);
        }
    }
    p.touchStart.assign(n + 1, 0);
    for (size_t i = 0; i < n; i++) {
        p.touchStart[i] = p.touch.size();
        const size_t s = streamOf[i];
        const ZlSeekTable& t = tables[s];
        for (size_t f = first[i]; f < last[i]; f++) {
            const size_t id = mark[s][f - lo[s]];
            p.touch.push_back(id);
            if (p.decodes[id].item != ZL_RANGE_SCRATCH) continue;
            const u64 a = std::max((u64)offset[i], t.dOff[f]), b = std::min((u64)offset[i] + p.result[i], t.dOff[f + 1]);
            if (b > a) p.pieces.push_back({i, p.decodes[id].place + (a - t.dOff[f]), b - a, a - offset[i]});
        }
    }
    p.touchStart[n] = p.touch.size();
}

// The items' results from the engine's per-decode results: an item fails with the first of its frames (in stream order) that failed, or
// with corruption_detected when that frame produced a size other than its table's Decompressed_Size.
static inline void zl_ranges_results(const ZlRangesPlan& p, const size_t* decodeRes, size_t* result, size_t n)
{
    for (size_t i = 0; i < n; i++) {
        result[i] = p.result[i];
        for (size_t j = p.touchStart[i]; j < p.touchStart[i + 1]; j++) {
            const size_t id = p.touch[j], r = decodeRes[id];
            if (zl_is_error(r)) { result[i] = r; break; }
            if (r != p.decodes[id].size) { result[i] = ZL_ERROR(corruption_detected); break; }
        }
    }
}
