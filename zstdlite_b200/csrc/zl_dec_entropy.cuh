// zl_dec_entropy.cuh -- entropy stage of the B200 Zstandard decoder: kernels K1a (literals) and K1b (sequences).
//
// Work unit for both kernels: one FRAME per QUAD (4 lanes), 8 frames per warp.
//   K1a  lane 0 walks frame/block/literal headers and reads the Huffman tree description; lanes 0..3 fill
//        the decode table cooperatively and decode the 4 Huffman streams, one stream per lane
//        (HUF_decompress4X, zstd.c:38653).  Shared memory per frame: the 2^11 x u16 table (~5 KB).
//   K1b  lane 0 parses the sequences header, lanes 0..2 build the LL / OF / ML FSE decode tables
//        concurrently (zstd.c:43497), lane 0 runs the serial 3-state FSE decode (zstd.c:44241) and
//        writes one u64 record per sequence.  Shared memory per frame: three packed u32 tables (~5.6 KB).
// Splitting the two keeps the per-frame shared-memory footprint small, which is what bounds the number
// of frames in flight per SM (the decode loops are dependent-latency chains; see DESIGN.md).
// Output goes to scratch arenas in HBM (literals, records, one ZlBlockHdr per block) consumed by K2.
//
// Reference behaviour restated here (file:line in /root/reference/src/zstd/zstd.c):
//   frame header 41050-41152, block header 43075, literals section 43146-43347,
//   HUF_readStats 3470, FSE_readNCount 3269, HUF_readDTableX1 38436, sequence headers 43707,
//   ZSTD_buildFSETable 43497, ZSTD_decodeSequence 44241, end-of-stream checks 44686 / 38647.
#pragma once
#include "zl_common.cuh"

// ---- packed FSE decode cell of the tiny Huffman-weight table (u32): nbBits[0:8) newStateBase[16:26) symbol[26:32)
ZL_HD u32 zl_fse_pack(u32 base, u32 nb, u32 add, u32 sym) { return nb | (add << 8) | (base << 16) | (sym << 26); }
#define ZL_FSE_NB(e) ((e) & 0xFFu)
#define ZL_FSE_BASE(e) (((e) >> 16) & 1023u)
#define ZL_FSE_SYM(e) ((e) >> 26)
// ---- packed LL / OF / ML decode cell (u16): symbol[0:6) ns[6:16), where ns in [1, 2*size) is the value
// ZSTD_buildFSETable (zstd.c:43605-43613) calls `nextState`: nbBits = log - highbit(ns), newStateBase = (ns << nbBits)
// - size.  16-bit cells halve the shared-memory footprint of a frame, which is what bounds the frames in flight per SM;
// the number of additional bits is a function of the symbol (OF: the symbol itself; LL / ML: ZlConstTables).
ZL_HD u16 zl_seq_cell(u32 ns, u32 sym) { return (u16)(sym | (ns << 6)); }
#define ZL_CELL_SYM(e) ((e) & 63u)
#define ZL_CELL_NS(e) ((e) >> 6)

// ---- backward bit reader (restates BIT_DStream_t, zstd.c:2352-2550) ---------------------------------------
// `wbase` is the frame's src pointer rounded down to 4 bytes, `bias` = src - wbase (0..3); stream positions
// are byte offsets relative to src.  (hi:lo) is a 64-bit window, next bit to consume = MSB of hi; `n` valid
// bits.  Refills are whole aligned 32-bit words.  Latency hiding: the word for the NEXT refill is already in
// a register (`nextw`, loaded one refill earlier), and its load hits L1 because the 32-byte sector two sectors
// further down the stream is requested with a prefetch each time the reader enters a new sector.
struct ZlBitR {
    u32 hi, lo;
    i32 n;
    u32 nextw;
    i32 wi;      // index of the word after `nextw` (next one to load)
    i32 wlow;    // word holding the first byte of the stream
};
ZL_HD u32 zl_ld_word(const u32* p)
{
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}
ZL_HD void zl_prefetch(const u32* p)
{
#if defined(__CUDA_ARCH__)
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
#else
    (void)p;
#endif
}
// Loads word `wi` (clamped to the stream: below the start the value is irrelevant, over-reading is detected by
// zl_br_remaining) without touching the loaded value, so the load stays in flight until the next refill.
ZL_HD u32 zl_br_fetch(ZlBitR& b, const u32* wbase)
{
    const i32 i = b.wi < b.wlow ? b.wlow : b.wi;
    if ((b.wi & 7) == 7) { const i32 pf = b.wi - 16; zl_prefetch(wbase + (pf < b.wlow ? b.wlow : pf)); }
    b.wi--;
    return zl_ld_word(wbase + i);
}
ZL_HD bool zl_br_init(ZlBitR& b, const u32* wbase, u32 bias, u32 beg, u32 end)
{
    if (end <= beg) return false;
    const u32 a = end - 1 + bias;
    const u32 W = zl_ld_word(wbase + (a >> 2));
    const u32 bsel = a & 3;
    const u32 L = (W >> (8 * bsel)) & 0xFF;
    if (!L) return false;                              // zstd.c:2369 end mark missing
    const u32 hb = zl_highbit(L);
    b.hi = zl_shl(W, 8 * (3 - bsel) + (8 - hb));       // drop bytes above the stream, the padding and the end mark
    b.lo = 0;
    b.n = (i32)(8 * bsel + hb);
    b.wi = (i32)(a >> 2) - 1;
    b.wlow = (i32)((beg + bias) >> 2);
    {   const i32 p1 = b.wi - 8, p2 = b.wi - 16;
        zl_prefetch(wbase + (p1 < b.wlow ? b.wlow : p1)); zl_prefetch(wbase + (p2 < b.wlow ? b.wlow : p2)); }
    b.nextw = zl_br_fetch(b, wbase);
    return true;
}
ZL_HD void zl_br_refill(ZlBitR& b, const u32* wbase)       // afterwards n >= 33
{
    if (b.n <= 32) {
        const u32 w = b.nextw;
        b.nextw = zl_br_fetch(b, wbase);
        b.hi |= zl_shr(w, (u32)b.n);
        b.lo = zl_shl(w, 32u - (u32)b.n);
        b.n += 32;
    }
}
ZL_HD u32 zl_br_peek(const ZlBitR& b, u32 k) { return zl_shr(b.hi, 32u - k); }       // k <= 32; 0 when k == 0
ZL_HD void zl_br_skip(ZlBitR& b, u32 k)                                               // k <= 32
{
    b.hi = zl_fsl(b.lo, b.hi, k);
    b.lo = zl_shl(b.lo, k);
    b.n -= (i32)k;
}
ZL_HD u32 zl_br_take(ZlBitR& b, u32 k) { const u32 v = zl_br_peek(b, k); zl_br_skip(b, k); return v; }
// bits of the stream not consumed yet; negative when the reader ran past the start
ZL_HD i32 zl_br_remaining(const ZlBitR& b, u32 bias, u32 beg)
{
    return b.n + 8 * (4 * (b.wi + 2) - (i32)(beg + bias));     // `nextw` (word wi+1) is loaded but not in (hi:lo) yet
}

// ---- FSE normalized-count header (forward, LSB first): zstd.c:3269-3409 ------------------------------------
// Returns bytes consumed, or 0 on error.
ZL_HD u32 zl_read_ncount(const u8* src, u32 srcSize, i16* norm, u32* maxSymIO, u32* tableLog)
{
    if (srcSize < 1) return 0;
    u32 maxSV1 = *maxSymIO + 1, sym = 0;
    u32 bitpos = 4;
    for (u32 i = 0; i < maxSV1; i++) norm[i] = 0;
    i32 nbBits = (i32)(src[0] & 15) + 5;
    if (nbBits > 15) return 0;
    *tableLog = (u32)nbBits;
    i32 remaining = (1 << nbBits) + 1, threshold = 1 << nbBits;
    nbBits++;
    bool prev0 = false;
    for (;;) {
        if (prev0) {
            for (;;) {
                u32 by = bitpos >> 3;
                u32 w = (by < srcSize ? src[by] : 0u) | ((by + 1 < srcSize ? (u32)src[by + 1] : 0u) << 8);
                w = (w >> (bitpos & 7)) & 3;
                bitpos += 2;
                sym += w;
                if (w != 3) break;
                if (sym >= maxSV1) break;
            }
            if (sym >= maxSV1) break;
        }
        {
            u32 by = bitpos >> 3;
            u32 v = 0;
            for (u32 i = 0; i < 4; i++) v |= (by + i < srcSize ? (u32)src[by + i] : 0u) << (8 * i);
            v >>= (bitpos & 7);                     // >= 25 valid bits, fields are <= 16 bits
            i32 max = (2 * threshold - 1) - remaining, count;
            if ((i32)(v & (u32)(threshold - 1)) < max) {
                count = (i32)(v & (u32)(threshold - 1));
                bitpos += (u32)nbBits - 1;
            } else {
                count = (i32)(v & (u32)(2 * threshold - 1));
                if (count >= threshold) count -= max;
                bitpos += (u32)nbBits;
            }
            count--;
            if (count >= 0) remaining -= count; else remaining += count;
            norm[sym++] = (i16)count;
            prev0 = (count == 0);
            if (remaining < threshold) {
                if (remaining <= 1) break;
                nbBits = (i32)zl_highbit((u32)remaining) + 1;
                threshold = 1 << (nbBits - 1);
            }
            if (sym >= maxSV1) break;
        }
    }
    if (remaining != 1) return 0;
    if (sym > maxSV1) return 0;
    *maxSymIO = sym - 1;
    u32 used = (bitpos + 7) >> 3;
    if (used > srcSize) return 0;
    return used;
}

// ---- FSE decode table build (one lane per table): zstd.c:43497-43613 ------------------------------------------
// `tbl` first receives symbols, then cells.
ZL_HD bool zl_fse_build(u16* tbl, const i16* norm, u32 maxSym, u32 log)
{
    u32 size = 1u << log, high = size - 1, mask = size - 1, step = (size >> 1) + (size >> 3) + 3;
    u16 next[64];
    for (u32 s = 0; s <= maxSym; s++) {
        if (norm[s] == -1) { tbl[high--] = (u16)s; next[s] = 1; }
        else next[s] = (u16)norm[s];
    }
    u32 pos = 0;
    for (u32 s = 0; s <= maxSym; s++) {
        i32 n = norm[s];
        for (i32 i = 0; i < n; i++) {
            tbl[pos] = (u16)s;
            pos = (pos + step) & mask;
            while (pos > high) pos = (pos + step) & mask;
        }
    }
    if (pos != 0) return false;
    for (u32 u = 0; u < size; u++) {
        u32 s = tbl[u];
        tbl[u] = zl_seq_cell(next[s]++, s);
    }
    return true;
}

// =================================================================================================== K0: frame / block index
// One thread per frame (zl_k_index): frame header (zstd.c:41050-41152), then every block header (43075) and -- for
// compressed blocks -- the literals section header (43146-43347) and the first bytes of the sequences section (nbSeq and
// the modes byte, 43707-43745).  That is enough to give every block its own slice of the literal and record arenas and
// to name, for every entropy table a block uses, the block that carries its description, so that K1a / K1b can decode
// all blocks of all frames independently of each other (a large frame no longer is one long serial chain).
// Compressed blocks are appended to a global unit list (one atomic per block); raw / RLE blocks need no entropy work.
// records reserved per block beyond nbSeq: a block regenerates <= 128 KiB, so a valid one splits at most two lengths (>= 65536);
// the generic step checks the exact capacity, the fast loop stops 4 short of it
#define ZL_REC_SLACK 8u
ZL_HD u32 zl_unit_append(u32* unitCount)
{
#if defined(__CUDA_ARCH__)
    return atomicAdd(unitCount, 1u);
#else
    return (*unitCount)++;
#endif
}
ZL_HD void zl_index_frame(const ZlFrameDesc& d, ZlFrameInfo& info, ZlBlockHdr* hdrs, u32 frameIdx, u32 dictID, u32 dictHasEntropy,
                          ZlUnit* units, u32* unitCount, u32 unitCap)
{
    u32 err = 0;
    info.err = 0; info.nblocks = 0; info.contentSize = ~0ull; info.totalOut = 0;
    info.checksumFlag = 0; info.checksum = 0; info.dictID = 0; info.blockSizeMax = ZL_BLOCKSIZE_MAX; info.pad = 0;
    const u8* ip = d.src;
    const u32 srcSize = d.srcSize;
    u32 pos = 0, blockSizeMax = ZL_BLOCKSIZE_MAX, nblocks = 0;
    do {
        if (srcSize < 5) { err = ZL_E_srcSize_wrong; break; }
        if (zl_rd32(ip) != ZL_MAGIC) { err = ZL_E_prefix_unknown; break; }
        const u32 fhd = ip[4];
        const u32 didCode = fhd & 3, single = (fhd >> 5) & 1, fcsID = fhd >> 6;
        const u32 didSz = didCode == 3 ? 4 : didCode, fcsSz = fcsID == 0 ? (single ? 1u : 0u) : (1u << fcsID);
        const u32 hs = 5 + (single ? 0 : 1) + didSz + fcsSz;
        if (srcSize < hs) { err = ZL_E_srcSize_wrong; break; }
        if (fhd & 8) { err = ZL_E_frameParameter_unsupported; break; }
        u32 p = 5;
        u64 window = 0;
        if (!single) {
            const u32 wl = ip[p++];
            const u32 wlog = (wl >> 3) + 10;
            if (wlog > 31) { err = ZL_E_frameParameter_windowTooLarge; break; }
            window = 1ull << wlog;
            window += (window >> 3) * (wl & 7);
        }
        u32 did = 0;
        if (didSz == 1) did = ip[p]; else if (didSz == 2) did = zl_rd16(ip + p); else if (didSz == 4) did = zl_rd32(ip + p);
        p += didSz;
        u64 fcs = ~0ull;
        if (fcsID == 0) { if (single) fcs = ip[p]; }
        else if (fcsID == 1) fcs = zl_rd16(ip + p) + 256;
        else if (fcsID == 2) fcs = zl_rd32(ip + p);
        else fcs = zl_rd64(ip + p);
        if (single) window = fcs;
        if (did != 0 && did != dictID) { err = ZL_E_dictionary_wrong; break; }      // zstd.c:41318
        blockSizeMax = window < ZL_BLOCKSIZE_MAX ? (u32)window : ZL_BLOCKSIZE_MAX;
        pos = hs;
        info.contentSize = fcs; info.checksumFlag = (fhd >> 2) & 1; info.dictID = did; info.blockSizeMax = blockSizeMax;
    } while (0);
    // ---- block walk
    u32 litUsed = 0, recUsed = 0;
    u32 outKnown = 0; bool outValid = d.large == 0;          // output position of the next block while it only depends on headers
    u64 seqTotal = 0;
    u32 hufDef = ZL_DEF_NONE, seqDef[3] = {ZL_DEF_NONE, ZL_DEF_NONE, ZL_DEF_NONE};
    bool hufValid = dictHasEntropy != 0, seqValid = dictHasEntropy != 0, lastSeen = false;
    const u8* src = d.src;
    while (!err && !lastSeen) {
        if (pos + 3 > srcSize) { err = ZL_E_srcSize_wrong; break; }
        const u32 bh = zl_rd24(src + pos);
        const u32 last = bh & 1, type = (bh >> 1) & 3, csize = bh >> 3;
        pos += 3;
        if (nblocks >= d.hdrCap) { err = ZL_E_INTERNAL_hdrCap; break; }
        ZlBlockHdr h;
        h.flags = last ? 4u : 0u; h.regenSize = 0; h.srcOff = 0; h.litOff = 0; h.litSize = 0; h.nrec = 0; h.recOff = 0;
        h.seqOff = 0; h.seqEnd = 0; h.litSecOff = 0; h.hufDef = ZL_DEF_NONE; h.seqDef[0] = h.seqDef[1] = h.seqDef[2] = ZL_DEF_NONE;
        h.nbSeq = 0; h.outOff = 0;
        if (type == 3) err = ZL_E_corruption_detected;
        else if (type == 1) {                                                    // RLE block, zstd.c:41510
            if (pos + 1 > srcSize) err = ZL_E_srcSize_wrong;
            else { h.flags |= 1u | ((u32)src[pos] << 8); h.regenSize = csize; pos += 1; if ((u64)outKnown + csize <= d.dstCap) outKnown += csize; else outValid = false; }
        } else if (type == 0) {                                                  // raw block, zstd.c:41497
            if (csize > srcSize - pos) err = ZL_E_srcSize_wrong;
            else { h.regenSize = csize; h.srcOff = pos; pos += csize; if ((u64)outKnown + csize <= d.dstCap) outKnown += csize; else outValid = false; }
        } else {
            if (csize > srcSize - pos) err = ZL_E_srcSize_wrong;
            else if (csize > blockSizeMax) err = ZL_E_srcSize_wrong;             // zstd.c:45099
            else if (csize < 2) err = ZL_E_corruption_detected;                  // MIN_CBLOCK_SIZE, zstd.c:43150
            else {
                const u32 blockEnd = pos + csize;
                const u8* bp = src + pos;
                const u32 ltype = bp[0] & 3, fmt = (bp[0] >> 2) & 3;
                u32 lhSize = 0, litSize = 0, litCSize = 0, litMode = 0, seqOff = 0;
                h.litSecOff = pos;
                if (ltype >= 2) {
                    u32 single = 0;
                    if (ltype == 3 && !hufValid) err = ZL_E_dictionary_corrupted;      // zstd.c:43160
                    else if (csize < 5) err = ZL_E_corruption_detected;
                    else {
                        const u32 lhc = zl_rd32(bp);
                        if (fmt < 2) { single = !fmt; lhSize = 3; litSize = (lhc >> 4) & 0x3FF; litCSize = (lhc >> 14) & 0x3FF; }
                        else if (fmt == 2) { lhSize = 4; litSize = (lhc >> 4) & 0x3FFF; litCSize = lhc >> 18; }
                        else { lhSize = 5; litSize = (lhc >> 4) & 0x3FFFF; litCSize = (lhc >> 22) + ((u32)bp[4] << 10); }
                        if (litSize > blockSizeMax) err = ZL_E_corruption_detected;
                        else if (!single && litSize < 6) err = ZL_E_literals_headerWrong;
                        else if (litCSize + lhSize > csize) err = ZL_E_corruption_detected;
                        else if (litSize == 0 || litCSize == 0) err = ZL_E_corruption_detected;
                        else if (litUsed + litSize > d.litCap) err = ZL_E_dstSize_tooSmall;   // more literals than dst can hold
                        else {
                            litMode = 2; h.litOff = litUsed; litUsed += litSize;
                            if (ltype == 2) hufDef = nblocks;
                            h.hufDef = hufDef; hufValid = true;
                            seqOff = pos + lhSize + litCSize;
                        }
                    }
                } else {
                    bool ok = true;
                    if (fmt == 0 || fmt == 2) { lhSize = 1; litSize = bp[0] >> 3; }
                    else if (fmt == 1) { lhSize = 2; litSize = zl_rd16(bp) >> 4; }
                    else { lhSize = 3; if (csize < 3) { ok = false; litSize = 0; } else litSize = zl_rd24(bp) >> 4; }
                    if (!ok) err = ZL_E_corruption_detected;
                    else if (litSize > blockSizeMax) err = ZL_E_corruption_detected;
                    else if (ltype == 0) {
                        if (lhSize + litSize > csize) err = ZL_E_corruption_detected;
                        else { litMode = 0; h.srcOff = pos + lhSize; seqOff = pos + lhSize + litSize; }
                    } else {
                        if (lhSize + 1 > csize) err = ZL_E_corruption_detected;
                        else { litMode = 1; h.flags |= (u32)bp[lhSize] << 8; seqOff = pos + lhSize + 1; }
                    }
                }
                if (!err) {       // sequences section: nbSeq and the modes byte (zstd.c:43720-43745)
                    u32 q = seqOff, nbSeq = 0;
                    if (q >= blockEnd) err = ZL_E_srcSize_wrong;
                    else {
                        nbSeq = src[q++];
                        if (nbSeq > 0x7F) {
                            if (nbSeq == 0xFF) { if (q + 2 > blockEnd) err = ZL_E_srcSize_wrong; else { nbSeq = zl_rd16(src + q) + 0x7F00; q += 2; } }
                            else { if (q >= blockEnd) err = ZL_E_srcSize_wrong; else nbSeq = ((nbSeq - 0x80) << 8) + src[q++]; }
                        }
                    }
                    if (!err && !nbSeq && q != blockEnd) err = ZL_E_corruption_detected;      // zstd.c:43736: nothing may follow nbSeq == 0
                    if (!err && nbSeq) {
                        if (q + 1 > blockEnd) err = ZL_E_srcSize_wrong;
                        else {
                            const u32 modes = src[q];
                            if (modes & 3) err = ZL_E_corruption_detected;
                            for (u32 t = 0; t < 3 && !err; t++) {
                                const u32 mode = (modes >> (6 - 2 * t)) & 3;
                                if (mode != 3) seqDef[t] = nblocks;
                                else if (seqDef[t] == ZL_DEF_NONE && !seqValid) err = ZL_E_corruption_detected;   // zstd.c:43682
                                h.seqDef[t] = seqDef[t];
                            }
                        }
                        if (!err) {
                            seqTotal += nbSeq;
                            if (seqTotal > (u64)d.dstCap / 3 + 8) err = ZL_E_corruption_detected;          // more sequences than dst could hold
                            else if ((u64)recUsed + nbSeq + ZL_REC_SLACK + 1u > d.recCap) err = ZL_E_INTERNAL_hdrCap;   // many blocks: retry with the worst-case arena
                        }
                    }
                    if (!err) { h.nbSeq = nbSeq; h.recOff = recUsed; if (nbSeq) recUsed += (nbSeq + ZL_REC_SLACK + 1u) & ~1u; }   // even: the execute kernel loads record pairs
                }
                h.flags |= 2u | (litMode << 4);
                h.litSize = litSize; h.seqOff = seqOff; h.seqEnd = blockEnd;
                if (!err) {
                    if (h.nbSeq) outValid = false;
                    else if (outValid && litMode == 2 && (u64)outKnown + litSize <= d.dstCap) { h.flags |= ZL_BLK_DIRECT; h.outOff = outKnown; outKnown += litSize; }
                    else outValid = false;
                }
                pos = blockEnd;
            }
        }
        if (err) break;
        hdrs[nblocks] = h;
        if ((h.flags & 3) == 2 && (((h.flags >> 4) & 3) == 2 || h.nbSeq)) {      // entropy work to do
            const u32 u = zl_unit_append(unitCount);
            if (u < unitCap) { units[u].frame = frameIdx; units[u].block = nblocks; } else err = ZL_E_INTERNAL_hdrCap;
        }
        nblocks++;
        lastSeen = last != 0;
    }
    if (!err) {
        if (info.checksumFlag) {
            if (pos + 4 > srcSize) err = ZL_E_checksum_wrong;                                              // zstd.c:41651
            else { info.checksum = zl_rd32(src + pos); pos += 4; }
        }
        if (!err && pos != srcSize) err = ZL_E_srcSize_wrong;       // one frame per batch item
    }
    info.err = err; info.nblocks = nblocks;
}

// =================================================================================================== K1a: literals
// Work unit: one compressed block whose literals are Huffman-coded (quad per unit, 8 units per warp).
struct ZlLitCtl {
    u32 err;
    u32 hufLog, nsym;
    u32 needHufFill, nStreams, sStrict;
    u32 sBeg[4], sEnd[4], sOut[4], sLen[4], sErr[4];
};
struct ZlLitSm {
    u16 huf[2048];
    u8 weights[256];
    union {
        u16 symStart[256];
        u32 wtbl[64];
    } u;
    ZlLitCtl ctl;
};

// Huffman tree description (lane 0): zstd.c:3470-3540, weights via FSE 3875/3790.
// Fills f.weights / f.u.symStart, ctl.hufLog, ctl.nsym.  Returns bytes consumed or 0 on error.
ZL_HD u32 zl_huf_read_stats(ZlLitSm& f, const u8* src, u32 srcSize, const u32* wbase, u32 bias, u32 srcOff)
{
    if (!srcSize) return 0;
    u32 hdr = src[0], nsym = 0, iSize;
    u8* w = f.weights;
    if (hdr >= 128) {
        nsym = hdr - 127;
        iSize = (nsym + 1) / 2;
        if (iSize + 1 > srcSize) return 0;
        for (u32 n = 0; n < nsym; n++) { u32 b = src[1 + n / 2]; w[n] = (u8)((n & 1) ? (b & 15) : (b >> 4)); }
    } else {
        iSize = hdr;
        if (iSize + 1 > srcSize) return 0;
        i16 norm[16];
        u32 maxSym = 12, tlog;                 // weights are <= HUF_TABLELOG_MAX (12); FSE_MAX_SYMBOL_VALUE is 255 in
        // the reference but any symbol > 12 is rejected at zstd.c:3509, so a 13-symbol alphabet is equivalent.
        u32 nc = zl_read_ncount(src + 1, iSize, norm, &maxSym, &tlog);
        if (!nc || tlog > 6) return 0;
        u32* t = f.u.wtbl;
        {   // tiny FSE table (zstd.c:3692-3790)
            u32 size = 1u << tlog, high = size - 1, mask = size - 1, step = (size >> 1) + (size >> 3) + 3, pos = 0;
            u16 next[16];
            for (u32 s = 0; s <= maxSym; s++) { if (norm[s] == -1) { t[high--] = s; next[s] = 1; } else next[s] = (u16)norm[s]; }
            for (u32 s = 0; s <= maxSym; s++) for (i32 i = 0; i < norm[s]; i++) {
                t[pos] = s; pos = (pos + step) & mask; while (pos > high) pos = (pos + step) & mask; }
            if (pos != 0) return 0;
            for (u32 u = 0; u < size; u++) { u32 s = t[u]; u32 ns = next[s]++; u32 nb = tlog - zl_highbit(ns);
                t[u] = zl_fse_pack((ns << nb) - size, nb, 0, s); }
        }
        ZlBitR b;
        u32 beg = srcOff + 1 + nc, end = srcOff + 1 + iSize;
        if (!zl_br_init(b, wbase, bias, beg, end)) return 0;
        zl_br_refill(b, wbase);
        u32 s1 = zl_br_take(b, tlog), s2 = zl_br_take(b, tlog);
        for (;;) {                                   // alternate the two states until the stream overflows
            if (nsym > 253) return 0;
            zl_br_refill(b, wbase);
            u32 e = t[s1]; w[nsym++] = (u8)ZL_FSE_SYM(e); s1 = ZL_FSE_BASE(e) + zl_br_take(b, ZL_FSE_NB(e));
            if (zl_br_remaining(b, bias, beg) < 0) { w[nsym++] = (u8)ZL_FSE_SYM(t[s2]); break; }
            if (nsym > 253) return 0;
            e = t[s2]; w[nsym++] = (u8)ZL_FSE_SYM(e); s2 = ZL_FSE_BASE(e) + zl_br_take(b, ZL_FSE_NB(e));
            if (zl_br_remaining(b, bias, beg) < 0) { w[nsym++] = (u8)ZL_FSE_SYM(t[s1]); break; }
        }
    }
    u32 rank[13], total = 0;
    for (u32 i = 0; i < 13; i++) rank[i] = 0;
    for (u32 n = 0; n < nsym; n++) { if (w[n] > 12) return 0; rank[w[n]]++; total += (1u << w[n]) >> 1; }
    if (!total) return 0;
    u32 tableLog = zl_highbit(total) + 1;
    if (tableLog > 11) return 0;       // format limit (RFC 8878 4.2.1); libzstd tolerates 12, see DESIGN.md
    u32 rest = (1u << tableLog) - total, last = zl_highbit(rest) + 1;
    if ((1u << zl_highbit(rest)) != rest) return 0;
    w[nsym++] = (u8)last; rank[last]++;
    if (rank[1] < 2 || (rank[1] & 1)) return 0;
    u32 start[13], acc = 0;
    for (u32 wv = 1; wv <= tableLog; wv++) { start[wv] = acc; acc += rank[wv] << (wv - 1); }
    for (u32 n = 0; n < nsym; n++) { u32 wv = w[n]; if (wv) { f.u.symStart[n] = (u16)start[wv]; start[wv] += 1u << (wv - 1); } }
    f.ctl.hufLog = tableLog; f.ctl.nsym = nsym;
    return iSize + 1;
}

// cooperative table fill, lane q of 4: zstd.c:38506-38568 (cell = nbBits<<8 | symbol)
ZL_HD void zl_huf_fill(ZlLitSm& f, u32 q)
{
    u32 tlog = f.ctl.hufLog, nsym = f.ctl.nsym;
    for (u32 n = q; n < nsym; n += 4) {
        u32 wv = f.weights[n];
        if (!wv) continue;
        u32 len = 1u << (wv - 1), st = f.u.symStart[n];
        u16 cell = (u16)(((tlog + 1 - wv) << 8) | n);
        for (u32 k = 0; k < len; k++) f.huf[st + k] = cell;
    }
}

#define ZL_NO_RING 0xFFFFFFFFu       // `ring` argument of the decoders: no stream ring (the CPU emulation)
#if defined(__CUDACC__)
// ---- device-only fast paths: branch-free refills (predicated PTX loads write straight into the look-ahead register,
// so the load stays in flight until the next refill), shared-space table loads, rotated loops. ------------------------
__device__ __forceinline__ u32 zl_smem_addr(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ u32 zl_lds32(u32 a) { u32 v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ u32 zl_lds16(u32 a) { u32 v; asm("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
// if (n <= 32) { window |= nextw << (32 - n); nextw = *next word*; n += 32; }   -- no branch, no select on the window:
// bits of (hi:lo) below the n valid ones are always zero and the clamped shifts make both ORs no-ops when n > 32.
// The look-ahead load and the L1 prefetch of the sector two sectors further down are predicated PTX, so the
// compiler cannot turn them into divergent branches.
#ifndef ZL_PF_DIST
#define ZL_PF_DIST 16         // words between the lane's position and its L1 prefetch
#endif
#define ZL_REFILL_DEV()                                                                                        \
    {                                                                                                          \
        const u32 need_ = (n <= 32) ? 1u : 0u;                                                                 \
        hi |= zl_shr(nextw, (u32)n);                                                                           \
        lo |= zl_shl(nextw, 32u - (u32)n);                                                                     \
        const i32 i_ = wi < wlow ? wlow : wi;                                                                  \
        const i32 pf_ = (wi - ZL_PF_DIST) < wlow ? wlow : (wi - ZL_PF_DIST);                                   \
        const u32 pfneed_ = need_ & (((u32)wi & 7u) == 7u ? 1u : 0u);                                          \
        asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %3, 0;\n\tsetp.ne.u32 q, %4, 0;\n\t"              \
                     "@p ld.global.nc.u32 %0, [%1];\n\t@q prefetch.global.L1 [%2];\n\t}"                          \
                     : "+r"(nextw) : "l"(wbase + i_), "l"(wbase + pf_), "r"(need_), "r"(pfneed_));             \
        n += (i32)(need_ << 5);                                                                                \
        wi -= (i32)need_;                                                                                      \
    }
// ---- stream ring: the 64-bit reader of the fast loops ------------------------------------------------------------------------
// A lane's ring is NS 16-byte slots, contiguous in shared memory at `ring` (aligned to 16 NS): chunk c of the stream (the 16 bytes at
// wb16 + 16 c, `wb16` = the frame's src rounded down to 16 bytes) lives in slot c & (NS-1), so stream word w is at
// ring | (4 w & (16 NS - 4)).  The reader keeps one number, `pos`: the stream bits below the next unread one, counted from wb16.
// A reload takes the three words that hold the 64 bits below pos and funnel-shifts them into (hi:lo), the next bit to consume being
// the MSB of hi: after every reload all 64 bits are valid, whatever pos is (the byte-granular container of BIT_reloadDStream keeps
// >= 57).  Chunks are copied by cp.async: when pos enters chunk X, chunk X-(NS-1) is fetched into the slot chunk X+1 has left, never
// below `clow`, the chunk that holds the stream's first byte (bits read below the start reach only a stream that runs past its
// start, which the exact count in pos rejects).  A reload moves pos by less than 128 bits, so it issues at most one copy.
#define ZL_LIT_RING_NS 8          // literal lanes: 128 bytes each, 4 KB per warp
#define ZL_SEQ_RING_NS 4          // sequence units: 64 bytes each, 1 KB per warp
__device__ __forceinline__ u32 zl_ring_lds(u32 a) { u32 v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
// chunks c0 .. c0-(NS-1) below the unread bit, c0 = (pos - 1) >> 7; slots under the start get chunk clow (never read for a valid stream)
template <int NS>
__device__ __forceinline__ void zl_ring_start(u32 ring, const u32* wb16, i32 pos, i32 clow)
{
    const i32 c0 = (pos - 1) >> 7;
#pragma unroll
    for (i32 k = 0; k < NS; k++) {
        const i32 c = (c0 - k) < clow ? clow : (c0 - k);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(ring | (((u32)(c0 - k) & (u32)(NS - 1)) << 4)), "l"(wb16 + 4 * c) : "memory");
    }
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}
// Reload (hi:lo) at `pos`; `prev` = pos at the previous reload, `gb` = wb16 - 16 (NS-1), `cmin` = clow + NS-1.  SYNC = the
// commit / wait text placed between the copy and the word loads.
#define ZL_RING_RELOAD(NS, SYNC, ring, gb, cmin, pos, prev, hi, lo)                                                    \
    {                                                                                                                  \
        const i32 x_ = (pos) >> 7;                                                                                     \
        const u32 t_ = (u32)(pos) >> 3;                                                                                \
        const u32 need_ = ((u32)((pos) ^ (prev)) > 127u && x_ >= (cmin)) ? 1u : 0u;                                  \
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p cp.async.cg.shared.global [%0], [%1], 16;\n\t" SYNC "}" \
                     ::"r"(((t_ + 16u) & (16u * ((NS) - 1))) | (ring)), "l"((gb) + (i64)x_ * 16), "r"(need_) : "memory"); \
        const u32 w0_ = zl_ring_lds((t_ & (16u * (NS) - 4u)) | (ring));                                               \
        const u32 w1_ = zl_ring_lds(((t_ - 4u) & (16u * (NS) - 4u)) | (ring));                                        \
        const u32 w2_ = zl_ring_lds(((t_ - 8u) & (16u * (NS) - 4u)) | (ring));                                        \
        hi = __funnelshift_r(w1_, w0_, (u32)(pos));                                                                    \
        lo = __funnelshift_r(w2_, w1_, (u32)(pos));                                                                    \
    }
// hand-off to the generic reader: n = 32 + (pos & 31) bits in (hi:lo), the word below them in `nextw`
template <int NS>
__device__ __forceinline__ void zl_ring_to_br(ZlBitR& b, u32 ring, i32 pos, i32 s16)
{
    asm volatile("cp.async.wait_all;" ::: "memory");
    const u32 t = (u32)pos >> 3, r = (u32)pos & 31u;
    const u32 w0 = zl_ring_lds((t & (16u * NS - 4u)) | ring), w1 = zl_ring_lds(((t - 4u) & (16u * NS - 4u)) | ring),
              w2 = zl_ring_lds(((t - 8u) & (16u * NS - 4u)) | ring);
    b.hi = __funnelshift_r(w1, w0, r);
    b.lo = zl_shl(w1, 32u - r);
    b.n = 32 + (i32)r;
    b.nextw = w2;
    b.wi = (pos >> 5) - 3 - s16;
}
__device__ __forceinline__ u32 zl_selp(u32 a, u32 b, bool c)          // c ? a : b, guaranteed to stay a select
{
    u32 r;
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %3, 0;\n\tselp.u32 %0, %1, %2, p;\n\t}" : "=r"(r) : "r"(a), "r"(b), "r"((u32)c));
    return r;
}
__device__ __forceinline__ u32 zl_opaque(u32 x) { asm volatile("" : "+r"(x)); return x; }   // stops rematerialisation in loops
#endif

// one Huffman stream per lane: zstd.c:38626-38650.  Returns 0 when the stream ends exactly, 2 when bits are left over,
// 1 when the reader ran past the start (or the end mark is missing).
// `ring` (device only; ZL_NO_RING = none): shared-space address of this lane's ring (ZL_LIT_RING_NS slots).  With a ring the
// stream reaches the lane through cp.async and LDS instead of a global load per word: the per-warp scoreboard made every refill
// wait for the global load some other lane had issued one refill earlier (ncu: long scoreboard 6.5 of 10 cycles per issue).
// The ring loop decodes 20 symbols per iteration, five per reload (5 x 11 bits <= 64), and stores them as five aligned words.
ZL_HD u32 zl_huf_stream(const u16* huf, u32 tlog, const u32* wbase, u32 bias, u32 beg, u32 end, u8* out, u32 n, u32 ring = ZL_NO_RING)
{
    ZlBitR b;
    if (!zl_br_init(b, wbase, bias, beg, end)) return 1;
    const u32 sh = 32 - tlog;
    u32 i = 0;
#define ZL_HUF_SYM(dst) { const u32 e = huf[b.hi >> sh]; zl_br_skip(b, e >> 8); dst = e & 0xFF; }
    while (i < n && (((size_t)(out + i)) & 3)) { u32 s; zl_br_refill(b, wbase); ZL_HUF_SYM(s); out[i++] = (u8)s; }
#if defined(__CUDA_ARCH__)
    if (ring != ZL_NO_RING) {
        if (i + 20 <= n) {
            const i32 s16 = (i32)(((size_t)wbase >> 2) & 3);
            const u32* wb16 = wbase - s16;                             // 16-byte aligned; positions below are relative to it
            const i32 clow = (b.wlow + s16) >> 2;                      // chunk holding the first byte of the stream
            const u8* gb = reinterpret_cast<const u8*>(wb16) - 16 * (ZL_LIT_RING_NS - 1);
            const i32 cmin = clow + (ZL_LIT_RING_NS - 1);
            const u32 th = zl_smem_addr(huf);
            i32 pos = 32 * (b.wi + 2 + s16) + b.n, prev = pos;
            zl_ring_start<ZL_LIT_RING_NS>(ring, wb16, pos, clow);
            // a chunk is first read >= 13 reloads after its copy (7 chunks of lead, <= 55 bits per reload), so one group per
            // iteration and "wait_group 2" always cover it
#define ZL_HUF_SYM5(e0, e1, e2, e3, e4)                                                                                     \
            {                                                                                                               \
                u32 hi, lo;                                                                                                 \
                ZL_RING_RELOAD(ZL_LIT_RING_NS, "", ring, gb, cmin, pos, prev, hi, lo);                                      \
                prev = pos;                                                                                                 \
                e0 = zl_lds16(th + ((hi >> sh) << 1)); hi = __funnelshift_l(lo, hi, e0 >> 8); lo <<= e0 >> 8;              \
                e1 = zl_lds16(th + ((hi >> sh) << 1)); hi = __funnelshift_l(lo, hi, e1 >> 8); lo <<= e1 >> 8;              \
                e2 = zl_lds16(th + ((hi >> sh) << 1)); hi = __funnelshift_l(lo, hi, e2 >> 8); lo <<= e2 >> 8;              \
                e3 = zl_lds16(th + ((hi >> sh) << 1)); hi = __funnelshift_l(lo, hi, e3 >> 8);                              \
                e4 = zl_lds16(th + ((hi >> sh) << 1));                                                                      \
                pos -= (i32)((e0 >> 8) + (e1 >> 8) + (e2 >> 8) + (e3 >> 8) + (e4 >> 8));                                   \
            }
            do {
                u32 e[20];
                asm volatile("cp.async.wait_group 2;" ::: "memory");
                ZL_HUF_SYM5(e[0], e[1], e[2], e[3], e[4]);
                ZL_HUF_SYM5(e[5], e[6], e[7], e[8], e[9]);
                ZL_HUF_SYM5(e[10], e[11], e[12], e[13], e[14]);
                ZL_HUF_SYM5(e[15], e[16], e[17], e[18], e[19]);
                asm volatile("cp.async.commit_group;" ::: "memory");
#pragma unroll
                for (u32 k = 0; k < 5; k++)            // streaming stores: keep L1 for the table
                    __stcs((u32*)(out + i) + k, __byte_perm(__byte_perm(e[4 * k], e[4 * k + 1], 0x40u), __byte_perm(e[4 * k + 2], e[4 * k + 3], 0x40u), 0x5410u));
                i += 20;
            } while (i + 20 <= n);
#undef ZL_HUF_SYM5
            zl_ring_to_br<ZL_LIT_RING_NS>(b, ring, pos, s16);
        }
    } else {
        const u32 count = n;                       // `n` below is the window's valid-bit count (macro convention)
        u32 hi = b.hi, lo = b.lo, nextw = b.nextw;
        i32 wi = b.wi;
        const i32 wlow = b.wlow;
        const u32 th = zl_smem_addr(huf);
        {
            i32 n = b.n;
#define ZL_HUF_SYM_DEV(dst) { const u32 e = zl_lds16(th + ((hi >> sh) << 1)); const u32 nb = e >> 8; \
                              hi = zl_fsl(lo, hi, nb); lo <<= nb; n -= (i32)nb; dst = e & 0xFF; }
            while (i + 4 <= count) {
                u32 s0, s1, s2, s3;
                ZL_REFILL_DEV(); ZL_HUF_SYM_DEV(s0); ZL_HUF_SYM_DEV(s1);
                ZL_REFILL_DEV(); ZL_HUF_SYM_DEV(s2); ZL_HUF_SYM_DEV(s3);
                __stcs((u32*)(out + i), s0 | (s1 << 8) | (s2 << 16) | (s3 << 24));      // streaming store: keep L1 for the bitstreams
                i += 4;
            }
#undef ZL_HUF_SYM_DEV
            b.n = n;
        }
        b.hi = hi; b.lo = lo; b.nextw = nextw; b.wi = wi;
    }
#else
    while (i + 4 <= n) {
        u32 s0, s1, s2, s3;
        zl_br_refill(b, wbase); ZL_HUF_SYM(s0); ZL_HUF_SYM(s1);
        zl_br_refill(b, wbase); ZL_HUF_SYM(s2); ZL_HUF_SYM(s3);
        *(u32*)(out + i) = s0 | (s1 << 8) | (s2 << 16) | (s3 << 24);
        i += 4;
    }
#endif
    while (i < n) { u32 s; zl_br_refill(b, wbase); ZL_HUF_SYM(s); out[i++] = (u8)s; }
#undef ZL_HUF_SYM
    const i32 rem = zl_br_remaining(b, bias, beg);
    return rem == 0 ? 0u : (rem > 0 ? 2u : 1u);
}

// Literals of one block (lane 0): re-reads the section header K0 validated, loads the Huffman tree description from the
// block that carries it (this one, or an earlier one for "treeless" literals) and lays out the streams.
// useDictHuf is set when the tree is the dictionary's (the caller copies that table instead of filling one).
ZL_HD void zl_lit_unit_head(ZlLitSm& f, const ZlFrameDesc& d, const ZlBlockHdr* hdrs, u32 blk, const u32* wbase, u32 bias,
                            u32* useDictHuf)
{
    ZlLitCtl& c = f.ctl;
    const ZlBlockHdr& h = hdrs[blk];
    c.err = 0; c.needHufFill = 0; c.nStreams = 0; c.sStrict = 1; *useDictHuf = 0;
    if (((h.flags >> 4) & 3) != 2) return;                                   // raw / rle literals: nothing to decode
    const u8* src = d.src;
    const u8* bp = src + h.litSecOff;
    const u32 fmt = (bp[0] >> 2) & 3;
    const u32 lhc = zl_rd32(bp);
    u32 single = 0, lhSize, litSize, litCSize;
    if (fmt < 2) { single = !fmt; lhSize = 3; litSize = (lhc >> 4) & 0x3FF; litCSize = (lhc >> 14) & 0x3FF; }
    else if (fmt == 2) { lhSize = 4; litSize = (lhc >> 4) & 0x3FFF; litCSize = lhc >> 18; }
    else { lhSize = 5; litSize = (lhc >> 4) & 0x3FFFF; litCSize = (lhc >> 22) + ((u32)bp[4] << 10); }
    u32 hs = h.litSecOff + lhSize, hsz = litCSize;
    // the tree: zstd.c:43190-43260
    if (h.hufDef == ZL_DEF_NONE) *useDictHuf = 1;
    else {
        const ZlBlockHdr& dh = hdrs[h.hufDef];
        const u8* dp = src + dh.litSecOff;
        const u32 dfmt = (dp[0] >> 2) & 3;
        const u32 dlh = dfmt < 2 ? 3u : (dfmt == 2 ? 4u : 5u);
        const u32 dlhc = zl_rd32(dp);
        const u32 dcs = dfmt < 2 ? ((dlhc >> 14) & 0x3FFu) : (dfmt == 2 ? (dlhc >> 18) : ((dlhc >> 22) + ((u32)dp[4] << 10)));
        const u32 th = zl_huf_read_stats(f, dp + dlh, dcs, wbase, bias, dh.litSecOff + dlh);
        if (!th || th >= dcs) { c.err = ZL_E_corruption_detected; return; }
        c.needHufFill = 1;
        if (h.hufDef == blk) { hs += th; hsz -= th; }                        // own tree: the streams follow it
    }
    if (single) {
        c.nStreams = 1; c.sBeg[0] = hs; c.sEnd[0] = hs + hsz; c.sOut[0] = h.litOff; c.sLen[0] = litSize; c.sStrict = 1;
    } else if (hsz < 10) c.err = ZL_E_corruption_detected;                   // zstd.c:38659
    else {
        const u32 l1 = zl_rd16(src + hs), l2 = zl_rd16(src + hs + 2), l3 = zl_rd16(src + hs + 4);
        const u32 seg = (litSize + 3) / 4;
        if (6 + l1 + l2 + l3 > hsz || seg * 3 > litSize) c.err = ZL_E_corruption_detected;
        else {
            c.nStreams = 4;
            c.sBeg[0] = hs + 6; c.sEnd[0] = c.sBeg[0] + l1;
            c.sBeg[1] = c.sEnd[0]; c.sEnd[1] = c.sBeg[1] + l2;
            c.sBeg[2] = c.sEnd[1]; c.sEnd[2] = c.sBeg[2] + l3;
            c.sBeg[3] = c.sEnd[2]; c.sEnd[3] = hs + hsz;
            for (u32 k = 0; k < 4; k++) { c.sOut[k] = h.litOff + k * seg; c.sLen[k] = seg; }
            c.sLen[3] = litSize - 3 * seg;
            // libzstd's 4-stream decoder only insists on exact consumption when it cannot take its "fast" path, i.e. when a
            // stream is shorter than 8 bytes (HUF_DecompressFastArgs_init, zstd.c:38772-38850; the fast path checks the
            // regenerated sizes only); the single-stream decoder always does (zstd.c:38647).  Same here for bits LEFT OVER
            // (sErr == 2), so that a damaged frame without checksum decodes to the same bytes as with the reference.  A
            // reader that runs past the START of its stream (sErr == 1) is always an error here (zl_lit_unit_finish):
            // libzstd's fast loop reads on into the bytes in front of the stream and returns garbage -- the one place
            // where this decoder is deliberately stricter on damaged input (DESIGN.md, "Decoder limits").
            c.sStrict = (l1 < 8 || l2 < 8 || l3 < 8 || c.sEnd[3] - c.sBeg[3] < 8) ? 1u : 0u;
        }
    }
}
// after the streams ran (lane 0): 0 or the error of this block
ZL_HD u32 zl_lit_unit_finish(const ZlLitSm& f)
{
    const ZlLitCtl& c = f.ctl;
    if (c.err) return c.err;
    for (u32 k = 0; k < c.nStreams; k++) if (c.sErr[k] == 1 || (c.sErr[k] == 2 && c.sStrict)) return ZL_E_corruption_detected;
    return 0;
}

// =================================================================================================== K1b: sequences
struct ZlSeqCtl {
    u32 err;
    u32 nbSeq;
    u32 needBuild;      // bit t: build table t (0 LL, 1 OF, 2 ML) from norm[t]
    u32 useDict;        // bit t: table t is the dictionary's (the caller copies it)
    u32 tlog[3], maxSym[3], bErr[3];
    u32 bitBeg, bitEnd;
};
struct ZlSeqSm {            // 2,632 B: with 8 blocks per warp, 10 warps fit one SM's shared memory
    u16 fseLL[512];
    u16 fseML[512];
    u16 fseOF[256];
    ZlSeqCtl ctl;
};
#define ZL_NORM_STRIDE 64       // i16 per table in the per-unit normalized-count scratch (3 tables)

// One table description at src[ip..iend) for table t with the given mode (0 predefined, 1 RLE, 2 FSE-compressed): loads it
// into f (cell / norm + needBuild) when `load`, and returns the bytes it occupies (0xFFFFFFFF on error).
ZL_HD u32 zl_seq_table_desc(ZlSeqSm& f, const u8* src, u32 ip, u32 iend, u32 t, u32 mode, bool load, const ZlConstTables& ct, i16* norm)
{
    ZlSeqCtl& c = f.ctl;
    const u32 maxSymT[3] = {35, 31, 52}, maxLogT[3] = {9, 8, 9}, defLogT[3] = {6, 5, 6};
    u16* tbl = t == 0 ? f.fseLL : (t == 1 ? f.fseOF : f.fseML);
    i16* nt = norm + t * ZL_NORM_STRIDE;
    if (mode == 0) {                               // predefined
        if (load) {
            const i16* def = t == 0 ? ct.llDef : (t == 1 ? ct.ofDef : ct.mlDef);
            const u32 nsym = t == 0 ? 36 : (t == 1 ? 29 : 53);
            for (u32 s = 0; s < nsym; s++) nt[s] = def[s];
            c.maxSym[t] = nsym - 1; c.tlog[t] = defLogT[t]; c.needBuild |= 1u << t;
        }
        return 0;
    }
    if (mode == 1) {                               // RLE
        if (ip >= iend) return 0xFFFFFFFFu;
        const u32 sy = src[ip];
        if (sy > maxSymT[t]) return 0xFFFFFFFFu;
        if (load) { tbl[0] = zl_seq_cell(1, sy); c.tlog[t] = 0; }
        return 1;
    }
    u32 ms = maxSymT[t], tl;                       // FSE-compressed (the counts land in this table's scratch slot either way)
    const u32 hsz = zl_read_ncount(src + ip, iend - ip, nt, &ms, &tl);
    if (!hsz || tl > maxLogT[t]) return 0xFFFFFFFFu;
    if (load) { c.maxSym[t] = ms; c.tlog[t] = tl; c.needBuild |= 1u << t; }
    return hsz;
}

// sequences section header of block `blk` (lane 0): zstd.c:43707-43790.  A table in "repeat" mode is re-read from the
// block that last defined it (K0 recorded which one), so blocks decode independently of each other.
// `norm` = 3 x ZL_NORM_STRIDE i16 of scratch (global memory in the kernel).
ZL_HD void zl_seq_head(ZlSeqSm& f, const ZlFrameDesc& d, const ZlBlockHdr* hdrs, u32 blk, const ZlConstTables& ct, i16* norm)
{
    ZlSeqCtl& c = f.ctl;
    const ZlBlockHdr& h = hdrs[blk];
    c.err = 0; c.needBuild = 0; c.useDict = 0; c.nbSeq = h.nbSeq;
    c.bErr[0] = c.bErr[1] = c.bErr[2] = 0;
    if (!h.nbSeq) return;                          // (the index kernel checked that nothing follows nbSeq == 0, zstd.c:43736)
    const u8* src = d.src;
    u32 ip = h.seqOff + (h.nbSeq < 128 ? 1u : (h.nbSeq < 0x7F00 ? 2u : 3u));
    const u32 iend = h.seqEnd;
    const u32 modes = src[ip++];
    for (u32 t = 0; t < 3; t++) {
        const u32 mode = (modes >> (6 - 2 * t)) & 3;
        if (mode != 3) {
            const u32 used = zl_seq_table_desc(f, src, ip, iend, t, mode, true, ct, norm);
            if (used == 0xFFFFFFFFu) { c.err = ZL_E_corruption_detected; return; }
            ip += used;
        } else if (h.seqDef[t] == ZL_DEF_NONE) c.useDict |= 1u << t;
        else {                                          // walk the defining block's descriptions up to table t
            const ZlBlockHdr& dh = hdrs[h.seqDef[t]];
            u32 q = dh.seqOff + (dh.nbSeq < 128 ? 1u : (dh.nbSeq < 0x7F00 ? 2u : 3u));
            const u32 dm = src[q++];
            for (u32 tt = 0; tt <= t; tt++) {
                const u32 m2 = (dm >> (6 - 2 * tt)) & 3;
                if (m2 == 3) continue;                  // takes no bytes (and cannot be tt == t: K0 only names defining blocks)
                // earlier tables of that block are only measured; their counts go through table t's scratch slot
                const u32 used = tt == t ? zl_seq_table_desc(f, src, q, dh.seqEnd, t, m2, true, ct, norm)
                                         : (m2 == 2 ? [&]() { u32 ms = tt == 0 ? 35u : (tt == 1 ? 31u : 52u), tl; const u32 r = zl_read_ncount(src + q, dh.seqEnd - q, norm + t * ZL_NORM_STRIDE, &ms, &tl); return r ? r : 0xFFFFFFFFu; }()
                                                    : (m2 == 1 ? 1u : 0u));
                if (used == 0xFFFFFFFFu) { c.err = ZL_E_corruption_detected; return; }
                q += used;
            }
        }
    }
    c.bitBeg = ip; c.bitEnd = iend;
}

ZL_HD void zl_seq_fse_build(ZlSeqSm& f, u32 t, const i16* norm)
{
    ZlSeqCtl& c = f.ctl;
    c.bErr[t] = 0;
    if (!((c.needBuild >> t) & 1)) return;
    u16* tbl = t == 0 ? f.fseLL : (t == 1 ? f.fseOF : f.fseML);
    if (!zl_fse_build(tbl, norm + t * ZL_NORM_STRIDE, c.maxSym[t], c.tlog[t])) c.bErr[t] = 1;
}

// ---- sequence records (K1b -> K2) ---------------------------------------------------------------------------------------
// K1b only runs the part of ZSTD_decodeSequence (zstd.c:44241-44358) that is inherently serial: the three FSE state
// chains and the bit cursor.  Everything else -- extracting the additional bits, the base values, the repeat-offset
// history (zstd.c:44290-44326), the bounds checks of ZSTD_execSequence (44024-44066) -- happens in K2, 32 sequences at a
// time across the lanes of a warp.  A record is one u64 in one of two forms:
//   form A (bit 63 = 0)  [0:32) the 32 stream bits that start with this sequence's additional bits (OF, ML, LL in that order)
//                        [32:38) LL code  [38:44) ML code  [44:49) OF code           -- requires LL+ML+OF bits <= 32
//   form B (bit 63 = 1)  [0:16) litLength  [16:32) matchLength  [32:63) offBase      -- explicit values, written by the
//                        generic step; lengths >= 65536 are split: (65535, 0, 0) carries literals only, (0, m, 0) continues
//                        the previous match at the same offset without touching the history
// offBase = (1 << OFcode) + OFbits: 1..3 are the repeat codes, >= 4 is offset + 3 (zstd.c:19648-19652).
#define ZL_REC_B (1ull << 63)
ZL_HD u64 zl_rec_a(u32 snap, u32 llCode, u32 mlCode, u32 ofCode) { return (u64)snap | ((u64)(llCode | (mlCode << 6) | (ofCode << 12)) << 32); }
ZL_HD u64 zl_rec_b(u32 ll, u32 ml, u32 offBase) { return ZL_REC_B | ((u64)offBase << 32) | ((u64)ml << 16) | (u64)ll; }
// record -> (ll, ml, offBase); ct supplies the base / bits tables (zstd.c:15470-15495, 40060-40075)
ZL_HD void zl_rec_decode(u64 r, const u32* llBase, const u8* llBits, const u32* mlBase, const u8* mlBits, u32& ll, u32& ml, u32& ob)
{
    if (r & ZL_REC_B) { ll = (u32)r & 0xFFFFu; ml = ((u32)r >> 16) & 0xFFFFu; ob = (u32)(r >> 32) & 0x7FFFFFFFu; return; }
    const u32 snap = (u32)r, c = (u32)(r >> 32);
    const u32 llCode = c & 63u, mlCode = (c >> 6) & 63u, aOF = (c >> 12) & 31u;
    const u32 aML = mlBits[mlCode], aLL = llBits[llCode];
    ob = (1u << aOF) + zl_shr(snap, 32u - aOF);
    ml = mlBase[mlCode] + zl_shr(zl_shl(snap, aOF), 32u - aML);
    ll = llBase[llCode] + zl_shr(zl_shl(snap, aOF + aML), 32u - aLL);
}
// Repeat-offset history step (zstd.c:44290-44326): resolves offBase against h[3], updates h, returns the offset
// (0 = invalid: "rep0 - 1" with rep0 == 1).  ml == 0 records and offBase == 0 continuations leave the history alone.
ZL_HD u32 zl_rep_resolve(u32 h[3], u32 ll, u32 ml, u32 ob)
{
    if (ml == 0) return 0;
    if (ob == 0) return h[0];
    if (ob >= 4) { const u32 off = ob - 3; h[2] = h[1]; h[1] = h[0]; h[0] = off; return off; }
    const u32 idx = ob - 1 + (ll == 0 ? 1u : 0u);
    if (idx == 0) return h[0];
    const u32 off = idx == 1 ? h[1] : (idx == 2 ? h[2] : h[0] - 1);
    if (idx >= 2) h[2] = h[1];
    h[1] = h[0]; h[0] = off;
    return off;
}

struct ZlSeqRegs {
    u32 sLL, sOF, sML;
    u32 nrec, err;
};
// One sequence, generic form (first / last sequence of a block, more than 32 additional bits, lengths that may reach 65536).
template <bool kLast>
ZL_HD void zl_seq_step(const ZlSeqSm& f, ZlBitR& b, const u32* wbase, const ZlConstTables& ct, ZlSeqRegs& r, u64* rp, u32 recCap)
{
    zl_br_refill(b, wbase);                                              // n >= 33
    const u32 eLL = f.fseLL[r.sLL], eOF = f.fseOF[r.sOF], eML = f.fseML[r.sML];
    const u32 llCode = ZL_CELL_SYM(eLL), mlCode = ZL_CELL_SYM(eML);
    const u32 aOF = ZL_CELL_SYM(eOF), aML = ct.mlBits[mlCode], aLL = ct.llBits[llCode];
    const u32 cA = aOF + aML + aLL;
    u32 ofx, mlx, llx;
    if (cA <= 32) {
        const u32 hi = b.hi, lo = b.lo;
        ofx = zl_shr(hi, 32u - aOF);
        mlx = zl_shr(zl_fsl(lo, hi, aOF), 32u - aML);
        llx = zl_shr(zl_fsl(lo, hi, aOF + aML), 32u - aLL);
        zl_br_skip(b, cA);
    } else {                                                             // very long offsets + lengths
        ofx = zl_br_take(b, aOF);
        zl_br_refill(b, wbase);
        mlx = zl_br_take(b, aML);
        llx = zl_br_take(b, aLL);
    }
    if (!kLast) {                                                        // LL, ML, OF order: zstd.c:44347-44353
        zl_br_refill(b, wbase);
        const u32 gLL = f.ctl.tlog[0], gOF = f.ctl.tlog[1], gML = f.ctl.tlog[2];
        const u32 nLL = ZL_CELL_NS(eLL), nML = ZL_CELL_NS(eML), nOF = ZL_CELL_NS(eOF);
        const u32 bLL = gLL - zl_highbit(nLL), bML = gML - zl_highbit(nML), bOF = gOF - zl_highbit(nOF);
        const u32 hi = b.hi, lo = b.lo;
        r.sLL = ((nLL << bLL) - (1u << gLL)) + zl_shr(hi, 32u - bLL);
        r.sML = ((nML << bML) - (1u << gML)) + zl_shr(zl_fsl(lo, hi, bLL), 32u - bML);
        r.sOF = ((nOF << bOF) - (1u << gOF)) + zl_shr(zl_fsl(lo, hi, bLL + bML), 32u - bOF);
        zl_br_skip(b, bLL + bML + bOF);                                  // <= 26 bits
    }
    if (aOF >= 31) { r.err = ZL_E_corruption_detected; return; }         // offsets of 2 GiB and more exceed any history we accept
    u32 ll = ct.llBase[llCode] + llx;
    u32 ml = ct.mlBase[mlCode] + mlx;
    const u32 ob = (1u << aOF) + ofx;
    while (ll > 65535) {                                                 // lengths >= 65536: several records
        if (r.nrec >= recCap) { r.err = ZL_E_GENERIC; return; }
        rp[r.nrec++] = zl_rec_b(65535, 0, 0);
        ll -= 65535;
    }
    u32 first = 1;
    do {
        const u32 m = ml > 65535 ? 65535 : ml;
        if (r.nrec >= recCap) { r.err = ZL_E_GENERIC; return; }
        rp[r.nrec++] = zl_rec_b(ll, m, first ? ob : 0u);
        ll = 0; ml -= m; first = 0;
    } while (ml);
}

#if defined(__CUDACC__)
// code -> (base value | additional bits << 24) for LL (36 entries) then ML (53 entries), in shared memory
#define ZL_XTAB_WORDS (36 + 53)
// Fast path over consecutive non-last sequences whose additional bits fit one 32-bit snapshot and whose lengths fit
// 16 bits.  Returns how many sequences it consumed; it stops BEFORE any sequence it cannot handle (the generic
// zl_seq_step takes that one).  The loop is rotated: the three table cells of the next sequence are requested as soon as
// the new states are known.  States are kept "primed" (state + table size): a primed state is simply the cell's ns with
// the nbBits fresh stream bits shifted in from the right -- one funnel shift -- and indexes the table at (base - size).
// With a ring, one reload per sequence: a sequence takes at most 32 + 26 bits of the 64, and the reload for the next one
// runs beside that sequence's cell loads, off the chain of dependent instructions.
__device__ __forceinline__ u32 zl_seq_fast_loop(const ZlSeqSm& f, const u32* xtab, ZlBitR& b, const u32* wbase,
                                                ZlSeqRegs& r, u64* rp, u32 maxIter, u32 safeCap, u32 ring)
{
    const u32 gLL = f.ctl.tlog[0], gOF = f.ctl.tlog[1], gML = f.ctl.tlog[2];
    const u32 zLL = 1u << gLL, zOF = 1u << gOF, zML = 1u << gML;
    const u32 tLL = zl_opaque(zl_smem_addr(f.fseLL) - 2u * zLL), tOF = zl_opaque(zl_smem_addr(f.fseOF) - 2u * zOF),
              tML = zl_opaque(zl_smem_addr(f.fseML) - 2u * zML);
    const u32 kLL = 31u - gLL, kOF = 31u - gOF, kML = 31u - gML;          // nbBits = clz(ns) - k
    const u32 cLL = zl_opaque(zl_smem_addr(xtab)), cML = cLL + 36u * 4u;
    u32 sLL = r.sLL + zLL, sOF = r.sOF + zOF, sML = r.sML + zML;
    u64* wp = rp + r.nrec;
    const u32 room = safeCap > r.nrec ? safeCap - r.nrec : 0u;
    if (maxIter > room) maxIter = room;
    u32 eLL = zl_lds16(tLL + (sLL << 1)), eOF = zl_lds16(tOF + (sOF << 1)), eML = zl_lds16(tML + (sML << 1));
    u32 it = 0;
#define ZL_SEQ_HEAD                                                                                                         \
        const u32 llCode = ZL_CELL_SYM(eLL), mlCode = ZL_CELL_SYM(eML), aOF = ZL_CELL_SYM(eOF);                             \
        const u32 xl = zl_lds32(cLL + (llCode << 2)), xm = zl_lds32(cML + (mlCode << 2));                                   \
        const u32 nLL = ZL_CELL_NS(eLL), nML = ZL_CELL_NS(eML), nOF = ZL_CELL_NS(eOF);                                      \
        const u32 bLL = (u32)__clz((int)nLL) - kLL, bML = (u32)__clz((int)nML) - kML, bOF = (u32)__clz((int)nOF) - kOF;     \
        const u32 cA = aOF + (xl >> 24) + (xm >> 24);                                                                       \
        if (cA > 32 || llCode >= 35 || mlCode >= 50) break;                                                                 \
        const u32 d2 = bLL + bML, cB = d2 + bOF;
    if (ring != ZL_NO_RING) {
        const i32 s16 = (i32)(((size_t)wbase >> 2) & 3);
        const u32* wb16 = wbase - s16;
        const i32 clow = (b.wlow + s16) >> 2;
        const u8* gb = reinterpret_cast<const u8*>(wb16) - 16 * (ZL_SEQ_RING_NS - 1);
        const i32 cmin = clow + (ZL_SEQ_RING_NS - 1);
        i32 pos = 32 * (b.wi + 2 + s16) + b.n;
        zl_ring_start<ZL_SEQ_RING_NS>(ring, wb16, pos, clow);
        u32 hi, lo;
        // one group per sequence: a chunk is first read >= 4 reloads after its copy (3 chunks of lead, <= 58 bits per reload)
        ZL_RING_RELOAD(ZL_SEQ_RING_NS, "cp.async.commit_group;\n\tcp.async.wait_group 4;\n\t", ring, gb, cmin, pos, pos, hi, lo);
        while (it < maxIter) {
            ZL_SEQ_HEAD
            const u32 h2 = zl_fsl(lo, hi, cA), l2 = zl_shl(lo, cA);
            sLL = __funnelshift_l(h2, nLL, bLL);
            sML = __funnelshift_l(zl_fsl(l2, h2, bLL), nML, bML);
            sOF = __funnelshift_l(zl_fsl(l2, h2, d2), nOF, bOF);
            eLL = zl_lds16(tLL + (sLL << 1)); eOF = zl_lds16(tOF + (sOF << 1)); eML = zl_lds16(tML + (sML << 1));
            __stcs(wp++, zl_rec_a(hi, llCode, mlCode, aOF));
            const i32 np = pos - (i32)(cA + cB);
            ZL_RING_RELOAD(ZL_SEQ_RING_NS, "cp.async.commit_group;\n\tcp.async.wait_group 4;\n\t", ring, gb, cmin, np, pos, hi, lo);
            pos = np;
            it++;
        }
        zl_ring_to_br<ZL_SEQ_RING_NS>(b, ring, pos, s16);
    } else {
        u32 hi = b.hi, lo = b.lo, nextw = b.nextw;
        i32 n = b.n, wi = b.wi;
        const i32 wlow = b.wlow;
        while (it < maxIter) {
            ZL_SEQ_HEAD
            ZL_REFILL_DEV();
            const u32 snap = hi;
            hi = zl_fsl(lo, hi, cA); lo = zl_shl(lo, cA); n -= (i32)cA;
            ZL_REFILL_DEV();
            sLL = __funnelshift_l(hi, nLL, bLL);
            sML = __funnelshift_l(zl_fsl(lo, hi, bLL), nML, bML);
            sOF = __funnelshift_l(zl_fsl(lo, hi, d2), nOF, bOF);
            hi = zl_fsl(lo, hi, cB); lo <<= cB; n -= (i32)cB;
            eLL = zl_lds16(tLL + (sLL << 1)); eOF = zl_lds16(tOF + (sOF << 1)); eML = zl_lds16(tML + (sML << 1));
            __stcs(wp++, zl_rec_a(snap, llCode, mlCode, aOF));
            it++;
        }
        b.hi = hi; b.lo = lo; b.nextw = nextw; b.n = n; b.wi = wi;
    }
#undef ZL_SEQ_HEAD
    r.sLL = sLL - zLL; r.sOF = sOF - zOF; r.sML = sML - zML;
    r.nrec += it;
    return it;
}
#endif

// serial sequence decode of one block (lane 0): zstd.c:44627-44700.  Completes the block's ZlBlockHdr (nrec, recOff);
// the regenerated size is only known once K2 has added up the lengths.
// `xtab` and `ring` (the unit's stream ring, ZL_SEQ_RING_NS slots; ZL_NO_RING = none) are only used by the device fast path
// (null / none in the CPU emulation).
// `recs` = this block's slice of the record arena (room for nbSeq + 4 records: a block regenerates <= 128 KiB, so at most
// two lengths can be split); returns the number of records written.
ZL_HD u32 zl_seq_decode(ZlSeqSm& f, u64* recs, const u32* wbase, u32 bias, const ZlConstTables& ct, const u32* xtab, u32 ring = ZL_NO_RING)
{
    (void)xtab; (void)ring;
    ZlSeqCtl& c = f.ctl;
    if (!c.err && c.needBuild) { for (u32 t = 0; t < 3; t++) if (c.bErr[t]) c.err = ZL_E_corruption_detected; }
    u64* rp = recs;
    const u32 recCap = c.nbSeq + ZL_REC_SLACK;
    ZlSeqRegs r;
    r.nrec = 0; r.err = 0;
    if (!c.err && c.nbSeq) {
        ZlBitR b;
        if (!zl_br_init(b, wbase, bias, c.bitBeg, c.bitEnd)) c.err = ZL_E_corruption_detected;
        else {
            zl_br_refill(b, wbase);
            r.sLL = zl_br_take(b, c.tlog[0]);
            r.sOF = zl_br_take(b, c.tlog[1]);
            zl_br_refill(b, wbase);
            r.sML = zl_br_take(b, c.tlog[2]);
            const u32 nbSeq = c.nbSeq;
            const u32 safeCap = recCap - 4;                  // split path re-checks exactly
            for (u32 i = 0; i + 1 < nbSeq; i++) {
#if defined(__CUDA_ARCH__)
                i += zl_seq_fast_loop(f, xtab, b, wbase, r, rp, nbSeq - 1 - i, safeCap, ring);
                if (r.nrec >= safeCap || i + 1 >= nbSeq) break;
#endif
                zl_seq_step<false>(f, b, wbase, ct, r, rp, recCap);
                if (r.err || r.nrec >= safeCap) break;
            }
            if (!r.err && r.nrec >= safeCap && nbSeq > 1) r.err = ZL_E_corruption_detected;
            if (!r.err) zl_seq_step<true>(f, b, wbase, ct, r, rp, recCap);
            if (!r.err && zl_br_remaining(b, bias, c.bitBeg) != 0) r.err = ZL_E_corruption_detected;      // zstd.c:44686
            if (r.err) c.err = r.err;
        }
    }
    return c.err ? 0u : r.nrec;
}

