// zl_dec_kernels.cu -- the decode kernels and their launchers (sm_100a).
//   K1a zl_k_literals / K1b zl_k_sequences   quad-per-frame entropy decode -> literal / record / header arenas
//   K2 zl_k_execute   warp-per-frame sequence execution -> frame output
//   K3 zl_k_checksum  quad-per-frame XXH64 of the output, compared with the frame trailer (and a seek table's checksum)
//   zl_k_range_scatter  warp-per-piece copy-out of zl_decompress_ranges
//   zl_k_idx_*          the frame index of a stream in device memory (zl_dec_index.cuh)
#include "zl_dec_entropy.cuh"
#include "zl_dec_exec.cuh"
#include "zl_dec_large.cuh"
#include "zl_launch.h"
#include "zl_plan.h"
#include "zl_dec_index.cuh"
#include <mutex>
#include <stdlib.h>

__constant__ ZlConstTables c_tables = {
    ZL_LL_BASE_INIT, ZL_ML_BASE_INIT, ZL_LL_BITS_INIT, ZL_ML_BITS_INIT,
    ZL_LL_DEFNORM_INIT, ZL_ML_DEFNORM_INIT, ZL_OF_DEFNORM_INIT};

// ---- K0: index ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
zl_k_index(const ZlFrameDesc* __restrict__ descs, ZlFrameInfo* __restrict__ infos, ZlBlockHdr* hdrArena, ZlUnit* units, u32* unitCount,
           u32 unitCap, u32 nframes, u32 frameBase, const ZlDictDev* dict)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nframes) return;
    const ZlFrameDesc d = descs[i];
    ZlFrameInfo info;
    zl_index_frame(d, info, hdrArena + d.hdrBase, frameBase + i, dict ? dict->dictID : 0u, (dict && dict->hasEntropy) ? 1u : 0u,
                   units, unitCount, unitCap);
    infos[i] = info;
}

// Units are fetched dynamically, 8 at a time per warp (one per quad), so expensive and cheap blocks balance across the grid.
__device__ __forceinline__ u32 zl_fetch_units(u32* cursor, u32 lane, u32 count = ZL_QUADS_PER_WARP)
{
    u32 base = 0;
    if (lane == 0) base = atomicAdd(cursor, count);
    return __shfl_sync(0xFFFFFFFFu, base, 0);
}

// ---- K1a: literals ------------------------------------------------------------------------------------------
#ifndef ZL_LIT_RING
#define ZL_LIT_RING 1        // 0: stream words by global loads (the round-1 path, kept for A/B measurements)
#endif
// descs / infos are indexed by the GLOBAL frame number carried by the unit
__global__ void __launch_bounds__(32)
zl_k_literals(const ZlFrameDesc* __restrict__ descs, ZlFrameInfo* __restrict__ infos, const ZlBlockHdr* hdrArena,
              u8* litArena, const ZlUnit* __restrict__ units, const u32* __restrict__ unitCount, u32* cursor, const ZlDictDev* dict)
{
    extern __shared__ __align__(128) u8 smraw[];
    // stream ring first (its lanes' slots must be aligned to their 128 bytes, zl_huf_stream), then the eight units
    const u32 ringBytes = ZL_LIT_RING ? 32u * 16u * ZL_LIT_RING_NS : 0u;
    ZlLitSm* fs = reinterpret_cast<ZlLitSm*>(smraw + ringBytes);
    const u32 lane = threadIdx.x, quad = lane >> 2, q = lane & 3;
    const u32 qmask = 0xFu << (quad * 4);
    ZlLitSm& f = fs[quad];
    const u32 ring = ZL_LIT_RING ? zl_smem_addr(smraw) + lane * 16u * ZL_LIT_RING_NS : ZL_NO_RING;
    // the dictionary's Huffman table, once per CTA (behind the units): units with treeless literals that fall back on it decode from this
    // copy instead of copying 4 KB each (config 3: every object of a few hundred bytes did -- 512 load/store pairs per lane and unit)
    u16* dictHuf = reinterpret_cast<u16*>(smraw + ringBytes + ZL_QUADS_PER_WARP * sizeof(ZlLitSm));
    if (dict && dict->hasEntropy) {
        const uint4* g = reinterpret_cast<const uint4*>(dict->huf);
        for (u32 i = lane; i < 2048 * 2 / 16; i += 32) reinterpret_cast<uint4*>(dictHuf)[i] = g[i];
        __syncwarp();
    }
    const u32 nunits = *unitCount;
    for (;;) {
        const u32 ubase = zl_fetch_units(cursor, lane);
        if (ubase >= nunits) break;
        const u32 u = ubase + quad;
        if (u < nunits) {
            const ZlUnit un = units[u];
            const ZlFrameDesc d = descs[un.frame];
            const ZlBlockHdr* hdrs = hdrArena + d.hdrBase;
            const u32 litMode = (hdrs[un.block].flags >> 4) & 3;
            if (litMode == 2) {                                        // (units with raw / rle literals only have sequences)
                // ZL_BLK_DIRECT: the block's literals ARE its output
                u8* lits = (hdrs[un.block].flags & ZL_BLK_DIRECT) ? d.dst + hdrs[un.block].outOff - hdrs[un.block].litOff : litArena + d.litBase;
                const u32 bias = (u32)(((size_t)d.src) & 3);
                const u32* wbase = reinterpret_cast<const u32*>(d.src - bias);
                u32 useDict = 0;
                if (q == 0) zl_lit_unit_head(f, d, hdrs, un.block, wbase, bias, &useDict);
                useDict = __shfl_sync(qmask, useDict, quad * 4);
                __syncwarp(qmask);
                const u32 fill = f.ctl.needHufFill, ns = f.ctl.err ? 0u : f.ctl.nStreams;
                if (useDict) { if (q == 0) f.ctl.hufLog = dict->hufLog; }      // zstd.c:42140-42159: the dictionary's tree (the CTA's copy)
                else if (fill && !f.ctl.err) zl_huf_fill(f, q);
                __syncwarp(qmask);
                if (q < ns)
                    f.ctl.sErr[q] = zl_huf_stream(useDict ? dictHuf : f.huf, f.ctl.hufLog, wbase, bias, f.ctl.sBeg[q], f.ctl.sEnd[q],
                                                  lits + f.ctl.sOut[q], f.ctl.sLen[q], ring);
                __syncwarp(qmask);
                if (q == 0) { const u32 e = zl_lit_unit_finish(f); if (e) infos[un.frame].err = e; }
                __syncwarp(qmask);
            }
        }
        __syncwarp();
    }
}

// ---- K1b: sequences -----------------------------------------------------------------------------------------
#define ZL_XTAB_BYTES ((ZL_XTAB_WORDS * 4 + 15) & ~15)
#ifndef ZL_SEQ_RING
#define ZL_SEQ_RING 1        // 0: stream words by global loads (kept for A/B measurements)
#endif
__global__ void __launch_bounds__(32)
zl_k_sequences(const ZlFrameDesc* __restrict__ descs, ZlFrameInfo* __restrict__ infos, ZlBlockHdr* hdrArena,
               u64* recArena, i16* normArena, const ZlUnit* __restrict__ units, const u32* __restrict__ unitCount, u32* cursor,
               const ZlDictDev* dict)
{
    extern __shared__ __align__(128) u8 smraw[];
    // stream ring first (its units' slots must be aligned to their 64 bytes, zl_seq_fast_loop), then the code table and the units
    const u32 ringBytes = ZL_SEQ_RING ? 16u * ZL_SEQ_RING_NS * ZL_SEQ_UNITS : 0u;
    u32* xtab = reinterpret_cast<u32*>(smraw + ringBytes);
    ZlSeqSm* fs = reinterpret_cast<ZlSeqSm*>(smraw + ringBytes + ZL_XTAB_BYTES);
    const ZlConstTables& ct = c_tables;          // constant memory: only the header parser and the rare generic step index it
    // ZL_SEQ_G lanes share a unit (ZL_SEQ_UNITS units per warp): lane 0 of the group runs the serial chains, all of them build the tables
    const u32 lane = threadIdx.x, quad = lane / ZL_SEQ_G, q = lane % ZL_SEQ_G;
    const u32 qmask = (0xFFFFFFFFu >> (32 - ZL_SEQ_G)) << (quad * ZL_SEQ_G);
    for (u32 i = lane; i < ZL_XTAB_WORDS; i += 32)
        xtab[i] = i < 36 ? (c_tables.llBase[i] | ((u32)c_tables.llBits[i] << 24)) : (c_tables.mlBase[i - 36] | ((u32)c_tables.mlBits[i - 36] << 24));
    __syncwarp();
    ZlSeqSm& f = fs[quad];
    const u32 ring = ZL_SEQ_RING ? zl_smem_addr(smraw) + quad * 16u * ZL_SEQ_RING_NS : ZL_NO_RING;
    i16* norm = normArena + ((size_t)blockIdx.x * ZL_SEQ_UNITS + quad) * (3 * ZL_NORM_STRIDE);     // scratch per resident unit
    const u32 nunits = *unitCount;
    // few units in all (one large frame, the first small slices of a host-buffer call): a warp takes 8 of them instead of 16, so that
    // they spread over twice as many warps (a 16 MB frame of 123 blocks: 4.31 ms with 16 in lockstep, 4.07 with 8).  Not by units per
    // CTA of this grid: the kernels of the other slices of a batch share the SMs, and a half-used CTA still holds 16 units' tables.
    const u32 take = (nunits <= 1024u && ZL_SEQ_UNITS > 8u) ? 8u : (u32)ZL_SEQ_UNITS;
    for (;;) {
        const u32 ubase = zl_fetch_units(cursor, lane, take);
        if (ubase >= nunits) break;
        const u32 u = ubase + quad;
        if (quad < take && u < nunits) {
            const ZlUnit un = units[u];
            const ZlFrameDesc d = descs[un.frame];
            ZlBlockHdr* hdrs = hdrArena + d.hdrBase;
            if (hdrs[un.block].nbSeq) {
                const u32 bias = (u32)(((size_t)d.src) & 3);
                const u32* wbase = reinterpret_cast<const u32*>(d.src - bias);
                if (q == 0) zl_seq_head(f, d, hdrs, un.block, ct, norm);
                __syncwarp(qmask);
                const u32 build = f.ctl.err ? 0u : f.ctl.needBuild, useDict = f.ctl.err ? 0u : f.ctl.useDict;
                if (useDict) {                                     // zstd.c:42140-42159: tables of the dictionary
                    if (useDict & 1) { for (u32 i = q; i < 512; i += ZL_SEQ_G) f.fseLL[i] = dict->fseLL[i]; if (q == 0) f.ctl.tlog[0] = dict->tlog[0]; }
                    if (useDict & 2) { for (u32 i = q; i < 256; i += ZL_SEQ_G) f.fseOF[i] = dict->fseOF[i]; if (q == 0) f.ctl.tlog[1] = dict->tlog[1]; }
                    if (useDict & 4) { for (u32 i = q; i < 512; i += ZL_SEQ_G) f.fseML[i] = dict->fseML[i]; if (q == 0) f.ctl.tlog[2] = dict->tlog[2]; }
                }
                if (build) {
#if ZL_SEQ_G >= 3
                    if (q < 3) zl_seq_fse_build(f, q, norm);
#elif ZL_SEQ_G == 2
                    if (q == 0) { zl_seq_fse_build(f, 0, norm); zl_seq_fse_build(f, 1, norm); } else zl_seq_fse_build(f, 2, norm);     // LL + OF | ML
#else
                    for (u32 t = 0; t < 3; t++) zl_seq_fse_build(f, t, norm);
#endif
                }
                __syncwarp(qmask);
                if (q == 0) {
                    const u32 nrec = zl_seq_decode(f, recArena + d.recBase + hdrs[un.block].recOff, wbase, bias, ct, xtab, ring);
                    hdrs[un.block].nrec = nrec;
                    if (f.ctl.err) infos[un.frame].err = f.ctl.err;
                }
                __syncwarp(qmask);
            }
        }
        __syncwarp();
    }
}

template <bool kDict>
__global__ void __launch_bounds__(ZL_EXEC_WARPS * 32, ZL_EXEC_MIN_CTAS)
zl_k_execute(const ZlFrameDesc* __restrict__ descs, ZlFrameInfo* __restrict__ infos,
             const ZlBlockHdr* __restrict__ hdrArena, const u64* __restrict__ recArena,
             const u8* __restrict__ litArena, u64* __restrict__ results, u32 nframes, const ZlDictDev* dict)
{
    __shared__ u32 xtab[ZL_XTAB_WORDS];
    __shared__ __align__(16) ZlExecSm execSm[ZL_EXEC_WARPS];
    __shared__ u32 rcp[64];                                           // zl_mod_small
    for (u32 i = threadIdx.x; i < ZL_XTAB_WORDS; i += ZL_EXEC_WARPS * 32)
        xtab[i] = i < 36 ? (c_tables.llBase[i] | ((u32)c_tables.llBits[i] << 24)) : (c_tables.mlBase[i - 36] | ((u32)c_tables.mlBits[i - 36] << 24));
    if (threadIdx.x < 64) rcp[threadIdx.x] = threadIdx.x ? 0xFFFFFFFFu / threadIdx.x : 0u;
    __syncthreads();
    const u32 lane = threadIdx.x & 31;
    const u32 frame = blockIdx.x * ZL_EXEC_WARPS + (threadIdx.x >> 5);
    if (frame >= nframes) return;
    const ZlFrameInfo info = infos[frame];
    if (info.err) { if (lane == 0) results[frame] = (u64)0 - (u64)info.err; return; }
    const ZlFrameDesc d = descs[frame];
    if (d.large) return;                                              // large frames: zl_dec_large.cuh
    const ZlBlockHdr* hdrs = hdrArena + d.hdrBase;
    const u8* dictContent = kDict ? dict->content : nullptr;
    const u32 dictSize = kDict ? dict->contentSize : 0u;
    u32 hist[3] = {1, 4, 8};                                          // zstd.c:15416
    if (kDict && dict->hasEntropy) { hist[0] = dict->rep[0]; hist[1] = dict->rep[1]; hist[2] = dict->rep[2]; }   // zstd.c:42140-42159
    u32 op = 0, err = 0;
    for (u32 b = 0; b < info.nblocks && !err; b++) {
        const ZlBlockHdr h = hdrs[b];
        const u32 type = h.flags & 3;
        const u32 room = d.dstCap - op;
        if (type != 2) {                                              // raw / RLE block (zstd.c:41497-41520)
            if (h.regenSize > room) { err = ZL_E_dstSize_tooSmall; break; }
            if (type == 0) zl_warp_copy(d.dst + op, d.src + h.srcOff, h.regenSize, lane);
            else zl_warp_fill(d.dst + op, (h.flags >> 8) & 0xFF, h.regenSize, lane);
            op += h.regenSize;
        } else if (h.flags & ZL_BLK_DIRECT) {                           // already in place (literal kernel); the index kernel checked the room
            op += h.litSize;
        } else {
            const u32 litMode = (h.flags >> 4) & 3;
            const u8* lit = litMode == 0 ? d.src + h.srcOff : litArena + d.litBase + h.litOff;
            u32 cap = room, capErr = ZL_E_dstSize_tooSmall, regen = 0;
            if (cap > ZL_BLOCKSIZE_MAX) { cap = ZL_BLOCKSIZE_MAX; capErr = ZL_E_corruption_detected; }
            err = zl_exec_block<kDict>(d.dst, op, cap, capErr, h, lit, (h.flags >> 8) & 0xFF, litMode, recArena + d.recBase + h.recOff,
                                       dictContent, dictSize, hist, xtab, rcp, &execSm[threadIdx.x >> 5], lane, regen);
            op += regen;
        }
        __syncwarp();
    }
    if (!err && info.contentSize != ~0ull && info.contentSize != (u64)op) err = ZL_E_corruption_detected;      // zstd.c:41646
    if (lane == 0) {
        results[frame] = err ? (u64)0 - (u64)err : (u64)op;
        infos[frame].err = err; infos[frame].totalOut = op;
    }
}

// ---- large frames: L1 .. L4 (zl_dec_large.cuh) ------------------------------------------------------------------------
#define ZL_L_WARPS 4
__device__ __forceinline__ void zl_fill_xtab(u32* xtab, u32 tid, u32 nthreads)
{
    for (u32 i = tid; i < ZL_XTAB_WORDS; i += nthreads)
        xtab[i] = i < 36 ? (c_tables.llBase[i] | ((u32)c_tables.llBits[i] << 24)) : (c_tables.mlBase[i - 36] | ((u32)c_tables.mlBits[i - 36] << 24));
}
// grid: x strides over the blocks of the frame, y = large frame, z * ZL_L_WARPS + warp = chunk of the block
__global__ void __launch_bounds__(ZL_L_WARPS * 32)
zl_k_lblock_scan(const u32* __restrict__ largeIdx, const ZlFrameDesc* __restrict__ descs, const ZlFrameInfo* __restrict__ infos,
                 const ZlBlockHdr* __restrict__ hdrArena, const u64* __restrict__ recArena, ZlLChunk* lcArena)
{
    __shared__ u32 xtab[ZL_XTAB_WORDS];
    zl_fill_xtab(xtab, threadIdx.x, ZL_L_WARPS * 32);
    __syncthreads();
    const u32 frame = largeIdx[blockIdx.y], c = blockIdx.z * ZL_L_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const ZlFrameInfo info = infos[frame];
    if (info.err) return;
    const ZlFrameDesc d = descs[frame];
    ZlLChunk* lc = lcArena + ((d.recBase >> ZL_LCHUNK_LOG) + d.hdrBase);
    for (u32 b = blockIdx.x; b < info.nblocks; b += gridDim.x) {
        const ZlBlockHdr h = hdrArena[d.hdrBase + b];
        if ((h.flags & 3) != 2 || !h.nrec || c >= zl_lchunks(h.nrec)) continue;
        const u32 r0 = c << ZL_LCHUNK_LOG, r1 = min(h.nrec, r0 + ZL_LCHUNK_RECS);
        zl_lchunk_scan(recArena + d.recBase + h.recOff, r0, r1, xtab, lane, lc[zl_lchunk_index(h.recOff, b) + c]);
    }
}
// L2a / L2c: thread per block (x strides over the blocks of the frame, y = large frame)
__global__ void __launch_bounds__(128)
zl_k_lblock_compose(const u32* __restrict__ largeIdx, const ZlFrameDesc* __restrict__ descs, const ZlFrameInfo* __restrict__ infos,
                    const ZlBlockHdr* __restrict__ hdrArena, ZlLBlock* lbArena, ZlLChunk* lcArena, u32 spread)
{
    const u32 frame = largeIdx[blockIdx.y];
    const ZlFrameInfo info = infos[frame];
    if (info.err) return;
    const ZlFrameDesc d = descs[frame];
    ZlLChunk* lc = lcArena + ((d.recBase >> ZL_LCHUNK_LOG) + d.hdrBase);
    for (u32 b = blockIdx.x * 128 + threadIdx.x; b < info.nblocks; b += gridDim.x * 128) {
        const ZlBlockHdr h = hdrArena[d.hdrBase + b];
        ZlLChunk* C = lc + zl_lchunk_index(h.recOff, b);
        if (spread) zl_lblock_spread(h, lbArena[d.hdrBase + b], C);
        else zl_lblock_compose(h, C, lbArena[d.hdrBase + b]);
    }
}
__global__ void __launch_bounds__(32)
zl_k_lframe_prefix(const u32* __restrict__ largeIdx, const ZlFrameDesc* __restrict__ descs, ZlFrameInfo* __restrict__ infos,
                   const ZlBlockHdr* __restrict__ hdrArena, ZlLBlock* lbArena, const ZlDictDev* dict)
{
    const u32 frame = largeIdx[blockIdx.x];
    if (threadIdx.x != 0) return;
    const ZlFrameInfo info = infos[frame];
    if (info.err) return;
    const ZlFrameDesc d = descs[frame];
    u32 r0 = 1, r1 = 4, r2 = 8, total = 0;                            // zstd.c:15416
    if (dict && dict->hasEntropy) { r0 = dict->rep[0]; r1 = dict->rep[1]; r2 = dict->rep[2]; }
    const u32 err = zl_lframe_prefix(d, info, hdrArena + d.hdrBase, lbArena + d.hdrBase, r0, r1, r2, &total);
    infos[frame].err = err; infos[frame].totalOut = total;
}
template <bool kDict>
__global__ void __launch_bounds__(ZL_L_WARPS * 32)
zl_k_lblock_emit(const u32* __restrict__ largeIdx, const ZlFrameDesc* __restrict__ descs, ZlFrameInfo* __restrict__ infos,
                 const ZlBlockHdr* __restrict__ hdrArena, const u64* __restrict__ recArena, const u8* __restrict__ litArena,
                 const ZlLBlock* __restrict__ lbArena, const ZlLChunk* __restrict__ lcArena, u32* parentArena, const ZlDictDev* dict)
{
    __shared__ u32 xtab[ZL_XTAB_WORDS];
    zl_fill_xtab(xtab, threadIdx.x, ZL_L_WARPS * 32);
    __syncthreads();
    const u32 frame = largeIdx[blockIdx.y], c = blockIdx.z * ZL_L_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const ZlFrameInfo info = infos[frame];
    if (info.err) return;
    const ZlFrameDesc d = descs[frame];
    const ZlLChunk* lc = lcArena + ((d.recBase >> ZL_LCHUNK_LOG) + d.hdrBase);
    for (u32 b = blockIdx.x; b < info.nblocks; b += gridDim.x) {
        const ZlBlockHdr h = hdrArena[d.hdrBase + b];
        const bool comp = (h.flags & 3) == 2;
        const u32 nch = comp ? zl_lchunks(h.nrec) : 1u;
        if (c >= nch) continue;
        const u32 litMode = (h.flags >> 4) & 3;
        const u8* lit = litMode == 0 ? d.src + h.srcOff : litArena + d.litBase + h.litOff;
        const u32 r0 = c << ZL_LCHUNK_LOG, r1 = comp ? min(h.nrec, r0 + ZL_LCHUNK_RECS) : 0u;
        const u32 err = zl_lchunk_emit<kDict>(d.dst, parentArena + d.parBase, d, h, lbArena[d.hdrBase + b], lc[comp ? zl_lchunk_index(h.recOff, b) + c : 0u], r0, r1,
                                              c + 1 == nch, lit, recArena + d.recBase + h.recOff, kDict ? dict->content : nullptr,
                                              kDict ? dict->contentSize : 0u, xtab, lane);
        if (err && lane == 0) infos[frame].err = err;
    }
}
// one pass of pointer jumping over the bytes of the large frames; remain[pass] counts the bytes still open after it
__global__ void __launch_bounds__(256)
zl_k_ljump(const u32* __restrict__ largeIdx, const ZlFrameDesc* __restrict__ descs, const ZlFrameInfo* __restrict__ infos, u32* parentArena,
           u32* remain, u32 pass)
{
    if (pass > 1 && remain[pass - 1] == 0) return;                    // everything was final already
    const u32 frame = largeIdx[blockIdx.y];
    const ZlFrameInfo info = infos[frame];
    if (info.err) return;
    const ZlFrameDesc d = descs[frame];
    u32* parent = parentArena + d.parBase;
    u8* out = d.dst;
    u32 open = 0;
    for (u32 p = blockIdx.x * 256 + threadIdx.x; p < info.totalOut; p += gridDim.x * 256) {
        const u32 v = parent[p];
        if (v >= ZL_PAR_DONE) continue;
        const u32 pv = __ldcg(parent + v);                             // (another thread may be updating it: any value it held is valid)
        if (pv >= ZL_PAR_DONE) {
            if ((pv & 0xFFu) < pass) { out[p] = __ldcg(out + v); parent[p] = ZL_PAR_DONE | pass; }
            else open++;                                               // made final in this very pass: readable after the kernel boundary
        } else {
            // two hops per pass: chains shrink four-fold, half as many passes
            const u32 pv2 = __ldcg(parent + pv);
            if (pv2 >= ZL_PAR_DONE) {
                if ((pv2 & 0xFFu) < pass) { out[p] = __ldcg(out + pv); parent[p] = ZL_PAR_DONE | pass; }
                else { parent[p] = pv; open++; }
            } else { parent[p] = pv2; open++; }
        }
    }
    open = __reduce_add_sync(0xFFFFFFFFu, open);
    if ((threadIdx.x & 31) == 0 && open) atomicAdd(remain + pass, open);
}
__global__ void __launch_bounds__(128)
zl_k_lfinish(const u32* __restrict__ largeIdx, u32 nLarge, ZlFrameInfo* __restrict__ infos, u64* __restrict__ results, const u32* __restrict__ remain, u32 lastPass)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nLarge) return;
    const u32 frame = largeIdx[i];
    u32 err = infos[frame].err;
    if (!err && remain[lastPass] != 0) err = ZL_E_GENERIC;            // (cannot happen: ceil(log2 n) + 1 passes resolve any chain)
    infos[frame].err = err;
    results[frame] = err ? (u64)0 - (u64)err : (u64)infos[frame].totalOut;
}

// expect (optional, in launch order): a value every frame's hash must also match -- the checksums of a seek table (zl_seek.h).  A frame
// with one is hashed even when it has no trailer of its own.
static __device__ __forceinline__ bool zl_checksum_ok(const ZlFrameInfo& info, const u32* expect, u32 frame, u64 h)
{
    return (!info.checksumFlag || (u32)h == info.checksum) && (!expect || (u32)h == expect[frame]);
}
__global__ void __launch_bounds__(128)
zl_k_checksum(const ZlFrameDesc* __restrict__ descs, const ZlFrameInfo* __restrict__ infos, u64* __restrict__ results, u32 nframes,
              const u32* __restrict__ expect)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    const u32 frame = t >> 2, q = t & 3, lane = threadIdx.x & 31;
    const u32 qbase = lane & ~3u, qmask = 0xFu << qbase;
    if (frame >= nframes) return;
    const ZlFrameInfo info = infos[frame];
    if (info.err || (!info.checksumFlag && !expect)) return;
    if (descs[frame].large && !(((size_t)descs[frame].dst) & 15)) return;          // zl_k_checksum_large
    const u64 h = zl_quad_xxh64(descs[frame].dst, info.totalOut, q, qmask, qbase);
    if (q == 0 && !zl_checksum_ok(info, expect, frame, h)) results[frame] = (u64)0 - (u64)ZL_E_checksum_wrong;   // zstd.c:41650-41657
}

// large frames: a warp per frame (zl_warp_xxh64); frames whose output is not 16-byte aligned keep the quad path of zl_k_checksum
__global__ void __launch_bounds__(32)
zl_k_checksum_large(const u32* __restrict__ largeIdx, const ZlFrameDesc* __restrict__ descs, const ZlFrameInfo* __restrict__ infos, u64* __restrict__ results,
                    const u32* __restrict__ expect)
{
    __shared__ __align__(16) u8 buf[2][ZL_XXH_CHUNK];
    const u32 frame = largeIdx[blockIdx.x], lane = threadIdx.x;
    const ZlFrameInfo info = infos[frame];
    if (info.err || (!info.checksumFlag && !expect) || (((size_t)descs[frame].dst) & 15)) return;
    const u64 h = zl_warp_xxh64(descs[frame].dst, info.totalOut, buf, lane);
    if (lane == 0 && !zl_checksum_ok(info, expect, frame, h)) results[frame] = (u64)0 - (u64)ZL_E_checksum_wrong;   // zstd.c:41650-41657
}

// generic XXH64 of independent buffers (used by the compressor for frame trailers)
__global__ void __launch_bounds__(128)
zl_k_xxh64(const u8* const* __restrict__ ptrs, const u32* __restrict__ sizes, u64* __restrict__ out, u32 n)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    const u32 i = t >> 2, q = t & 3, lane = threadIdx.x & 31;
    const u32 qbase = lane & ~3u, qmask = 0xFu << qbase;
    if (i >= n) return;
    if (sizes[i] >= ZL_LARGE_FRAME_BYTES && !(((size_t)ptrs[i]) & 15)) return;       // zl_k_xxh64_large
    const u64 h = zl_quad_xxh64(ptrs[i], sizes[i], q, qmask, qbase);
    if (q == 0) out[i] = h;
}
__global__ void __launch_bounds__(32)
zl_k_xxh64_large(const u8* const* __restrict__ ptrs, const u32* __restrict__ sizes, u64* __restrict__ out, u32 n)
{
    __shared__ __align__(16) u8 buf[2][ZL_XXH_CHUNK];
    const u32 i = blockIdx.x;
    if (sizes[i] < ZL_LARGE_FRAME_BYTES || (((size_t)ptrs[i]) & 15)) return;
    const u64 h = zl_warp_xxh64(ptrs[i], sizes[i], buf, threadIdx.x);
    if (threadIdx.x == 0) out[i] = h;
}

// copy-out of zl_decompress_ranges: the pieces of the frames decoded into scratch, cut into items of <= ZL_SCATTER_BYTES, a warp each
#define ZL_SCATTER_WARPS 4
__global__ void __launch_bounds__(ZL_SCATTER_WARPS * 32)
zl_k_range_scatter(const ZlScatterItem* __restrict__ items, u32 n)
{
    const u32 i = blockIdx.x * ZL_SCATTER_WARPS + (threadIdx.x >> 5);
    if (i >= n) return;
    const ZlScatterItem it = items[i];
    zl_warp_copy(it.dst, it.src, it.bytes, threadIdx.x & 31);
}

// ---- launchers ---------------------------------------------------------------------------------------
size_t zl_literals_smem_bytes() { return ZL_QUADS_PER_WARP * sizeof(ZlLitSm) + (ZL_LIT_RING ? 32 * 16 * ZL_LIT_RING_NS : 0); }
static size_t zl_literals_smem_dict_bytes() { return zl_literals_smem_bytes() + 2048 * sizeof(u16); }      // + the dictionary's Huffman table
size_t zl_sequences_smem_bytes() { return ZL_XTAB_BYTES + ZL_SEQ_UNITS * sizeof(ZlSeqSm) + (ZL_SEQ_RING ? 16 * ZL_SEQ_RING_NS * ZL_SEQ_UNITS : 0); }

// occupancy of the two persistent entropy kernels, per device (function attributes are per device too); guarded: contexts of
// several host threads may decode for the first time at once
struct ZlDevLimits { int sms = 0, litPerSm = 0, seqPerSm = 0; };
static ZlDevLimits g_limits[64];
static std::mutex g_limitsMutex;
cudaError_t zl_decode_grid_limits(u32* litCtas, u32* seqCtas)
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> g(g_limitsMutex);
    ZlDevLimits& D = g_limits[dev];
    if (!D.sms) {
        int sms = 0, lit = 0, seq = 0;
        e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return e;
        const size_t smA = zl_literals_smem_bytes(), smB = zl_sequences_smem_bytes();
        e = cudaFuncSetAttribute(zl_k_literals, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)zl_literals_smem_dict_bytes());
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(zl_k_sequences, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smB);
        if (e != cudaSuccess) return e;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&lit, zl_k_literals, 32, smA);
        if (e != cudaSuccess) return e;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&seq, zl_k_sequences, 32, smB);
        if (e != cudaSuccess) return e;
        D.litPerSm = lit < 1 ? 1 : lit; D.seqPerSm = seq < 1 ? 1 : seq; D.sms = sms;
    }
    // (development switches: fewer resident CTAs of the shared-memory-bound entropy kernels leave room for execute CTAs beside them)
    static const int capLit = getenv("ZL_LIT_CTAS_PER_SM") ? atoi(getenv("ZL_LIT_CTAS_PER_SM")) : 0, capSeq = getenv("ZL_SEQ_CTAS_PER_SM") ? atoi(getenv("ZL_SEQ_CTAS_PER_SM")) : 0;
    const int lit = capLit > 0 && capLit < D.litPerSm ? capLit : D.litPerSm, seq = capSeq > 0 && capSeq < D.seqPerSm ? capSeq : D.seqPerSm;
    *litCtas = (u32)(D.sms * lit); *seqCtas = (u32)(D.sms * seq);
    return cudaSuccess;
}

cudaError_t zl_launch_decode(const ZlDecodeLaunch& L, cudaStream_t st)
{
    if (L.nframes == 0) return cudaSuccess;
    unsigned long long nk = 0;
    const size_t smA = L.dict ? zl_literals_smem_dict_bytes() : zl_literals_smem_bytes(), smB = zl_sequences_smem_bytes();
    u32 litCtas = 0, seqCtas = 0;
    cudaError_t e = zl_decode_grid_limits(&litCtas, &seqCtas);
    if (e != cudaSuccess) return e;
    // persistent grids: never more CTAs than fit the device at once or than there could be units (8 per CTA)
    const u32 maxCtas = (L.unitCap + ZL_QUADS_PER_WARP - 1) / ZL_QUADS_PER_WARP;
    if (litCtas > maxCtas) litCtas = maxCtas;
    const u32 maxSeqCtas = (L.unitCap + ZL_SEQ_UNITS - 1) / ZL_SEQ_UNITS;
    if (seqCtas > maxSeqCtas) seqCtas = maxSeqCtas;
    if (seqCtas > L.normSlots / ZL_SEQ_UNITS) seqCtas = L.normSlots / ZL_SEQ_UNITS;
    if (!litCtas) litCtas = 1;
    if (!seqCtas) seqCtas = 1;
    cudaEvent_t* ev = L.stageEv;
    if (ev) cudaEventRecord(ev[0], st);
    cudaMemsetAsync(L.counters, 0, 3 * sizeof(u32), st);              // unit count, literal cursor, sequence cursor
    zl_k_index<<<(L.nframes + 127) / 128, 128, 0, st>>>(L.descs, L.infos, L.hdrArena, L.units, L.counters, L.unitCap, L.nframes, L.frameBase, L.dict);
    nk++;
    const bool useSide = L.side && !ev;
    if (useSide) { cudaEventRecord(L.sideFork, st); cudaStreamWaitEvent(L.side, L.sideFork, 0); }
    zl_k_literals<<<litCtas, 32, smA, st>>>(L.descsAll, L.infosAll, L.hdrArena, L.litArena, L.units, L.counters, L.counters + 1, L.dict);
    nk++;
    if (ev) cudaEventRecord(ev[1], st);
    zl_k_sequences<<<seqCtas, 32, smB, useSide ? L.side : st>>>(L.descsAll, L.infosAll, L.hdrArena, L.recArena, L.normArena, L.units, L.counters, L.counters + 2, L.dict);
    nk++;
    if (useSide) { cudaEventRecord(L.sideJoin, L.side); cudaStreamWaitEvent(st, L.sideJoin, 0); }
    if (ev) cudaEventRecord(ev[2], st);
    const u32 g2 = (L.nframes + ZL_EXEC_WARPS - 1) / ZL_EXEC_WARPS;
    if (L.dict)
        zl_k_execute<true><<<g2, ZL_EXEC_WARPS * 32, 0, st>>>(L.descs, L.infos, L.hdrArena, L.recArena, L.litArena, L.results, L.nframes, L.dict);
    else
        zl_k_execute<false><<<g2, ZL_EXEC_WARPS * 32, 0, st>>>(L.descs, L.infos, L.hdrArena, L.recArena, L.litArena, L.results, L.nframes, nullptr);
    nk++;
    if (L.nLarge) {                                                   // block-parallel path for the large frames of this slice
        // x strides over the blocks (about one CTA per 16 KiB of content, at most one per possible block), z covers the chunks of a block
        u32 gxb = (u32)(L.largeMaxBytes >> 14) + 64;
        if (gxb > L.largeMaxBlocks) gxb = L.largeMaxBlocks;
        const dim3 gb(gxb ? gxb : 1u, L.nLarge, (ZL_LCHUNK_MAX + ZL_L_WARPS - 1) / ZL_L_WARPS);
        zl_k_lblock_scan<<<gb, ZL_L_WARPS * 32, 0, st>>>(L.largeIdx, L.descs, L.infos, L.hdrArena, L.recArena, L.lcArena);
        nk++;
        const dim3 gt((gxb + 127) / 128 ? (gxb + 127) / 128 : 1u, L.nLarge);
        zl_k_lblock_compose<<<gt, 128, 0, st>>>(L.largeIdx, L.descs, L.infos, L.hdrArena, L.lbArena, L.lcArena, 0u);
        nk++;
        zl_k_lframe_prefix<<<L.nLarge, 32, 0, st>>>(L.largeIdx, L.descs, L.infos, L.hdrArena, L.lbArena, L.dict);
        nk++;
        zl_k_lblock_compose<<<gt, 128, 0, st>>>(L.largeIdx, L.descs, L.infos, L.hdrArena, L.lbArena, L.lcArena, 1u);
        nk++;
        if (L.dict) zl_k_lblock_emit<true><<<gb, ZL_L_WARPS * 32, 0, st>>>(L.largeIdx, L.descs, L.infos, L.hdrArena, L.recArena, L.litArena, L.lbArena, L.lcArena, L.parentArena, L.dict);
        else zl_k_lblock_emit<false><<<gb, ZL_L_WARPS * 32, 0, st>>>(L.largeIdx, L.descs, L.infos, L.hdrArena, L.recArena, L.litArena, L.lbArena, L.lcArena, L.parentArena, nullptr);
        nk++;
        cudaMemsetAsync(L.remain, 0, (ZL_LJUMP_MAX_PASSES + 2) * sizeof(u32), st);
        u32 gx = (u32)((L.largeMaxBytes + 255) / 256);
        if (gx > 148u * 64u) gx = 148u * 64u;
        const dim3 gj(gx ? gx : 1u, L.nLarge);
        u32 pass = 1, lastPass = 0;
        for (;;) {
            const u32 group = pass == 1 ? 6u : 4u;                    // passes are launched in groups; the host looks at the counter in between
            for (u32 k = 0; k < group && pass <= ZL_LJUMP_MAX_PASSES; k++, pass++) {
                zl_k_ljump<<<gj, 256, 0, st>>>(L.largeIdx, L.descs, L.infos, L.parentArena, L.remain, pass);
                nk++;
            }
            lastPass = pass - 1;
            u32 open = 1;
            if (cudaMemcpyAsync(L.remainHost, L.remain + lastPass, sizeof(u32), cudaMemcpyDeviceToHost, st) != cudaSuccess) break;
            if (cudaStreamSynchronize(st) != cudaSuccess) break;
            open = *L.remainHost;
            if (!open || pass > ZL_LJUMP_MAX_PASSES) break;
        }
        zl_k_lfinish<<<(L.nLarge + 127) / 128, 128, 0, st>>>(L.largeIdx, L.nLarge, L.infos, L.results, L.remain, lastPass);
        nk++;
    }
    if (ev) cudaEventRecord(ev[3], st);
    if (L.verifyChecksum) {
        const u32 g3 = (L.nframes * 4 + 127) / 128;
        zl_k_checksum<<<g3, 128, 0, st>>>(L.descs, L.infos, L.results, L.nframes, L.expect);
        if (L.nLarge) { zl_k_checksum_large<<<L.nLarge, 32, 0, st>>>(L.largeIdx, L.descs, L.infos, L.results, L.expect); nk++; }
        nk++;
    }
    if (ev) cudaEventRecord(ev[4], st);
    if (L.launched) *L.launched += nk;
    return cudaGetLastError();
}

// Descriptors of a slice of SMALL frames, built on the device from the caller's four arrays (configs[3]: 1e5 objects of a few hundred bytes --
// the host used to spend ~10 ns per frame planning and writing 80-byte descriptors, 1.0 of a 2.0 ms call whose kernels take 0.8 ms; now
// it copies 32 bytes per frame).  raw = [src pointers | dst pointers | source sizes | capacities], cnt u64 each.  One CTA: the arena
// offsets of a frame are the exclusive prefix sums of the per-frame capacities (zl_plan_frame), four frames per thread and step.
#define ZL_BUILD_THREADS 1024
#define ZL_BUILD_PER 4
__global__ void __launch_bounds__(ZL_BUILD_THREADS)
zl_k_build_descs(const u64* __restrict__ raw, u32 cnt, ZlFrameDesc* __restrict__ descs, u64 lit0, u64 rec0, u64 hdr0, int worst)
{
    __shared__ u64 wsum[3][ZL_BUILD_THREADS / 32];
    __shared__ u64 carry[3];
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 3) carry[tid] = tid == 0 ? lit0 : (tid == 1 ? rec0 : hdr0);
    __syncthreads();
    for (u32 base = 0; base < cnt; base += ZL_BUILD_THREADS * ZL_BUILD_PER) {
        const u32 f0 = base + tid * ZL_BUILD_PER;
        u32 litCap[ZL_BUILD_PER], recCap[ZL_BUILD_PER], hdrCap[ZL_BUILD_PER], ssz[ZL_BUILD_PER], dcap[ZL_BUILD_PER];
        u64 v[3] = {0, 0, 0};
#pragma unroll
        for (int k = 0; k < ZL_BUILD_PER; k++) {
            const u32 f = f0 + k;
            ssz[k] = f < cnt ? (u32)raw[2 * (size_t)cnt + f] : 0u;
            dcap[k] = f < cnt ? (u32)raw[3 * (size_t)cnt + f] : 0u;
            zl_plan_frame(ssz[k], dcap[k], worst != 0, &litCap[k], &recCap[k], &hdrCap[k]);
            if (f < cnt) { v[0] += ((u64)litCap[k] + 15) & ~15ull; v[1] += recCap[k]; v[2] += hdrCap[k]; }
        }
        u64 inc[3];
#pragma unroll
        for (int q = 0; q < 3; q++) {
            u64 x = v[q];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const u64 y = __shfl_up_sync(ZL_FULL, x, d); if (lane >= (u32)d) x += y; }
            inc[q] = x;
            if (lane == 31) wsum[q][warp] = x;
        }
        __syncthreads();
        if (warp < 3) {                                           // warp q scans the 32 warp totals of quantity q
            u64 x = wsum[warp][lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const u64 y = __shfl_up_sync(ZL_FULL, x, d); if (lane >= (u32)d) x += y; }
            wsum[warp][lane] = x;
        }
        __syncthreads();
        u64 at[3];
#pragma unroll
        for (int q = 0; q < 3; q++) at[q] = carry[q] + (warp ? wsum[q][warp - 1] : 0ull) + inc[q] - v[q];
#pragma unroll
        for (int k = 0; k < ZL_BUILD_PER; k++) {
            const u32 f = f0 + k;
            if (f < cnt) {
                ZlFrameDesc d;
                d.src = reinterpret_cast<const u8*>(raw[f]); d.dst = reinterpret_cast<u8*>(raw[(size_t)cnt + f]);
                d.srcSize = ssz[k]; d.dstCap = dcap[k];
                d.litBase = at[0]; d.recBase = at[1]; d.hdrBase = at[2]; d.parBase = 0;
                d.litCap = litCap[k]; d.recCap = recCap[k]; d.hdrCap = hdrCap[k]; d.large = 0;
                descs[f] = d;
                at[0] += ((u64)litCap[k] + 15) & ~15ull; at[1] += recCap[k]; at[2] += hdrCap[k];
            }
        }
        __syncthreads();
        if (tid < 3) carry[tid] += wsum[tid][ZL_BUILD_THREADS / 32 - 1];
        __syncthreads();
    }
}
cudaError_t zl_launch_build_descs(const u64* raw, u32 cnt, ZlFrameDesc* descs, u64 lit0, u64 rec0, u64 hdr0, bool worst, cudaStream_t st)
{
    if (!cnt) return cudaSuccess;
    zl_k_build_descs<<<1, ZL_BUILD_THREADS, 0, st>>>(raw, cnt, descs, lit0, rec0, hdr0, worst ? 1 : 0);
    return cudaGetLastError();
}

cudaError_t zl_launch_range_scatter(const ZlScatterItem* items, u32 n, cudaStream_t st)
{
    if (!n) return cudaSuccess;
    zl_k_range_scatter<<<(n + ZL_SCATTER_WARPS - 1) / ZL_SCATTER_WARPS, ZL_SCATTER_WARPS * 32, 0, st>>>(items, n);
    return cudaGetLastError();
}

cudaError_t zl_launch_xxh64(const u8* const* ptrs, const u32* sizes, u64* out, u32 n, cudaStream_t st, bool anyLarge)
{
    if (!n) return cudaSuccess;
    zl_k_xxh64<<<(n * 4 + 127) / 128, 128, 0, st>>>(ptrs, sizes, out, n);
    if (anyLarge) zl_k_xxh64_large<<<n, 32, 0, st>>>(ptrs, sizes, out, n);
    return cudaGetLastError();
}
