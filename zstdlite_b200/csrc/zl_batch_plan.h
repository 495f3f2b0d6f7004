// zl_batch_plan.h -- host-side plan of a batched decode (zl_api.cu): slices, frame order, copy runs of host buffers, arena shares,
// descriptors and the bytes copied back from staging.  No CUDA call: tests/host/batch_plan_check.cpp checks it on the CPU.
#pragma once
#include <algorithm>
#include "zl_host.h"              // (and <vector>)
#include "zl_plan.h"

// contiguous-run staging between host buffers and a device arena
struct ZlRun { size_t first, count; const uint8_t* hbase; size_t bytes; size_t devOff; };

// frames of the slices [cut[k], cut[k + 1]) -> contiguous host ranges as copy runs that do not cross a cut, placed in the device arena at
// 256-aligned offsets; runOf[i] = the run of frame i, runCut[k] = the first run of slice k (runCut[S] = all runs); returns the arena end
static inline size_t zl_build_runs(std::vector<ZlRun>& runs, u32* runOf, size_t* runCut, const void* const* ptr, const size_t* size, const size_t* cut, size_t S)
{
    size_t off = 0;
    for (size_t k = 0; k < S; k++) {
        runCut[k] = runs.size();
        for (size_t i = cut[k]; i < cut[k + 1]; i++) {
            const u8* p = (const u8*)ptr[i];
            if (runs.size() > runCut[k] && p == runs.back().hbase + runs.back().bytes) { runs.back().bytes += size[i]; runs.back().count++; }
            else runs.push_back({i, 1, p, size[i], off});
            runOf[i] = (u32)(runs.size() - 1);
            off = (runs.back().devOff + runs.back().bytes + 255) & ~(size_t)255;
        }
    }
    runCut[S] = runs.size();
    return off;
}
// Development switches of the decode planning (DESIGN.md §3.7), read once from the environment by zl_api.cu: ZL_DEC_SLICES=n,
// ZL_DEC_GRADE=n (slice counts), ZL_DEC_NOGRADE, ZL_DEC_NODEVBUILD, ZL_DEC_NOSORT, ZL_DEC_NOMID, ZL_DEC_NOLAZY
struct ZlDecTuning { int slices = 0, grade = 6; bool noGrade = false, noDevBuild = false, noSort = false, noMid = false, noLazy = false; };
struct ZlArenaSums { u64 lit, rec, hdr, par; };      // arena offsets: literal bytes, records, block headers, parent entries
struct ZlDecPlan {
    const void* const* src; const size_t* srcSize; void* const* dst; const size_t* dstCap;      // the call's arrays
    size_t nslices = 1, nLarge = 0;
    bool dev = false, worst = false, mid = false, graded = false, devBuild = false, lazyDescs = false;
    std::vector<u32> order;              // order[pos] = caller's index of the frame at position pos; slices are ranges of positions
    std::vector<size_t> cut;             // slice k = positions [cut[k], cut[k + 1])
    std::vector<ZlArenaSums> base;       // arena offsets at every slice start; base[nslices] = the totals
    std::vector<ZlRun> sruns, druns;     // host buffers: copy runs of the sources / destinations, slice k's [srunCut[k], srunCut[k + 1])
    std::vector<size_t> srunCut, drunCut;
    std::vector<u32> srunOf, drunOf;     // the run of every frame, by caller's index
    size_t srcTotal = 0, dstTotal = 0;   // end of the runs in the dSrc / dDst arenas
};
// One frame's scratch (zl_plan_frame) placed at `s`, which advances past it.  Block-parallel execute path (zl_dec_large.cuh): frames of >= 1 MiB,
// and with `mid` (batches of a few frames, where a warp walking a frame block after block is the whole critical path) all of > 2 blocks
static inline void zl_plan_desc(ZlFrameDesc& d, u32 srcSize, u32 dstCap, bool worst, bool mid, ZlArenaSums& s)
{
    d.srcSize = srcSize; d.dstCap = dstCap;
    zl_plan_frame(srcSize, dstCap, worst, &d.litCap, &d.recCap, &d.hdrCap);
    d.litBase = s.lit; d.recBase = s.rec; d.hdrBase = s.hdr; d.parBase = s.par;
    d.large = dstCap >= ZL_LARGE_FRAME_BYTES || (mid && dstCap > 2 * ZL_BLOCKSIZE_MAX) ? 1u : 0u;
    if (d.large) s.par += ((u64)dstCap + 3) & ~3ull;
    s.lit += ((u64)d.litCap + 15) & ~15ull; s.rec += d.recCap; s.hdr += d.hdrCap;
}
// Plans a batch of n frames (dev: the buffers are in device memory; oneSlice: profiling, or no internal streams).  Returns 0 or an error.
static inline size_t zl_dec_plan(ZlDecPlan& p, const void* const* src, const size_t* srcSize, void* const* dst, const size_t* dstCap,
                                 size_t n, bool dev, bool worst, bool oneSlice, const ZlDecTuning& t)
{
    if (n > 0x7FFFFFFFull / 8) return ZL_ERROR(memory_allocation);
    u64 contentTotal = 0;
    size_t maxSrc = 1, maxDst = 0;
    for (size_t i = 0; i < n; i++) { maxSrc = std::max(maxSrc, srcSize[i]); maxDst = std::max(maxDst, dstCap[i]); contentTotal += dstCap[i]; }
    if (maxSrc > 0xFFFFFFF0ull || maxDst > 0x7FFFFFF0ull) return ZL_ERROR(memory_allocation);
    p = ZlDecPlan(); p.src = src; p.srcSize = srcSize; p.dst = dst; p.dstCap = dstCap;
    p.dev = dev; p.worst = worst; p.mid = n <= 16 && !t.noMid;
    // ---- slices: contiguous frame ranges of about equal content; one slice when profiling or when the batch is small
    size_t S = 1;
    if (!oneSlice) {
        // Host buffers: slices overlap the PCIe copies with the kernels.  Device buffers: one slice per internal stream, so that
        // the three kernels of different slices run side by side (measured on config 2: 1 slice 10.3 ms, 4 or 8 slices 8.8 ms;
        // more slices than streams only queue behind each other and pay the ~1.5 ms chain latency of a frame again).
        S = dev ? n / ZL_DEC_SLICE_DEV_FRAMES : (size_t)(contentTotal / ZL_DEC_SLICE_BYTES);
        S = std::max<size_t>(1, std::min<size_t>({S, n / ZL_DEC_SLICE_MIN_FRAMES, ZL_DEC_MAX_SLICES}));
        if (t.slices > 0) S = std::min((size_t)t.slices, n);
    }
    // Host buffers, large batches: the device-to-host copy engine bounds the call, so it must start early and never run dry:
    // the first slices are small (their kernels end after little more than the chain latency of one frame, ~3 ms) and every
    // slice is as large as all before it together (1/32, 1/32, 1/16, 1/8, 1/4, 1/2), so the copy back of a slice covers the
    // kernels of the next.  (6, 7 or 8 graded slices measured the same: 23.4 - 23.7 ms per GiB step; the floor is the chain latency
    // of ONE frame through the three kernels, 2.4 ms, before the first copy back can start, plus 1.07 GB at the D2H rate)
    p.graded = !dev && S >= 6 && !t.noGrade;
    if (p.graded) S = std::min<size_t>(std::max(t.grade, 6), ZL_DEC_MAX_SLICES);
    p.nslices = S;
    // Many SMALL frames in device memory (configs[3]: 1e5 objects of a few hundred bytes): the descriptors are built on the device from the
    // caller's four arrays (zl_k_build_descs) -- the host copies 32 bytes per frame into pinned memory instead of planning and writing an
    // 80-byte descriptor per frame (~10 ns each: 1.0 ms of a 2.0 ms call whose kernels take 0.8 ms).  Slices are cut by frame count and
    // their arena shares sized from per-slice sums (upper bounds of the per-frame roundings); the kernel places the frames inside.
    p.devBuild = dev && !t.noDevBuild && S > 1 && n >= 4096 && maxSrc <= 4096 && maxDst <= 2 * ZL_BLOCKSIZE_MAX;
    // Scheduling order (device buffers): the frames are handed to the kernels by decreasing compressed size -- longest work
    // first, and frames of one kind next to each other, so that the quads of a warp and the warps of a CTA finish together.
    // Measured on config 2 with the families interleaved: 112 -> 143 GB/s.  Host buffers keep the caller's order: their slices are
    // contiguous runs of host memory for the copies, and the end-to-end time is bound by PCIe and the chain latency of one frame, not
    // by balance (measured: sorting inside the slices 40.3 -> 39.8 GB/s).  Batches of small frames -- config 3's objects of a few
    // hundred bytes -- are not sorted: the sort and the scattered access it causes cost the host 0.5 ms per 1e5 frames, the balance
    // it buys the kernels 0.08 ms.
    p.order.resize(n);
    if (dev && !t.noSort && maxSrc > 4096) {
        // stable counting sort by decreasing size class (4,096 classes): O(n), ~50 us for 16,384 frames
        int keyShift = 0;
        while ((maxSrc >> keyShift) >= 4096) keyShift++;
        u32 cnt[4096] = {0};
        for (size_t i = 0; i < n; i++) cnt[4095 - (srcSize[i] >> keyShift)]++;
        u32 run = 0;
        for (u32& c : cnt) { const u32 k = c; c = run; run += k; }
        for (size_t i = 0; i < n; i++) p.order[cnt[4095 - (srcSize[i] >> keyShift)]++] = (u32)i;
    } else
        for (size_t i = 0; i < n; i++) p.order[i] = (u32)i;
    p.cut.assign(S + 1, n);
    if (p.devBuild) for (size_t k = 0; k <= S; k++) p.cut[k] = n * k / S;
    else {
        p.cut[0] = 0;
        u64 acc = 0; size_t k = 1;
        for (size_t i = 0; i < n && k < S; i++) {
            acc += dstCap[p.order[i]];
            // graded: slice 0 and 1 take 1/2^(S-1) of the batch each, every later slice as much as all before it together
            const bool reached = p.graded ? (acc << (S - 1)) >= contentTotal * ((u64)1 << (k - 1)) : acc * S >= contentTotal * k;
            if (reached) p.cut[k++] = i + 1;
        }
    }
    p.srunCut.assign(S + 1, 0); p.drunCut.assign(S + 1, 0);
    if (!dev) {
        p.srunOf.resize(n); p.drunOf.resize(n);
        p.srcTotal = zl_build_runs(p.sruns, p.srunOf.data(), p.srunCut.data(), src, srcSize, p.cut.data(), S);
        p.dstTotal = zl_build_runs(p.druns, p.drunOf.data(), p.drunCut.data(), (const void* const*)dst, dstCap, p.cut.data(), S);
    }
    // ---- arena shares: the offsets at every slice start, and the totals
    p.base.resize(S + 1);
    ZlArenaSums s = {0, 0, 0, 0};
    if (p.devBuild) {
        for (size_t k = 0; k < S; k++) {
            p.base[k] = s;
            u64 sumSrc = 0, sumDst = 0;
            for (size_t i = p.cut[k]; i < p.cut[k + 1]; i++) { sumSrc += srcSize[i]; sumDst += dstCap[i]; }
            unsigned long long bl, br, bh;                                     // >= the sums of the frames' litCap (16-aligned), recCap (even) and hdrCap
            zl_plan_slice_bound(sumSrc, sumDst, p.cut[k + 1] - p.cut[k], worst, &bl, &br, &bh);
            s.hdr += bh; s.rec += br; s.lit += bl;
        }
        p.base[S] = s;
    } else {
        size_t k = 0;
        for (size_t pos = 0; pos < n; pos++) {
            while (k < S && pos == p.cut[k]) p.base[k++] = s;
            const size_t i = p.order[pos];
            ZlFrameDesc d;
            zl_plan_desc(d, (u32)srcSize[i], (u32)dstCap[i], worst, p.mid, s);
            p.nLarge += d.large;
        }
        while (k <= S) p.base[k++] = s;
    }
    // Descriptors of a slice are written right before the slice is launched, so that the device starts after 1/8 of the host work and
    // the rest of it hides behind the kernels (config 3's 1e5 small frames: 8 MB of descriptors, 1.0 of 2.4 ms spent before the first
    // launch).  Batches with large frames (their index is uploaded up front) write everything first.
    p.lazyDescs = p.nLarge == 0 && S > 1 && !t.noLazy && !p.devBuild;
    return 0;
}
// Descriptors of positions [a, b) into hd[a, b), their arenas placed from `s` on; the frames' device addresses are the caller's pointers
// (device batches) or their places in the dSrc / dDst arenas (host batches)
static inline void zl_plan_fill_descs(const ZlDecPlan& p, size_t a, size_t b, ZlArenaSums s, const u8* dSrc, u8* dDst, ZlFrameDesc* hd)
{
    for (size_t pos = a; pos < b; pos++) {
        const size_t i = p.order[pos];
        ZlFrameDesc& d = hd[pos];
        if (p.dev) { d.src = (const u8*)p.src[i]; d.dst = (u8*)p.dst[i]; }
        else {
            const ZlRun& rs = p.sruns[p.srunOf[i]]; const ZlRun& rd = p.druns[p.drunOf[i]];
            d.src = dSrc + rs.devOff + ((const u8*)p.src[i] - rs.hbase);
            d.dst = dDst + rd.devOff + ((const u8*)p.dst[i] - rd.hbase);
        }
        zl_plan_desc(d, (u32)p.srcSize[i], (u32)p.dstCap[i], p.worst, p.mid, s);
    }
}
// Copies from slice k's staged output (`staged`, laid out like the dDst arena) back to the caller's buffers: what each frame produced
// (results[i], at most its capacity), nothing of a failed frame; frames that filled their slot merge into one copy
static inline void zl_plan_unstage(const ZlDecPlan& p, size_t k, const u64* results, const u8* staged, std::vector<ZlCopySeg>& segs)
{
    segs.clear();
    for (size_t r = p.drunCut[k]; r < p.drunCut[k + 1]; r++) {
        const ZlRun& run = p.druns[r];
        size_t off = 0, segBeg = 0, segLen = 0;                      // the open copy [segBeg, segBeg + segLen) of the run
        auto close = [&]() { if (segLen) segs.push_back({(u8*)run.hbase + segBeg, staged + run.devOff + segBeg, segLen}); segLen = 0; };
        for (size_t i = run.first; i < run.first + run.count; i++) {
            const size_t got = (size_t)results[i], cap = p.dstCap[i], take = zl_is_error(got) ? 0 : std::min(got, cap);
            if (segBeg + segLen != off) { close(); segBeg = off; }
            segLen += take;
            if (take != cap) close();
            off += cap;
        }
        close();
    }
}
