// Test infrastructure: checks the host-side plan of a batched decode (zstdlite_b200/csrc/zl_batch_plan.h) on the CPU -- the exact plans of
// the benchmark's batch shapes and of every development switch, then properties of slices, descriptors, copy runs and unstaging copies over
// seeded random batches.  Built and run by tests/test_batch_plan.py; no CUDA call is made.  The plan only does arithmetic on the buffer
// addresses, so the batches use made-up addresses.
#include "zl_batch_plan.h"
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <vector>

static int bad = 0;
#define CHECK(c) do { if (!(c)) { if (bad++ < 20) printf("FAIL line %d: %s\n", __LINE__, #c); } } while (0)

static unsigned long long rngState = 88172645463325252ull;
static unsigned long long rnd() { rngState ^= rngState << 13; rngState ^= rngState >> 7; rngState ^= rngState << 17; return rngState; }
static size_t rndIn(size_t lo, size_t hi) { return lo + (size_t)(rnd() % (hi - lo + 1)); }

struct Batch {
    std::vector<const void*> src; std::vector<void*> dst; std::vector<size_t> srcSize, dstCap;
    size_t n() const { return src.size(); }
};
// frames back to back in host (or device) memory; brk[i]: frame i starts a new range (a gap before it, in source and destination)
static Batch layout(const std::vector<size_t>& ssz, const std::vector<size_t>& dcap, const std::vector<bool>& brk)
{
    Batch b; b.srcSize = ssz; b.dstCap = dcap;
    uintptr_t s = (uintptr_t)1 << 40, d = (uintptr_t)3 << 40;
    for (size_t i = 0; i < ssz.size(); i++) {
        if (brk[i]) { s += 1 + rnd() % 4096; d += 1 + rnd() % 4096; }
        b.src.push_back((const void*)s); b.dst.push_back((void*)d);
        s += ssz[i]; d += dcap[i];
    }
    return b;
}
static ZlDecPlan plan(const Batch& b, bool dev, const ZlDecTuning& t = ZlDecTuning(), bool oneSlice = false, bool worst = false)
{
    ZlDecPlan p;
    CHECK(zl_dec_plan(p, b.src.data(), b.srcSize.data(), b.dst.data(), b.dstCap.data(), b.n(), dev, worst, oneSlice, t) == 0);
    return p;
}
static std::vector<size_t> sliceSizes(const ZlDecPlan& p)
{
    std::vector<size_t> s;
    for (size_t k = 0; k < p.nslices; k++) s.push_back(p.cut[k + 1] - p.cut[k]);
    return s;
}
static bool identity(const ZlDecPlan& p)
{
    for (size_t i = 0; i < p.order.size(); i++) if (p.order[i] != i) return false;
    return true;
}
// order is a permutation; with `sorted`, by decreasing size class (the counting sort's key) and stable
static void checkOrder(const Batch& b, const ZlDecPlan& p, bool sorted)
{
    const size_t n = b.n();
    std::vector<bool> seen(n, false);
    for (size_t pos = 0; pos < n; pos++) { CHECK(p.order[pos] < n && !seen[p.order[pos]]); if (p.order[pos] < n) seen[p.order[pos]] = true; }
    if (!sorted) { CHECK(identity(p)); return; }
    size_t maxSrc = 1;
    for (size_t s : b.srcSize) maxSrc = std::max(maxSrc, s);
    int shift = 0;
    while ((maxSrc >> shift) >= 4096) shift++;
    for (size_t pos = 1; pos < n; pos++) {
        const size_t c0 = b.srcSize[p.order[pos - 1]] >> shift, c1 = b.srcSize[p.order[pos]] >> shift;
        CHECK(c0 > c1 || (c0 == c1 && p.order[pos - 1] < p.order[pos]));
    }
}

// ---- exact plans of the benchmark's shapes and of the development switches
static void exactPlans()
{
    // 16,384 frames of 64 KiB content, compressed to 20 - 40 KB, back to back in one buffer
    std::vector<size_t> ssz(16384), dcap(16384, 65536);
    for (size_t& s : ssz) s = rndIn(20000, 40000);
    const Batch big = layout(ssz, dcap, std::vector<bool>(16384, false));
    const ZlDecPlan host = plan(big, false);
    CHECK(host.nslices == 6 && host.graded && !host.devBuild && host.lazyDescs && host.nLarge == 0);
    CHECK(sliceSizes(host) == (std::vector<size_t>{512, 512, 1024, 2048, 4096, 8192}));
    checkOrder(big, host, false);
    CHECK(host.sruns.size() == 6 && host.druns.size() == 6);                 // one run per slice: the frames are contiguous
    const ZlDecPlan dev = plan(big, true);
    CHECK(dev.nslices == 8 && !dev.graded && !dev.devBuild && dev.lazyDescs && dev.sruns.empty());
    CHECK(sliceSizes(dev) == std::vector<size_t>(8, 2048));
    checkOrder(big, dev, true);
    // 1e5 small frames in device memory
    std::vector<size_t> sss(100000), sdc(100000);
    for (size_t i = 0; i < sss.size(); i++) { sss[i] = rndIn(40, 4096); sdc[i] = rndIn(100, 4096); }
    const Batch small = layout(sss, sdc, std::vector<bool>(100000, true));
    const ZlDecPlan dsmall = plan(small, true);
    CHECK(dsmall.nslices == 8 && dsmall.devBuild && !dsmall.lazyDescs && dsmall.nLarge == 0);
    for (size_t k = 0; k <= 8; k++) CHECK(dsmall.cut[k] == 100000 * k / 8);
    checkOrder(small, dsmall, false);

    // every switch changes what it names and nothing else
    ZlDecTuning t;
    t.slices = 3;
    ZlDecPlan q = plan(big, false, t);
    CHECK(q.nslices == 3 && !q.graded && q.lazyDescs && identity(q));
    for (size_t k = 0; k <= 3; k++) CHECK(q.cut[k] == (16384 * k + 2) / 3);                   // equal content: the first frame that reaches k/3
    t = ZlDecTuning(); t.noGrade = true;
    q = plan(big, false, t);
    CHECK(q.nslices == 8 && !q.graded && q.lazyDescs && identity(q) && sliceSizes(q) == std::vector<size_t>(8, 2048));
    t = ZlDecTuning(); t.grade = 8;
    q = plan(big, false, t);
    CHECK(q.nslices == 8 && q.graded && sliceSizes(q) == (std::vector<size_t>{128, 128, 256, 512, 1024, 2048, 4096, 8192}));
    t = ZlDecTuning(); t.noSort = true;
    q = plan(big, true, t);
    CHECK(q.nslices == dev.nslices && q.cut == dev.cut && q.lazyDescs && !q.devBuild && identity(q));
    t = ZlDecTuning(); t.noLazy = true;
    q = plan(big, true, t);
    CHECK(q.nslices == dev.nslices && q.cut == dev.cut && q.order == dev.order && !q.lazyDescs);
    t = ZlDecTuning(); t.noDevBuild = true;
    q = plan(small, true, t);
    CHECK(q.nslices == 8 && !q.devBuild && identity(q));
    // batches of a few frames: those of more than two blocks take the block-parallel path, unless ZL_DEC_NOMID (>= 1 MiB only)
    std::vector<size_t> fsz(8, 100000), fdc(8, 512u << 10);
    fdc[3] = 2u << 20;
    const Batch few = layout(fsz, fdc, std::vector<bool>(8, true));
    CHECK(plan(few, true).nLarge == 8 && plan(few, false).nLarge == 8);
    t = ZlDecTuning(); t.noMid = true;
    q = plan(few, true, t);
    CHECK(q.nLarge == 1 && q.nslices == 1 && !q.lazyDescs);
    // profiling (or no internal streams): one slice
    q = plan(big, false, ZlDecTuning(), true);
    CHECK(q.nslices == 1 && !q.graded && q.cut == (std::vector<size_t>{0, 16384}) && q.sruns.size() == 1);
    q = plan(small, true, ZlDecTuning(), true);
    CHECK(q.nslices == 1 && !q.devBuild);
}

// ---- properties over random batches
struct Span { u64 at, len; };
// the spans tile [0, total): sorted by start, each starts where the one before ends
static bool tiles(std::vector<Span> v, u64 total)
{
    std::sort(v.begin(), v.end(), [](const Span& x, const Span& y) { return x.at != y.at ? x.at < y.at : x.len < y.len; });
    u64 end = 0;
    for (const Span& s : v) { if (s.at != end) return false; end += s.len; }
    return end == total;
}
static void checkRuns(const ZlDecPlan& p, const std::vector<ZlRun>& runs, const std::vector<size_t>& runCut, const void* const* ptr,
                      const size_t* size, size_t total)
{
    const size_t S = p.nslices;
    CHECK(runCut[0] == 0 && runCut[S] == runs.size());
    size_t next = 0;                                                  // the runs cover the frames in order
    for (size_t k = 0; k < S; k++)
        for (size_t r = runCut[k]; r < runCut[k + 1]; r++) {
            const ZlRun& run = runs[r];
            CHECK(run.first == next && run.count > 0 && run.first >= p.cut[k] && run.first + run.count <= p.cut[k + 1]);
            CHECK(run.devOff % 256 == 0 && run.devOff + run.bytes <= total);
            if (r > 0) CHECK(run.devOff >= runs[r - 1].devOff + runs[r - 1].bytes);
            if (r > runCut[k]) CHECK(run.hbase != runs[r - 1].hbase + runs[r - 1].bytes);          // maximal inside a slice
            size_t off = 0;
            for (size_t i = run.first; i < run.first + run.count; i++) { CHECK((const u8*)ptr[i] == run.hbase + off); off += size[i]; }
            CHECK(off == run.bytes);
            next = run.first + run.count;
        }
    CHECK(next == p.cut[S]);
}
static void randomPlans()
{
    const uintptr_t dSrcBase = (uintptr_t)5 << 40, dDstBase = (uintptr_t)7 << 40;
    for (int trial = 0; trial < 400; trial++) {
        const int shape = trial % 4;              // 0: small frames, 1: mixed, 2: a few large frames, 3: many frames of 64 KiB
        const size_t n = shape == 2 ? rndIn(1, 24) : (shape == 0 ? rndIn(1, 12000) : rndIn(1, 6000));
        const size_t smax = shape == 0 ? 4096 : (shape == 2 ? 3000000 : 70000), dmax = shape == 0 ? 4096 : (shape == 2 ? 4u << 20 : 300000);
        std::vector<size_t> ssz(n), dcap(n);
        std::vector<bool> brk(n);
        const unsigned brkPct = (unsigned)(rnd() % 101);
        for (size_t i = 0; i < n; i++) {
            ssz[i] = shape == 3 ? rndIn(30000, 50000) : rndIn(rnd() % 8 ? 1 : 0, smax);
            dcap[i] = shape == 3 ? 65536 : rndIn(0, dmax);
            brk[i] = rnd() % 100 < brkPct;
        }
        const Batch b = layout(ssz, dcap, brk);
        const bool dev = rnd() & 1, worst = rnd() % 4 == 0, oneSlice = rnd() % 8 == 0;
        ZlDecTuning t;
        if (rnd() % 4 == 0) t.slices = (int)rndIn(1, 12);
        if (rnd() % 4 == 0) t.grade = (int)rndIn(0, 10);
        t.noGrade = rnd() % 5 == 0; t.noDevBuild = rnd() % 5 == 0; t.noSort = rnd() % 5 == 0; t.noMid = rnd() % 5 == 0; t.noLazy = rnd() % 5 == 0;
        const ZlDecPlan p = plan(b, dev, t, oneSlice, worst);
        const size_t S = p.nslices;
        // slices
        CHECK(S >= 1 && p.cut.size() == S + 1 && p.cut[0] == 0 && p.cut[S] == n);
        for (size_t k = 0; k < S; k++) CHECK(p.cut[k] <= p.cut[k + 1]);
        CHECK(!oneSlice || S == 1);
        CHECK(!p.devBuild || dev);
        CHECK(!p.lazyDescs || (S > 1 && !p.devBuild && p.nLarge == 0));
        checkOrder(b, p, dev && !t.noSort && *std::max_element(ssz.begin(), ssz.end()) > 4096);
        CHECK(p.base.size() == S + 1);
        // descriptors written slice by slice (as the launch loop does) tile the four arenas and end at the totals; the same as all at once
        std::vector<ZlFrameDesc> hd(n), all(n);
        const u8* dSrc = (const u8*)dSrcBase; u8* dDst = (u8*)dDstBase;
        for (size_t k = 0; k < S; k++) zl_plan_fill_descs(p, p.cut[k], p.cut[k + 1], p.base[k], dSrc, dDst, hd.data());
        if (!p.devBuild) {
            zl_plan_fill_descs(p, 0, n, p.base[0], dSrc, dDst, all.data());
            CHECK(memcmp(hd.data(), all.data(), n * sizeof(ZlFrameDesc)) == 0);
            std::vector<Span> lit, rec, hdr, par;
            size_t large = 0;
            for (size_t pos = 0; pos < n; pos++) {
                const ZlFrameDesc& d = hd[pos];
                u32 lc, rc, hc;
                zl_plan_frame((u32)ssz[p.order[pos]], (u32)dcap[p.order[pos]], worst, &lc, &rc, &hc);
                CHECK(d.srcSize == ssz[p.order[pos]] && d.dstCap == dcap[p.order[pos]] && d.litCap == lc && d.recCap == rc && d.hdrCap == hc);
                lit.push_back({d.litBase, ((u64)d.litCap + 15) & ~15ull}); rec.push_back({d.recBase, d.recCap}); hdr.push_back({d.hdrBase, d.hdrCap});
                if (d.large) { par.push_back({d.parBase, ((u64)d.dstCap + 3) & ~3ull}); large++; }
                CHECK(d.large == (d.dstCap >= ZL_LARGE_FRAME_BYTES || (n <= 16 && !t.noMid && d.dstCap > 2 * ZL_BLOCKSIZE_MAX)));
            }
            CHECK(large == p.nLarge);
            const ZlArenaSums& tot = p.base[S];
            CHECK(tiles(lit, tot.lit) && tiles(rec, tot.rec) && tiles(hdr, tot.hdr) && tiles(par, tot.par));
            for (size_t k = 0; k < S; k++) if (p.cut[k] < n) CHECK(hd[p.cut[k]].litBase == p.base[k].lit && hd[p.cut[k]].hdrBase == p.base[k].hdr);
        } else
            // the device builds these descriptors from the slice bases: the per-frame sums of a slice stay inside its share
            for (size_t k = 0; k < S; k++) {
                const size_t e = p.cut[k + 1] - 1;
                const ZlArenaSums& b0 = p.base[k], &b1 = p.base[k + 1];
                CHECK(b0.lit % 16 == 0 && b0.rec % 2 == 0 && b1.lit >= b0.lit && b1.rec >= b0.rec && b1.hdr >= b0.hdr && b1.par == 0);
                if (p.cut[k + 1] > p.cut[k])
                    CHECK(hd[e].litBase + ((hd[e].litCap + 15) & ~15ull) <= b1.lit && hd[e].recBase + hd[e].recCap <= b1.rec && hd[e].hdrBase + hd[e].hdrCap <= b1.hdr);
            }
        if (dev) {
            for (size_t pos = 0; pos < n; pos++) CHECK(hd[pos].src == b.src[p.order[pos]] && hd[pos].dst == b.dst[p.order[pos]]);
            CHECK(p.sruns.empty() && p.druns.empty());
            continue;
        }
        // host buffers: copy runs, and every frame's device address inside its run
        checkRuns(p, p.sruns, p.srunCut, b.src.data(), b.srcSize.data(), p.srcTotal);
        checkRuns(p, p.druns, p.drunCut, (const void* const*)b.dst.data(), b.dstCap.data(), p.dstTotal);
        for (size_t pos = 0; pos < n; pos++) {
            const size_t i = p.order[pos];
            const ZlRun& rs = p.sruns[p.srunOf[i]]; const ZlRun& rd = p.druns[p.drunOf[i]];
            CHECK(i >= rs.first && i < rs.first + rs.count && i >= rd.first && i < rd.first + rd.count);
            CHECK(hd[pos].src >= dSrc + rs.devOff && hd[pos].src + ssz[i] <= dSrc + rs.devOff + rs.bytes);
            CHECK(hd[pos].dst >= dDst + rd.devOff && hd[pos].dst + dcap[i] <= dDst + rd.devOff + rd.bytes);
            CHECK(hd[pos].src - (dSrc + rs.devOff) == (const u8*)b.src[i] - rs.hbase && hd[pos].dst - (dDst + rd.devOff) == (u8*)b.dst[i] - rd.hbase);
        }
        // unstaging: exactly min(result, dstCap) bytes of every successful frame, from its place in the staged arena to its buffer,
        // nothing of a failed one; copies never touch each other (adjacent full frames are one copy)
        std::vector<u64> res(n);
        for (size_t i = 0; i < n; i++) {
            const unsigned kind = (unsigned)(rnd() % 6);
            res[i] = kind == 0 ? (u64)ZL_ERROR(corruption_detected) : kind == 1 ? (u64)rndIn(0, dcap[i]) : kind == 2 ? (u64)dcap[i] + rndIn(0, 100) : (u64)dcap[i];
        }
        const u8* staged = (const u8*)((uintptr_t)9 << 40);
        std::vector<ZlCopySeg> segs;
        for (size_t k = 0; k < S; k++) {
            zl_plan_unstage(p, k, res.data(), staged, segs);
            std::vector<Span> want, got;
            u64 wantBytes = 0, gotBytes = 0;
            for (size_t i = p.cut[k]; i < p.cut[k + 1]; i++) {
                const u64 take = zl_is_error((size_t)res[i]) ? 0 : std::min<u64>(res[i], dcap[i]);
                if (take) want.push_back({(u64)(uintptr_t)b.dst[i], take});
                wantBytes += take;
            }
            for (const ZlCopySeg& s : segs) {
                CHECK(s.bytes > 0);
                got.push_back({(u64)(uintptr_t)s.dst, s.bytes});
                gotBytes += s.bytes;
                bool placed = false;                     // the source is the destination's place in the staged copy of its run
                for (size_t r = p.drunCut[k]; r < p.drunCut[k + 1]; r++) {
                    const ZlRun& run = p.druns[r];
                    if ((const u8*)s.dst >= run.hbase && (const u8*)s.dst + s.bytes <= run.hbase + run.bytes)
                        placed = (const u8*)s.src == staged + run.devOff + ((const u8*)s.dst - run.hbase);
                }
                CHECK(placed);
            }
            CHECK(gotBytes == wantBytes);
            std::sort(got.begin(), got.end(), [](const Span& x, const Span& y) { return x.at < y.at; });
            for (size_t j = 1; j < got.size(); j++) CHECK(got[j - 1].at + got[j - 1].len < got[j].at);
            for (const Span& w : want) {                 // inside one copy (with the byte count equal, nothing else is copied)
                auto it = std::upper_bound(got.begin(), got.end(), w.at, [](u64 v, const Span& s) { return v < s.at; });
                CHECK(it != got.begin() && w.at + w.len <= (it - 1)->at + (it - 1)->len);
            }
        }
    }
}

int main()
{
    exactPlans();
    randomPlans();
    printf("bad=%d\n", bad);
    return bad ? 1 : 0;
}
