// Test infrastructure: checks the host-side plan of a compress batch (zstdlite_b200/csrc/zl_enc_plan.h) on the CPU -- the exact plans of
// the benchmark's shapes and of every development switch, then properties of waves, parts, descriptors, far tables, host placement, gather
// tables and split frames over seeded random batches.  Built and run by tests/test_enc_plan.py; no CUDA call is made.  The plan only does
// arithmetic on the buffer addresses, so the batches use made-up addresses.
#include "zl_enc_plan.h"
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
static const size_t KiB = 1024, MiB = KiB * KiB, GiB = MiB * KiB;

// a batch of frames in device memory: sources back to back from 1 << 40, destination slots from 3 << 40
struct Batch {
    std::vector<const u8*> src; std::vector<u8*> dst; std::vector<size_t> srcSize, dstCap;
    explicit Batch(const std::vector<size_t>& sizes) : srcSize(sizes)
    {
        uintptr_t s = (uintptr_t)1 << 40, d = (uintptr_t)3 << 40;
        for (size_t n : sizes) { src.push_back((const u8*)s); dst.push_back((u8*)d); dstCap.push_back(n + 64); s += n + 16; d += n + 64; }
    }
    size_t n() const { return srcSize.size(); }
};
static std::vector<size_t> waveCuts(const Batch& b)
{
    size_t wb = 0;
    CHECK(zl_enc_wave_blocks(b.srcSize.data(), b.n(), &wb) == 0);
    std::vector<size_t> cut{0};
    while (cut.back() < b.n()) cut.push_back(zl_enc_wave_end(b.srcSize.data(), b.n(), cut.back(), wb));
    return cut;
}
static ZlEncWave layout(const Batch& b, size_t f0, size_t f1, bool stats = false, const ZlEncParams& P = zl_enc_params(3),
                        const ZlEncTuning& t = ZlEncTuning())
{
    ZlEncWave w;
    CHECK(zl_enc_wave_layout(w, b.src.data(), b.srcSize.data(), b.dst.data(), b.dstCap.data(), f0, f1, stats, P, t) == 0);
    return w;
}
// descriptors of a whole wave, part by part as the launch loop writes them
struct Descs { std::vector<ZlEncFrame> f; std::vector<ZlEncBlock> b; std::vector<const u8*> hp; std::vector<u32> hs; std::vector<ZlEncPart> parts; };
static Descs fill(ZlEncWave& w, u32 dictID, u32 checksum)
{
    Descs d;
    d.f.resize(w.nf); d.b.resize(w.nb); d.hp.resize(w.nf); d.hs.resize(w.nf);
    for (size_t p = 0; p < w.parts; p++)
        d.parts.push_back(zl_enc_fill_part(w, p, dictID, checksum, d.f.data(), d.b.data(), checksum ? d.hp.data() : nullptr, checksum ? d.hs.data() : nullptr));
    return d;
}
static std::vector<size_t> chunkSizes(const ZlSplitPlan& p)
{
    std::vector<size_t> s;
    for (size_t k = 0; k + 1 < p.cstart.size(); k++) s.push_back(p.cstart[k + 1] - p.cstart[k]);
    return s;
}

// ---- exact plans of the benchmark's shapes and of the development switches
static void exactPlans()
{
    // configs[2]: 32,768 frames of 128 KiB in device memory
    const Batch big(std::vector<size_t>(32768, 128 * KiB));
    CHECK(waveCuts(big) == (std::vector<size_t>{0, 8192, 16384, 24576, 32768}));
    ZlEncWave w = layout(big, 8192, 16384);
    CHECK(w.nf == 8192 && w.nb == 8192 && w.parts == 1 && w.maxBlock == 128 * KiB && w.S == 131072);
    CHECK(w.slotM == 131072 && w.slotRec == 26246 && w.slotLit == 131088 && w.streamCapWords == 11269 && w.streamWordsPerBlock == 4 * 11269 && w.seqCapWords == 32768);
    Descs d = fill(w, 0, 0);
    CHECK(d.parts.size() == 1 && d.parts[0].nb == 8192 && d.parts[0].nSmall == 0 && w.farEntries == 0);

    // the dictionary leg: 1e5 objects of 200 - 1,000 bytes in device memory, one wave in four parts
    std::vector<size_t> objs(100000);
    for (size_t& s : objs) s = rndIn(200, 1000);
    objs[777] = 1000;
    const Batch small(objs);
    CHECK(waveCuts(small) == (std::vector<size_t>{0, 100000}));
    w = layout(small, 0, 100000);
    CHECK(w.parts == 4 && w.S == 1024 && w.nb == 100000);
    for (size_t p = 0; p <= 4; p++) CHECK(w.partCut[p] == 100000 * p / 4);
    d = fill(w, 0, 0);
    CHECK(w.farEntries == 0 && d.parts[0].nSmall == 25000 && d.parts[3].b0 == 75000);
    for (const ZlEncFrame& f : d.f) CHECK(f.pad == 0);
    CHECK(layout(small, 0, 100000, true).parts == 1);                                  // statistics mode
    ZlEncTuning t;
    t.parts = 1;
    CHECK(layout(small, 0, 100000, false, zl_enc_params(3), t).parts == 1);

    // zl_compress_split: 4 GiB on the host as 128 KiB frames is pipelined with growing chunks; in device memory it is not
    ZlSplitPlan sp = zl_enc_split_plan(4 * GiB, 128 * KiB, false);
    CHECK(sp.pipelined && sp.nf == 32768 && sp.chunkFrames == 8192);
    CHECK(chunkSizes(sp) == (std::vector<size_t>{1024, 2048, 4096, 8192, 8192, 8192, 1024}));
    sp = zl_enc_split_plan(4 * GiB, 128 * KiB, true);
    CHECK(!sp.pipelined && sp.nf == 32768 && sp.cstart.empty());
    sp = zl_enc_split_plan(17001 * 16 * KiB, 16 * KiB, false);
    CHECK(sp.pipelined && chunkSizes(sp) == (std::vector<size_t>{1024, 2048, 4096, 8192, 1641}));
    CHECK(!zl_enc_split_plan(64 * MiB, 128 * KiB, false).pipelined);                    // one chunk

    // one 256 MiB frame: one wave of 2,048 blocks with a far table; none with windowLog 17 or ZL_ENC_NOFAR
    const Batch one(std::vector<size_t>{256 * MiB});
    CHECK(waveCuts(one) == (std::vector<size_t>{0, 1}));
    w = layout(one, 0, 1);
    d = fill(w, 0, 0);
    CHECK(w.nb == 2048 && w.farEntries == zl_far_entries(256 * MiB) && d.f[0].pad == ((u64)zl_far_log(256 * MiB) << 56));
    ZlEncParams P = zl_enc_params(3);
    zl_enc_tune_params(P, false, 17, ZlEncTuning());
    w = layout(one, 0, 1, false, P);
    d = fill(w, 0, 0);
    CHECK(w.farEntries == 0 && d.f[0].pad == 0);
    t = ZlEncTuning(); t.noFar = true;
    w = layout(one, 0, 1, false, zl_enc_params(3), t);
    d = fill(w, 0, 0);
    CHECK(w.farEntries == 0 && d.f[0].pad == 0 && w.nb == 2048);

    // a 2 GiB frame (16,384 blocks) among 128 KiB frames forms a wave of its own; its far tables would exceed the budget
    std::vector<size_t> mixed(20, 128 * KiB);
    mixed[10] = 2 * GiB;
    const Batch mix(mixed);
    CHECK(waveCuts(mix) == (std::vector<size_t>{0, 10, 11, 20}));
    w = layout(mix, 10, 11);
    d = fill(w, 0, 0);
    CHECK(w.nb == 16384 && w.farEntries == 0 && d.f[0].pad == 0);

    // an input of >= 0xFFFFFFF0 bytes is refused; more than 0x3FFFFFFF blocks in a wave cannot be reserved
    const std::vector<size_t> huge{100, 0xFFFFFFF0ull};
    size_t wb = 0;
    CHECK(zl_enc_wave_blocks(huge.data(), 2, &wb) == ZL_ERROR(srcSize_wrong));
    const std::vector<size_t> many(0x40000000ull / 8192 + 1, 0xFFFFFFEFull);
    std::vector<const u8*> nsrc(many.size()); std::vector<u8*> ndst(many.size());
    ZlEncWave wm;
    CHECK(zl_enc_wave_layout(wm, nsrc.data(), many.data(), ndst.data(), many.data(), 0, many.size(), false, zl_enc_params(3), ZlEncTuning()) == ZL_ERROR(memory_allocation));

    // every switch changes what it names and nothing else
    ZlEncParams base = zl_enc_params(3), q = base;
    zl_enc_tune_params(q, false, 0, ZlEncTuning());
    CHECK(memcmp(&q, &base, sizeof(q)) == 0);
    t = ZlEncTuning(); t.hlog = true; t.hlogS = 16; t.hlogL = 17;
    zl_enc_tune_params(q, false, 0, t);
    CHECK(q.hlogS == 16 && q.hlogL == 17 && q.level == base.level && q.mls == base.mls && q.farMaxOff == base.farMaxOff);
    q = base; zl_enc_tune_params(q, true, 0, t);                                        // not with a dictionary
    CHECK(memcmp(&q, &base, sizeof(q)) == 0);
    q = zl_enc_params(1); zl_enc_tune_params(q, false, 0, t);                           // level 1 has no long table
    CHECK(q.hlogS == 16 && q.hlogL == 0);
    for (int wl : {18, 20, 23}) { q = base; zl_enc_tune_params(q, false, wl, ZlEncTuning()); CHECK(q.farMaxOff == (1u << wl) && q.hlogS == base.hlogS); }
    q = base; zl_enc_tune_params(q, false, 27, ZlEncTuning());
    CHECK(q.farMaxOff == ZL_FAR_MAX_OFF);
    t = ZlEncTuning(); t.parts = 2;
    ZlEncWave w2 = layout(small, 0, 100000, false, zl_enc_params(3), t), w4 = layout(small, 0, 100000);
    CHECK(w2.parts == 2 && w2.partCut[1] == 50000 && w2.S == w4.S && w2.nb == w4.nb && w2.farMaxOff == w4.farMaxOff);
    t.parts = 9;
    CHECK(layout(small, 0, 100000, false, zl_enc_params(3), t).parts == 4);
    t = ZlEncTuning(); t.noFar = true;
    w2 = layout(big, 0, 8192, false, zl_enc_params(3), t); w4 = layout(big, 0, 8192);
    CHECK(w2.farMaxOff == 0 && w4.farMaxOff == ZL_FAR_MAX_OFF && w2.parts == w4.parts && w2.S == w4.S && w2.nb == w4.nb);
    t = ZlEncTuning();
    CHECK(zl_enc_side(t, 8192) && zl_enc_side(t, 1));
    t.side = 1;
    CHECK(zl_enc_side(t, 1024) && !zl_enc_side(t, 1025));
    t.side = 0;
    CHECK(!zl_enc_side(t, 1));
}

// ---- properties over random batches
struct Span { u64 at, len; };
static bool tiles(std::vector<Span> v, u64 from, u64 to)
{
    std::sort(v.begin(), v.end(), [](const Span& x, const Span& y) { return x.at != y.at ? x.at < y.at : x.len < y.len; });
    u64 end = from;
    for (const Span& s : v) { if (s.at != end) return false; end += s.len; }
    return end == to;
}
static size_t rndFrame()
{
    switch (rnd() % 8) {
    case 0: return 0;
    case 1: return rndIn(1, 2048);
    case 2: case 3: return rndIn(2049, 128 * KiB);
    case 4: case 5: return rndIn(128 * KiB + 1, 8 * MiB);
    case 6: return rndIn(8 * MiB + 1, 40 * MiB);
    default: return rnd() % 4 ? rndIn(1, 300) : rndIn(100 * MiB, 200 * MiB);
    }
}
static void checkWave(const Batch& b, ZlEncWave& w, size_t waveBlocks, u32 dictID, u32 checksum)
{
    CHECK(w.nb <= waveBlocks || w.nf == 1);
    CHECK(w.partCut[0] == 0 && w.partCut[w.parts] == w.nf && w.parts >= 1 && w.parts <= ZL_ENC_PARTS);
    for (size_t p = 0; p < w.parts; p++) CHECK(w.partCut[p] < w.partCut[p + 1]);
    const Descs d = fill(w, dictID, checksum);
    size_t nextBlock = 0;
    u64 farEnd = 0;
    for (size_t p = 0; p < w.parts; p++) {
        const ZlEncPart& q = d.parts[p];
        CHECK(q.fa == w.partCut[p] && q.fb == w.partCut[p + 1] && q.b0 == nextBlock);
        u32 nSmall = 0;
        bool anyLarge = false;
        for (size_t r = q.fa; r < q.fb; r++) {
            const size_t i = w.f0 + r, s = b.srcSize[i];
            const ZlEncFrame& f = d.f[r];
            CHECK(f.dst == b.dst[i] && f.dstCap == b.dstCap[i] && f.checksumFlag == checksum && f.nblocks == zl_enc_nblocks(s));
            // the blocks tile the frame's input; one FIRST, one LAST
            std::vector<Span> spans;
            u32 firsts = 0, lasts = 0;
            for (size_t k = 0; k < f.nblocks; k++) {
                const ZlEncBlock& bk = d.b[q.b0 + f.firstBlock + k];
                CHECK(bk.frame == r - q.fa && bk.pad == k * ZL_BLOCKSIZE_MAX && bk.srcSize <= ZL_BLOCKSIZE_MAX && (bk.srcSize > 0 || s == 0));
                spans.push_back({(u64)(bk.src - b.src[i]), bk.srcSize});
                firsts += (bk.flags & ZL_BLK_FIRST) != 0; lasts += (bk.flags & ZL_BLK_LAST) != 0;
                CHECK(((bk.flags & ZL_BLK_FIRST) != 0) == (k == 0) && ((bk.flags & ZL_BLK_LAST) != 0) == (k + 1 == f.nblocks));
                if (bk.srcSize && bk.srcSize <= ZL_SMALL_BLOCK) nSmall++;
            }
            CHECK(tiles(spans, 0, s) && firsts == 1 && lasts == 1);
            if (r > q.fa) CHECK(f.firstBlock == d.f[r - 1].firstBlock + d.f[r - 1].nblocks);
            else CHECK(f.firstBlock == 0);
            // far tables: only for eligible frames, in frame order, disjoint, inside the budget, first come first served
            const bool eligible = f.nblocks > 1 && s < 0xFFFFFF00ull && w.farMaxOff;
            if (f.pad) {
                const u64 off = f.pad & ((1ull << 56) - 1), lg = f.pad >> 56;
                CHECK(eligible && off == farEnd && lg == zl_far_log(s) && off + zl_far_entries(s) <= (1ull << 30));
                farEnd = off + zl_far_entries(s);
            } else CHECK(!eligible || farEnd + zl_far_entries(s) > (1ull << 30) || (farEnd == 0 && zl_far_entries(s) > (1ull << 30)));
            u8 hdr[24] = {};
            const u32 hs = zl_write_frame_header(hdr, s, dictID, checksum, f.pad ? w.farMaxOff : 0u);
            CHECK(f.hdrSize == hs && memcmp(f.hdr, hdr, hs) == 0);
            if (checksum) { CHECK(d.hp[r] == b.src[i] && d.hs[r] == (u32)s); anyLarge |= s >= ZL_LARGE_FRAME_BYTES; }
        }
        CHECK(q.nSmall == nSmall && q.anyLarge == anyLarge);
        nextBlock = q.b0 + q.nb;
    }
    CHECK(nextBlock == w.nb && farEnd == w.farEntries && w.farEntries <= (1ull << 30));
}
static void randomWaves()
{
    for (int trial = 0; trial < 300; trial++) {
        // shape 0: many small frames (parts); 5: frames of 4 - 9 MiB, whose far tables outgrow the budget of a wave; else mixed
        const int shape = trial % 10;
        const size_t n = shape == 0 ? rndIn(16384, 20000) : shape == 5 ? rndIn(100, 300) : rndIn(1, 60);
        std::vector<size_t> sizes(n);
        for (size_t& s : sizes) s = shape == 0 ? rndIn(0, 3000) : shape == 5 ? rndIn(4 * MiB, 9 * MiB) : rndFrame();
        const Batch b(sizes);
        size_t wb = 0;
        CHECK(zl_enc_wave_blocks(b.srcSize.data(), n, &wb) == 0);
        const std::vector<size_t> cut = waveCuts(b);
        CHECK(cut.front() == 0 && cut.back() == n);
        for (size_t k = 0; k + 1 < cut.size(); k++) CHECK(cut[k] < cut[k + 1]);
        const u32 dictID = rnd() % 3 == 0 ? (u32)rndIn(1, 0xFFFFFFFFull) : 0u, checksum = (u32)(rnd() & 1);
        ZlEncParams P = zl_enc_params((int)rndIn(1, 3));
        ZlEncTuning t;
        if (rnd() % 4 == 0) zl_enc_tune_params(P, dictID != 0, (int)rndIn(17, 31), t);
        if (rnd() % 6 == 0) t.noFar = true;
        if (rnd() % 6 == 0) t.parts = (int)rndIn(0, 6);
        for (size_t k = 0; k + 1 < cut.size(); k++) {
            ZlEncWave w = layout(b, cut[k], cut[k + 1], rnd() % 8 == 0, P, t);
            checkWave(b, w, wb, dictID, checksum);
        }
    }
}

// host buffers: placement, the staging decision and the staged upload
static void randomPlacement()
{
    for (int trial = 0; trial < 300; trial++) {
        const size_t n = trial % 5 == 0 ? rndIn(200, 3000) : rndIn(1, 80);
        const unsigned brkPct = (unsigned)(rnd() % 101);
        std::vector<const void*> src(n); std::vector<size_t> ssz(n), cap(n);
        uintptr_t s = (uintptr_t)1 << 40;
        for (size_t i = 0; i < n; i++) {
            ssz[i] = rnd() % 16 == 0 ? rndIn(1, 100 * MiB) : rndFrame() % (2 * MiB);
            cap[i] = ssz[i] + rndIn(0, 600);
            if (rnd() % 100 < brkPct) s += rndIn(1, 4096);
            src[i] = (const void*)s; s += ssz[i];
        }
        ZlEncPlace p;
        zl_enc_place(p, src.data(), ssz.data(), cap.data(), n);
        const u8* dSrc = (const u8*)((uintptr_t)5 << 40); u8* dDst = (u8*)((uintptr_t)7 << 40);
        std::vector<const u8*> dsrc(n); std::vector<u8*> ddst(n);
        zl_enc_place_ptrs(p, src.data(), cap.data(), n, dSrc, dDst, dsrc.data(), ddst.data());
        CHECK(p.srcTotal == p.runs.back().devOff + p.runs.back().bytes);
        for (size_t r = 0; r < p.runs.size(); r++) {
            CHECK(p.runs[r].devOff % 256 == 0);
            if (r) CHECK(p.runs[r].devOff >= p.runs[r - 1].devOff + p.runs[r - 1].bytes);
        }
        std::vector<Span> slots;
        for (size_t i = 0; i < n; i++) {
            const ZlRun& r = p.runs[p.runOf[i]];
            CHECK(i >= r.first && i < r.first + r.count);
            CHECK(dsrc[i] >= dSrc + r.devOff && dsrc[i] + ssz[i] <= dSrc + r.devOff + r.bytes && dsrc[i] - (dSrc + r.devOff) == (const u8*)src[i] - r.hbase);
            CHECK((ddst[i] - dDst) % 16 == 0);
            slots.push_back({(u64)(ddst[i] - dDst), (cap[i] + 15) & ~(u64)15});
        }
        CHECK(tiles(slots, 0, p.dstTotal));
        int asked = 0;
        const bool pg = rnd() & 1;
        const bool staged = zl_enc_staged(p, n, [&] { asked++; return pg; });
        const bool spread = p.runs.size() > 64 || n > 256;
        CHECK(staged == (spread || (p.srcTotal >= 4 * MiB && pg)));
        CHECK(asked == (!spread && p.srcTotal >= 4 * MiB ? 1 : 0));
        // the staged upload: copies [from, to) chain from 0 to srcTotal; the segments packed before each lie inside it and tile the runs
        u8* hs = (u8*)((uintptr_t)9 << 40);
        const std::vector<ZlUpload> ups = zl_enc_stage_uploads(p, hs);
        size_t at = 0;
        std::vector<Span> packed, want;
        for (const ZlUpload& u : ups) {
            CHECK(u.from == at && u.to > u.from);
            at = u.to;
            for (const ZlCopySeg& g : u.segs) {
                const u64 off = (u64)((u8*)g.dst - hs);
                CHECK(g.bytes > 0 && g.bytes <= 64 * MiB && off >= u.from && off + g.bytes <= u.to);
                packed.push_back({off, g.bytes});
                const ZlRun* run = nullptr;
                for (const ZlRun& r : p.runs) if (off >= r.devOff && off < r.devOff + r.bytes) run = &r;
                CHECK(run && off + g.bytes <= run->devOff + run->bytes && (const u8*)g.src == run->hbase + (off - run->devOff));
            }
        }
        CHECK(at == (p.srcTotal ? p.srcTotal : 0));
        for (const ZlRun& r : p.runs) if (r.bytes) want.push_back({r.devOff, r.bytes});
        std::sort(packed.begin(), packed.end(), [](const Span& x, const Span& y) { return x.at < y.at; });
        std::vector<Span> merged;                       // adjacent pieces of one run merge back into the run
        for (const Span& g : packed) { if (!merged.empty() && merged.back().at + merged.back().len == g.at) merged.back().len += g.len; else merged.push_back(g); }
        std::vector<Span> wantMerged;
        for (const Span& g : want) { if (!wantMerged.empty() && wantMerged.back().at + wantMerged.back().len == g.at) wantMerged.back().len += g.len; else wantMerged.push_back(g); }
        CHECK(merged.size() == wantMerged.size());
        for (size_t k = 0; k < merged.size() && k < wantMerged.size(); k++) CHECK(merged[k].at == wantMerged[k].at && merged[k].len == wantMerged[k].len);
    }
}

// gather tables and split frames
static void randomGatherSplit()
{
    for (int trial = 0; trial < 300; trial++) {
        const size_t n = rndIn(1, 5000);
        std::vector<u64> res(n), t(3 * n);
        std::vector<u8*> ddst(n);
        for (size_t i = 0; i < n; i++) {
            res[i] = rnd() % 7 == 0 ? (u64)ZL_ERROR(dstSize_tooSmall) : (u64)rndIn(0, 200000);
            ddst[i] = (u8*)(((uintptr_t)7 << 40) + i * 200064);
        }
        const size_t total = zl_enc_gather_table(t.data(), res.data(), ddst.data(), n);
        const u8* const* ptr = reinterpret_cast<const u8* const*>(t.data() + 2 * n);
        u64 sum = 0;
        for (size_t i = 0; i < n; i++) {
            const u64 got = zl_is_error((size_t)res[i]) ? 0 : res[i];
            CHECK(t[i] == got && t[n + i] == sum && ptr[i] == ddst[i]);
            sum += got;
        }
        CHECK(total == sum);

        const size_t frameSize = rnd() % 3 ? rndIn(1, 300000) : (size_t)1 << rndIn(10, 20);
        const size_t bytes = rnd() % 10 == 0 ? 0 : rndIn(1, 64 * frameSize);
        const ZlSplitPlan sp = zl_enc_split_plan(bytes, frameSize, rnd() & 1);
        CHECK(sp.nf == (bytes ? (bytes + frameSize - 1) / frameSize : 1));
        const size_t slot = (frameSize + 64 + 15) & ~(size_t)15;
        std::vector<const u8*> dsrc(sp.nf); std::vector<size_t> ssz(sp.nf); std::vector<u8*> dd(sp.nf);
        const u8* base = (const u8*)((uintptr_t)1 << 40); u8* dbase = (u8*)((uintptr_t)3 << 40);
        zl_enc_split_frames(base, bytes, frameSize, dbase, slot, sp.nf, dsrc.data(), ssz.data(), dd.data());
        std::vector<Span> spans;
        for (size_t i = 0; i < sp.nf; i++) {
            CHECK(dd[i] == dbase + i * slot && (i + 1 == sp.nf ? ssz[i] <= frameSize : ssz[i] == frameSize));
            spans.push_back({(u64)(dsrc[i] - base), ssz[i]});
        }
        CHECK(tiles(spans, 0, bytes));
        if (!bytes) CHECK(sp.nf == 1 && ssz[0] == 0);
        if (sp.pipelined) {                             // chunks: 1/8 of a full one, doubling, then full ones, the last short
            const std::vector<size_t> cs = chunkSizes(sp);
            CHECK(sp.cstart.front() == 0 && sp.cstart.back() == sp.nf && cs.size() >= 2);
            size_t want = std::max<size_t>(sp.chunkFrames / 8, 1);
            for (size_t k = 0; k + 1 < cs.size(); k++) { CHECK(cs[k] == want); want = std::min(want * 2, sp.chunkFrames); }
            CHECK(cs.back() >= 1 && cs.back() <= want);
        }
    }
    // the pipelined rule over frame sizes: chunks of <= ZL_WAVE_BLOCKS blocks and <= 1 GiB, >= 64 MiB, >= 2 of them, host buffers only
    for (size_t fs : {16 * KiB, 100 * KiB, 128 * KiB, 1 * MiB, 8 * MiB, 300 * MiB, 2 * GiB})
        for (size_t total : {1 * GiB, 3 * GiB, 8 * GiB}) {
            const ZlSplitPlan sp = zl_enc_split_plan(total, fs, false);
            const size_t cf = std::min<size_t>(ZL_WAVE_BLOCKS / zl_enc_nblocks(fs), GiB / fs);
            CHECK(sp.chunkFrames == cf && sp.pipelined == (cf >= 1 && sp.nf >= 2 * cf && cf * fs >= 64 * MiB));
            CHECK(!zl_enc_split_plan(total, fs, true).pipelined);
        }
}

int main()
{
    exactPlans();
    randomWaves();
    randomPlacement();
    randomGatherSplit();
    printf("bad=%d\n", bad);
    return bad ? 1 : 0;
}
