// The frame index of a device stream (zstdlite_b200/csrc/zl_stream_index.h) on the CPU: the ZL_HD bodies of I1-I4 run in host loops
// with the kernels' pass structure (tiles, one scan, double-buffered marking passes in groups of 4, frontier rounds) and are compared
// with the serial walk (zl_host_find_frame_size frame after frame) over seeded random streams, under single faults, with the shipped
// step cap and a small one.  Also checks the decode plan against a byte-level model of ZSTD_decompressDCtx.  Prints "bad=0" when all hold.
#include <cstdio>
#include <random>
#include "zl_stream_index.h"

static size_t g_bad = 0, g_streams = 0, g_faults = 0;
#define CHECK(c, ...) do { if (!(c)) { if (g_bad++ < 20) { printf("FAIL %s:%d ", __FILE__, __LINE__); printf(__VA_ARGS__); printf("\n"); } } } while (0)

struct Work { u64 steps = 0, passes = 0, rounds = 0, maxRoundPasses = 0; };

// the index as the device builds it; `head` misaligns the stream inside its 16-byte chunks
static size_t index_host(const std::vector<u8>& s, u32 W, u32 R, u32 head, std::vector<ZlStreamFrame>& frames, Work& work)
{
    frames.clear();
    const u64 srcSize = s.size();
    if (!srcSize) return 0;
    if (srcSize < 5) return ZL_ERROR(srcSize_wrong);
    const u64 lastChunk = (head + srcSize - 1) >> 4;
    std::vector<u8> mem((lastChunk + 2) * 16, 0);                       // (the chunk after the last is never read: zeros stand for it)
    memcpy(mem.data() + head, s.data(), srcSize);
    const u8* src = mem.data() + head;
    // I1: per tile counts, one scan, then the write pass in the kernels' order
    const u64 tileChunks = ZL_IDX_TILE_THREADS * ZL_IDX_TILE_CHUNKS, tiles = (lastChunk + tileChunks) / tileChunks;
    auto chunkMask = [&](u64 c) -> u32 {
        if (c > lastChunk) return 0;
        u32 w[8];
        for (int k = 0; k < 8; k++) w[k] = (c < lastChunk || k < 4) ? zl_rd32(mem.data() + c * 16 + 4 * k) : 0u;
        const i64 at = (i64)(c << 4) - (i64)head, lo = -at, hi = (i64)srcSize - 4 - at;
        return zl_idx_chunk_mask(w, lo < 0 ? 0 : (lo > 16 ? 16 : (int)lo), hi > 15 ? 15 : (hi < -1 ? -1 : (int)hi));
    };
    std::vector<u64> tileOff(tiles + 1, 0);
    for (u64 t = 0; t < tiles; t++) {
        u64 cnt = 0;
        for (u32 j = 0; j < ZL_IDX_TILE_CHUNKS; j++) for (u32 th = 0; th < ZL_IDX_TILE_THREADS; th++) cnt += __builtin_popcount(chunkMask((t * ZL_IDX_TILE_CHUNKS + j) * ZL_IDX_TILE_THREADS + th));
        tileOff[t + 1] = tileOff[t] + cnt;
    }
    const u64 n64 = tileOff[tiles];
    if (!n64) return ZL_ERROR(prefix_unknown);
    const u32 n = (u32)n64;
    std::vector<u64> cand(n);
    for (u64 t = 0; t < tiles; t++) {
        u64 w = tileOff[t];
        for (u32 j = 0; j < ZL_IDX_TILE_CHUNKS; j++) for (u32 th = 0; th < ZL_IDX_TILE_THREADS; th++) {
            const u64 c = (t * ZL_IDX_TILE_CHUNKS + j) * ZL_IDX_TILE_THREADS + th;
            for (u32 m = chunkMask(c); m; m &= m - 1) cand[w++] = (c << 4) + __builtin_ctz(m) - head;
        }
        CHECK(w == tileOff[t + 1], "tile %llu wrote %llu", (unsigned long long)t, (unsigned long long)w);
    }
    for (u32 i = 1; i < n; i++) CHECK(cand[i - 1] < cand[i], "candidates out of order");
    // I2
    std::vector<u32> link(n), errc(n), nblk(n), mark(n), j0(n), j1(n);
    for (u32 i = 0; i < n; i++) {
        zl_idx_extent(src, srcSize, cand.data(), n, i, W, link.data(), errc.data(), nblk.data());
        work.steps += link[i] == ZL_LINK_LONG ? W : nblk[i];
        mark[i] = i == 0 && cand[0] == 0;
    }
    ZlIdxStatus st{};
    for (u32 round = 0;; round++) {
        work.rounds++;
        j0 = link;
        u64 passes = 0;
        for (u32 pass = 0;; pass += 4) {
            CHECK(pass + 4 <= ZL_IDX_MAX_PASSES, "marking does not converge");
            if (pass + 4 > ZL_IDX_MAX_PASSES) return ZL_ERROR(GENERIC);
            u32 open[4] = {};
            for (u32 q = 0; q < 4; q++) {
                if (q > 0 && open[q - 1] == 0) break;
                passes++;
                const u32 p = pass + q;
                for (u32 v = 0; v < n; v++) open[q] += zl_idx_jump(v, p & 1 ? j1.data() : j0.data(), p & 1 ? j0.data() : j1.data(), mark.data());
            }
            if (open[3] == 0) break;
        }
        work.passes += passes; work.maxRoundPasses = std::max(work.maxRoundPasses, passes);
        st = ZlIdxStatus{cand[0], ~0u, ~0u, ~0u, 0};
        for (u32 v = 0; v < n; v++) if (mark[v] && link[v] >= ZL_LINK_NODES) { st.tail = v; st.link = link[v]; st.err = errc[v]; }
        if (st.first != 0 || st.link != ZL_LINK_LONG) break;
        for (u32 v = st.tail;;) {                                         // zl_k_idx_frontier
            zl_idx_extent(src, srcSize, cand.data(), n, v, 0, link.data(), errc.data(), nblk.data());
            work.steps += nblk[v];
            const u32 j = link[v];
            if (round < R || j >= ZL_LINK_NODES) break;
            mark[j] = 1; v = j;
        }
    }
    const size_t status = zl_idx_tail_error(n64, st.first, st.link, st.err);
    if (st.first == 0)
        for (u32 v = 0; v < n; v++) if (zl_idx_is_frame(mark.data(), link.data(), v)) frames.push_back(zl_idx_record(src, srcSize, cand.data(), link.data(), nblk.data(), v));
    return status;
}

// ---- stream generator --------------------------------------------------------------------------------------------------------------
static std::mt19937_64 rng(20261022);
static u32 rnd(u32 n) { return (u32)(rng() % n); }
static void put(std::vector<u8>& o, u64 v, int bytes) { for (int i = 0; i < bytes; i++) o.push_back((u8)(v >> (8 * i))); }
static const u8 kMagic[4] = {0x28, 0xB5, 0x2F, 0xFD};

static std::vector<u8> make_stream(int depth);
// raw block content: random bytes with planted look-alikes, a "magic then zeros" run, or a whole stream
static std::vector<u8> raw_payload(int depth, bool* embedded)
{
    std::vector<u8> b;
    const u32 kind = rnd(8);
    if (kind == 0 && depth < 1) { b = make_stream(depth + 1); *embedded = true; return b; }
    const u32 len = rnd(4) == 0 ? 3000 + rnd(2000) : rnd(300);
    for (u32 i = 0; i < len; i++) b.push_back((u8)rng());
    const u32 plants = rnd(4);
    for (u32 k = 0; k < plants && len > 16; k++) {
        const u32 at = rnd(len - 12);
        if (rnd(2)) memcpy(&b[at], kMagic, 4); else { b[at] = 0x50 + rnd(16); b[at + 1] = 0x2A; b[at + 2] = 0x4D; b[at + 3] = 0x18; }
        if (kind == 1) for (u32 i = at + 4; i < len; i++) b[i] = 0;       // every walk from here takes 3-byte empty raw blocks: LONG
    }
    return b;
}
struct Opt { bool checksum, fcs, single; };
static void make_frame(std::vector<u8>& o, int depth, u32 maxBlocks)
{
    const bool checksum = rnd(2), fcs = rnd(3) != 0, single = fcs && rnd(4) == 0;
    std::vector<u8> body; u64 content = 0;
    const u32 nb = rnd(5) == 0 ? 0 : 1 + rnd(maxBlocks);
    bool embedded = false;
    for (u32 b = 0; b < std::max(nb, 1u); b++) {
        const bool last = b + 1 >= std::max(nb, 1u);
        const u32 type = nb == 0 ? 0 : rnd(3);
        std::vector<u8> pay;
        u32 size = 0;
        if (type == 0) { if (nb) pay = raw_payload(depth, &embedded); size = (u32)pay.size(); content += size; }
        else if (type == 1) { size = 1 + rnd(5000); pay.push_back((u8)rng()); content += size; }
        else { size = 1 + rnd(200); for (u32 i = 0; i < size; i++) pay.push_back((u8)rng()); content += 3 * size; }
        put(body, ((u32)size << 3) | (type << 1) | (last ? 1 : 0), 3);
        body.insert(body.end(), pay.begin(), pay.end());
    }
    // an embedded stream ends the frame exactly: its raw block must be the last thing in it
    o.insert(o.end(), kMagic, kMagic + 4);
    const u32 fcsID = !fcs ? 0 : (content < 256 && single ? 0 : (content < 65536 + 256 ? 1 : 2));
    const u32 fhd = (fcsID << 6) | ((single ? 1u : 0u) << 5) | ((checksum && !embedded) ? 4u : 0u);
    o.push_back((u8)fhd);
    if (!single) o.push_back((u8)(rnd(8) << 3));                     // window 2^10 .. 2^17
    if (fcs) { if (fcsID == 0) put(o, content, 1); else if (fcsID == 1) put(o, content - 256, 2); else put(o, content, 4); }
    o.insert(o.end(), body.begin(), body.end());
    if (checksum && !embedded) put(o, rng(), 4);
}
static void make_skippable(std::vector<u8>& o)
{
    const u32 len = rnd(3) == 0 ? 0 : rnd(100);
    put(o, 0x184D2A50u + rnd(16), 4); put(o, len, 4);
    for (u32 i = 0; i < len; i++) o.push_back((u8)rng());
}
static u32 g_maxBlocks = 6;
static std::vector<u8> make_stream(int depth)
{
    std::vector<u8> o;
    const u32 frames = 1 + rnd(depth ? 3 : 12);
    if (rnd(4) == 0) make_skippable(o);
    for (u32 f = 0; f < frames; f++) { if (rnd(5) == 0) make_skippable(o); make_frame(o, depth, g_maxBlocks); }
    if (rnd(4) == 0) {                                                // a seek table: a skippable frame with the seekable footer
        const u32 n = 1 + rnd(4);
        put(o, 0x184D2A5Eu, 4); put(o, 8 * n + 9, 4);
        for (u32 i = 0; i < 2 * n; i++) put(o, rng(), 4);
        put(o, n, 4); o.push_back(0); put(o, 0x8F92EAB1u, 4);
    }
    return o;
}

// ---- comparisons -------------------------------------------------------------------------------------------------------------------
static void compare(const std::vector<u8>& s, u32 W, const char* what)
{
    std::vector<ZlStreamFrame> want, got;
    const size_t ws = zl_stream_walk(s.data(), s.size(), want);
    for (u32 head = 0; head < 16; head += 5) {
        Work work;
        const size_t gs = index_host(s, W, ZL_IDX_R, head, got, work);
        CHECK(gs == ws, "%s W=%u head=%u: status %zx, walk %zx (size %zu)", what, W, head, gs, ws, s.size());
        if (gs != ws) return;
        if (s.size() >= 5 && ws != ZL_ERROR(prefix_unknown)) {
            CHECK(got.size() == want.size(), "%s: %zu frames, walk %zu", what, got.size(), want.size());
            if (got.size() != want.size()) return;
            for (size_t k = 0; k < got.size(); k++) {
                const bool lastOfError = zl_is_error(ws) && k + 1 == got.size();
                CHECK(got[k].cOff == want[k].cOff && got[k].dSize == want[k].dSize && got[k].nblocks == want[k].nblocks && got[k].bsm == want[k].bsm &&
                      (lastOfError || got[k].cSize == want[k].cSize), "%s: frame %zu differs", what, k);
            }
        }
        // the bound: W steps per candidate in I2 plus the stream's own blocks in the frontier walks; at most R + 2 rounds of
        // ceil(log2 n) + 1 marking passes (run in groups of 4)
        u64 n = 0; for (size_t i = 0; i + 4 <= s.size(); i++) n += zl_idx_magic(zl_rd32(&s[i]));
        u32 lg = 0; while ((1ull << lg) < n) lg++;
        CHECK(work.steps <= (u64)W * n + s.size() / 3 * (ZL_IDX_R + 1), "%s: %llu block steps", what, (unsigned long long)work.steps);
        CHECK(work.rounds <= ZL_IDX_R + 2 && work.maxRoundPasses <= lg + 1 + 3, "%s: %llu rounds, %llu passes", what, (unsigned long long)work.rounds, (unsigned long long)work.maxRoundPasses);
    }
}

static void faults(const std::vector<u8>& s, u32 W)
{
    std::vector<ZlStreamFrame> f;
    if (zl_stream_walk(s.data(), s.size(), f) != 0) return;
    auto run = [&](std::vector<u8> t, const char* what) { g_faults++; compare(t, W, what); };
    for (int k = 0; k < 4; k++) run(std::vector<u8>(s.begin(), s.begin() + rnd((u32)s.size())), "truncated");
    for (u32 t = 1; t <= 4; t++) { std::vector<u8> x = s; for (u32 i = 0; i < t; i++) x.push_back((u8)rng()); run(x, "trailing bytes"); }
    const ZlStreamFrame& fr = f[rnd((u32)f.size())];
    { std::vector<u8> x = s; x[fr.cOff + 3] ^= 0x40; run(x, "non-magic at a boundary"); }
    if (fr.bsm != ZL_FRAME_SKIP) {
        ZlHostFrameHeader h; zl_frame_head(&h, &s[fr.cOff], s.size() - fr.cOff);
        { std::vector<u8> x = s; x[fr.cOff + h.headerSize] |= 6; run(x, "block type 3"); }
        { std::vector<u8> x = s; x[fr.cOff + 4] |= 8; run(x, "FHD bit 3"); }
        if (!((s[fr.cOff + 4] >> 5) & 1)) { std::vector<u8> x = s; x[fr.cOff + 5] = 0xFF; run(x, "window too large"); }
    }
}

// the decode plan against a model of ZSTD_decompressDCtx: frames in order, each at the running output size; frames without content size
// take their decoded size (or fail) in place
static void check_plan(const std::vector<ZlStreamFrame>& f)
{
    for (int rep = 0; rep < 4; rep++) {
        u64 need = 0; for (const ZlStreamFrame& x : f) if (x.bsm != ZL_FRAME_SKIP && x.dSize != ~0ull) need += x.dSize;
        const u64 cap = rep == 0 ? need + 100000 : (rep == 1 ? need : need + rnd(20000));
        ZlDevPlan p;
        const size_t r1 = zl_dev_plan_unknown(p, f, 0, cap);
        CHECK(r1 == 0, "plan refused a fitting stream");
        if (r1) continue;
        std::vector<size_t> ures(p.unknown.size());
        u64 prev = 0;
        for (size_t j = 0; j < p.unknown.size(); j++) {
            const ZlDevDecode& u = p.unknown[j]; const ZlStreamFrame& x = f[u.frame];
            CHECK(u.place % 16 == 0 && u.place >= prev && u.cap == std::min<u64>((u64)x.nblocks * x.bsm, cap), "scratch layout");
            prev = u.place + u.cap;
            ures[j] = rnd(6) == 0 ? ZL_ERROR(corruption_detected) : rnd((u32)std::min<u64>(u.cap, 9000) + 1);
        }
        CHECK(p.scratchBytes >= prev, "scratch size");
        zl_dev_plan_places(p, f, ures.data(), cap);
        std::vector<size_t> kres(p.known.size());
        for (size_t i = 0; i < kres.size(); i++) kres[i] = rnd(10) == 0 ? ZL_ERROR(checksum_wrong) : p.known[i].cap;
        const size_t got = zl_dev_plan_result(p, kres.data());
        // model
        u64 op = 0; size_t j = 0, i = 0, want = 0; bool done = false;
        std::vector<ZlDevPiece> pieces;
        for (size_t k = 0; k < f.size() && !done; k++) {
            if (f[k].bsm == ZL_FRAME_SKIP) continue;
            if (f[k].dSize == ~0ull) {
                const size_t r = ures[j]; const u64 from = p.unknown[j++].place;
                if (zl_is_error(r)) { want = r; done = true; break; }
                if (r > cap - op) { want = ZL_ERROR(dstSize_tooSmall); done = true; break; }
                for (u64 o = 0; o < r; o += ZL_SCATTER_BYTES) pieces.push_back({from + o, op + o, std::min<u64>(r - o, ZL_SCATTER_BYTES)});
                op += r;
            } else {
                if (f[k].dSize > cap - op) { want = ZL_ERROR(dstSize_tooSmall); done = true; break; }
                CHECK(i < p.known.size() && p.known[i].frame == k && p.known[i].place == op && p.known[i].cap == f[k].dSize, "known frame %zu", k);
                if (i < kres.size() && zl_is_error(kres[i]) && !done) { want = kres[i]; done = true; }
                i++;
                op += f[k].dSize;
            }
        }
        if (!done) want = op;
        CHECK(got == want, "plan result %zx, model %zx", got, want);
        if (!zl_is_error(want)) {
            CHECK(pieces.size() == p.pieces.size(), "pieces %zu, model %zu", p.pieces.size(), pieces.size());
            for (size_t k = 0; k < pieces.size() && k < p.pieces.size(); k++)
                CHECK(pieces[k].from == p.pieces[k].from && pieces[k].to == p.pieces[k].to && pieces[k].bytes == p.pieces[k].bytes, "piece %zu", k);
        }
    }
    // dstSize_tooSmall at the frame where the content sizes overflow, before any later structural error
    u64 need = 0; for (const ZlStreamFrame& x : f) if (x.bsm != ZL_FRAME_SKIP && x.dSize != ~0ull) need += x.dSize;
    ZlDevPlan p;
    if (need) CHECK(zl_dev_plan_unknown(p, f, ZL_ERROR(srcSize_wrong), need - 1) == ZL_ERROR(dstSize_tooSmall), "dstCapacity one byte short");
    CHECK(zl_dev_plan_unknown(p, f, ZL_ERROR(srcSize_wrong), need) == ZL_ERROR(srcSize_wrong), "structural error after the frames");
}

int main()
{
    // the host walk keeps its old results on the shared rule (spot checks of zl_host_find_frame_size's cases)
    { const u8 a[3] = {0x28, 0xB5, 0x2F}; CHECK(zl_frame_extent(a, 3, 0).err == ZL_ERROR(srcSize_wrong), "short prefix"); }
    { const u8 a[6] = {1, 2, 3, 4, 5, 6}; CHECK(zl_frame_extent(a, 6, 0).err == ZL_ERROR(prefix_unknown), "non-magic"); }
    { const u8 a[7] = {0x50, 0x2A, 0x4D, 0x18, 0, 0, 0}; CHECK(zl_frame_extent(a, 7, 0).err == ZL_ERROR(srcSize_wrong), "short skippable"); }
    { const u8 a[8] = {0x5F, 0x2A, 0x4D, 0x18, 0, 0, 0, 0}; const ZlExtent x = zl_frame_extent(a, 8, 0); CHECK(x.state == 0 && x.end == 8, "empty skippable"); }
    for (u32 W : {ZL_IDX_W, 4u}) {
        for (int t = 0; t < 300; t++) {
            g_maxBlocks = W == 4 ? 12 : 6;
            std::vector<u8> s = make_stream(0);
            g_streams++;
            compare(s, W, "stream");
            faults(s, W);
            std::vector<ZlStreamFrame> f;
            if (W == ZL_IDX_W && zl_stream_walk(s.data(), s.size(), f) == 0) check_plan(f);
        }
        // magic followed by zeros everywhere: every look-alike is LONG, and so is the true frame's walk with a small cap
        std::vector<u8> z;
        z.insert(z.end(), kMagic, kMagic + 4); z.push_back(0); z.push_back(0);
        for (int k = 0; k < 4000; k++) { put(z, 0, 3); if (k % 97 == 0) { put(z, 4 << 3, 3); z.insert(z.end(), kMagic, kMagic + 4); } }
        put(z, 1, 3);
        g_streams++;
        compare(z, W, "magic then zeros");
        for (u32 len : {0u, 1u, 2u, 3u, 4u}) compare(std::vector<u8>(z.begin(), z.begin() + len), W, "tiny");
    }
    printf("streams=%zu faults=%zu bad=%zu\n", g_streams, g_faults, g_bad);
    return g_bad ? 1 : 0;
}
