// Test infrastructure: checks the many-range plan of seekable streams (zl_ranges_streams / zl_ranges_plan / zl_ranges_results in
// zstdlite_b200/csrc/zl_seek.h) on the CPU against a byte-level model.  Seeded random streams (zero-size frames, tables with and without
// checksums, one with a broken table) and random item lists (duplicates, nested and overlapping ranges, neighbours sharing an edge
// frame, zero lengths, offsets at and past the end, capacities too small, null destinations).  Built and run by tests/test_ranges_plan.py;
// no CUDA call is made.
#include "zl_seek.h"
#include <cstdio>
#include <set>
#include <vector>

static int bad = 0;
#define CHECK(c) do { if (!(c)) { if (bad++ < 20) printf("FAIL line %d: %s\n", __LINE__, #c); } } while (0)

static unsigned long long rngState = 0x9E3779B97F4A7C15ull;
static unsigned long long rnd() { rngState ^= rngState << 13; rngState ^= rngState >> 7; rngState ^= rngState << 17; return rngState; }
static size_t rndIn(size_t lo, size_t hi) { return lo + (size_t)(rnd() % (hi - lo + 1)); }

// a stream's bytes: n frames of filler and the table; `broken` flips a reserved descriptor bit
static std::vector<u8> makeStream(const std::vector<u32>& c, const std::vector<u32>& d, bool ck, bool broken)
{
    std::vector<u32> sums;
    if (ck) for (size_t i = 0; i < c.size(); i++) sums.push_back((u32)rnd());
    std::vector<u8> b;
    for (size_t i = 0; i < c.size(); i++) b.insert(b.end(), c[i], (u8)i);
    const size_t at = b.size(), ts = zl_seek_table_size(c.size(), ck);
    b.resize(at + ts);
    zl_seek_write(b.data() + at, c.size(), c.data(), d.data(), ck ? sums.data() : nullptr);
    if (broken) b[b.size() - 5] |= 0x08;
    return b;
}
static size_t parse(ZlSeekTable& t, const std::vector<u8>& b)
{
    u32 n = 0; bool ck = false;
    const size_t tail = b.size() < ZL_SEEK_FOOTER ? b.size() : ZL_SEEK_FOOTER;
    const size_t size = zl_seek_footer(b.data() + b.size() - tail, b.size(), &n, &ck);
    if (zl_is_error(size)) return size;
    return zl_seek_parse(t, b.data() + b.size() - size, size, b.size());
}
// the model's content: byte x of stream s
static u32 model(size_t s, u64 x) { return (u32)(s * 1000003u + x); }

// what zl_decompress_range checks before it decodes, in its order
static size_t single(const ZlSeekTable& t, size_t tableErr, u64 off, u64 len, size_t cap, bool dstNull, ZlSeekPlan& sp)
{
    sp = ZlSeekPlan();
    if (zl_is_error(tableErr)) return tableErr;
    if (const size_t r = zl_seek_plan_range(sp, t, off, len)) return r;
    if (sp.bytes > cap) return ZL_ERROR(dstSize_tooSmall);
    if (!sp.bytes) return 0;
    if (dstNull) return ZL_ERROR(dstBuffer_null);
    return sp.bytes;
}

static size_t plansChecked = 0, itemsChecked = 0, sharedSeen = 0, directSeen = 0, piecesSeen = 0;

static void checkCall(int it)
{
    // streams: 1-4, a few of them the same stream again (another item key with the same bytes is a different stream)
    const size_t ns = rndIn(1, 4);
    std::vector<std::vector<u8>> bytes(ns);
    std::vector<ZlSeekTable> tables(ns);
    std::vector<size_t> tableErr(ns);
    for (size_t s = 0; s < ns; s++) {
        const size_t n = rndIn(1, it < 20 ? 4 : 30);
        std::vector<u32> c(n), d(n);
        for (size_t f = 0; f < n; f++) { c[f] = (u32)rndIn(9, 40); d[f] = rnd() % 4 == 0 ? 0u : (u32)rndIn(1, it % 3 == 0 ? 4 : 200); }
        if (it % 5 == 0) d[0] = 0;
        bytes[s] = makeStream(c, d, rnd() & 1, ns > 1 && s == 1 && it % 4 == 0);
        tableErr[s] = parse(tables[s], bytes[s]);
    }
    // items
    const size_t n = rndIn(1, 40);
    std::vector<const void*> src(n); std::vector<size_t> srcSize(n), offset(n), length(n), cap(n);
    std::vector<void*> dst(n);
    for (size_t i = 0; i < n; i++) {
        const size_t s = rndIn(0, ns - 1);
        const u64 total = zl_is_error(tableErr[s]) ? 1000 : tables[s].dOff[tables[s].n];
        src[i] = bytes[s].data(); srcSize[i] = bytes[s].size();
        const int kind = (int)rndIn(0, 9);
        if (kind == 0 && i) { src[i] = src[i - 1]; srcSize[i] = srcSize[i - 1]; offset[i] = offset[i - 1]; length[i] = length[i - 1]; }  // duplicate
        else if (kind == 1 && i && src[i - 1] == src[i] && length[i - 1] > 2) {                  // nested in the previous
            offset[i] = offset[i - 1] + 1; length[i] = length[i - 1] - 2;
        } else if (kind == 2 && i && src[i - 1] == src[i]) {                                      // starts where the previous ends
            offset[i] = offset[i - 1] + length[i - 1]; length[i] = rndIn(0, 300);
        } else if (kind == 3 && i && src[i - 1] == src[i] && length[i - 1]) {                    // overlaps the previous' end
            offset[i] = offset[i - 1] + length[i - 1] / 2; length[i] = length[i - 1];
        } else if (kind == 4) { offset[i] = total; length[i] = rndIn(0, 5); }
        else if (kind == 5) { offset[i] = total + rndIn(1, 3); length[i] = 1; }
        else if (kind == 6) { offset[i] = rndIn(0, total); length[i] = 0; }
        else if (kind == 7 && !zl_is_error(tableErr[s])) {                                       // from a frame boundary
            const ZlSeekTable& t = tables[s];
            offset[i] = t.dOff[rndIn(0, t.n)]; length[i] = rndIn(0, total + 10);
        } else { offset[i] = rndIn(0, total); length[i] = rnd() % 8 == 0 ? ~(size_t)0 : rndIn(1, total + 20); }
        const u64 want = offset[i] <= total ? std::min<u64>(length[i], total - offset[i]) : 0;
        cap[i] = rnd() % 10 == 0 && want ? want - 1 : want + rndIn(0, 3);
        dst[i] = rnd() % 20 == 0 ? nullptr : (void*)(uintptr_t)(0x10000 * (i + 1));
    }
    // streams are keyed by (src, srcSize)
    std::vector<size_t> streamOf(n), firstItem;
    const size_t nk = zl_ranges_streams(src.data(), srcSize.data(), n, streamOf.data(), firstItem);
    std::vector<size_t> keyStream(nk);                       // the test's stream of each key
    for (size_t k = 0; k < nk; k++) {
        keyStream[k] = ns;
        for (size_t s = 0; s < ns; s++) if (bytes[s].data() == src[firstItem[k]]) keyStream[k] = s;
        CHECK(keyStream[k] < ns && firstItem[k] < n && streamOf[firstItem[k]] == k);
        for (size_t j = 0; j < firstItem[k]; j++) CHECK(streamOf[j] != k);
    }
    for (size_t i = 0; i < n; i++) for (size_t j = 0; j < i; j++)
        CHECK((streamOf[i] == streamOf[j]) == (src[i] == src[j] && srcSize[i] == srcSize[j]));
    std::vector<ZlSeekTable> kt(nk);
    std::vector<size_t> kerr(nk);
    for (size_t k = 0; k < nk; k++) { kt[k] = tables[keyStream[k]]; kerr[k] = tableErr[keyStream[k]]; }

    ZlRangesPlan p;
    zl_ranges_plan(p, kt, kerr, streamOf.data(), offset.data(), length.data(), dst.data(), cap.data(), n);
    plansChecked++;
    CHECK(p.result.size() == n && p.touchStart.size() == n + 1 && p.touchStart[n] == p.touch.size());
    // every (stream, frame) at most once, in order
    std::set<std::pair<size_t, size_t>> seen;
    for (size_t k = 0; k < p.decodes.size(); k++) {
        const ZlRangeDecode& d = p.decodes[k];
        CHECK(d.stream < nk && d.frame < kt[d.stream].n && d.size == kt[d.stream].dSize[d.frame]);
        CHECK(seen.insert({d.stream, d.frame}).second);
        if (k) CHECK(std::make_pair(p.decodes[k - 1].stream, p.decodes[k - 1].frame) < std::make_pair(d.stream, d.frame));
    }
    // per item: the pre-decode result and the frames touched equal the single-range plan's
    std::vector<std::vector<size_t>> touchedBy(p.decodes.size());
    std::vector<ZlSeekPlan> sps(n);
    for (size_t i = 0; i < n; i++) {
        const size_t k = streamOf[i];
        const size_t want = single(kt[k], kerr[k], offset[i], length[i], cap[i], dst[i] == nullptr, sps[i]);
        CHECK(p.result[i] == want);
        const bool decodes = !zl_is_error(want) && want > 0;
        const size_t nt = p.touchStart[i + 1] - p.touchStart[i];
        CHECK(nt == (decodes ? sps[i].last - sps[i].first : 0));
        if (nt != (decodes ? sps[i].last - sps[i].first : 0)) continue;
        for (size_t j = 0; j < nt; j++) {
            const size_t id = p.touch[p.touchStart[i] + j];
            CHECK(id < p.decodes.size() && p.decodes[id].stream == k && p.decodes[id].frame == sps[i].first + j);
            if (id < p.decodes.size()) touchedBy[id].push_back(i);
        }
    }
    for (size_t id = 0; id < p.decodes.size(); id++) CHECK(!touchedBy[id].empty());
    // place every decode, direct ones into their item's output, the others into scratch (16-byte aligned, disjoint)
    const u32 NONE = 0xFFFFFFFFu;
    std::vector<std::vector<u32>> out(n);
    std::vector<std::vector<u8>> cover(n);
    for (size_t i = 0; i < n; i++) if (!zl_is_error(p.result[i])) { out[i].assign(p.result[i], NONE); cover[i].assign(p.result[i], 0); }
    std::vector<u32> scratch(p.scratchBytes, NONE);
    std::vector<u8> used(p.scratchBytes, 0);
    for (size_t id = 0; id < p.decodes.size(); id++) {
        const ZlRangeDecode& d = p.decodes[id];
        const ZlSeekTable& t = kt[d.stream];
        if (d.item != ZL_RANGE_SCRATCH) {
            directSeen++;
            const size_t i = d.item;
            CHECK(touchedBy[id].size() == 1 && touchedBy[id][0] == i);
            CHECK(t.dOff[d.frame] >= offset[i] && t.dOff[d.frame + 1] <= offset[i] + p.result[i] && d.place == t.dOff[d.frame] - offset[i]);
            if (d.place + d.size > out[i].size()) { CHECK(false); continue; }
            for (u32 x = 0; x < d.size; x++) { out[i][d.place + x] = model(keyStream[d.stream], t.dOff[d.frame] + x); cover[i][d.place + x]++; }
        } else {
            if (touchedBy[id].size() > 1) sharedSeen++;
            // a scratch frame is shared, or its only item wants part of it
            if (touchedBy[id].size() == 1) {
                const size_t i = touchedBy[id][0];
                CHECK(t.dOff[d.frame] < offset[i] || t.dOff[d.frame + 1] > offset[i] + p.result[i]);
            }
            CHECK(d.place % 16 == 0 && d.place + d.size <= p.scratchBytes);
            if (d.place + d.size > p.scratchBytes) continue;
            for (u32 x = 0; x < d.size; x++) { CHECK(!used[d.place + x]); used[d.place + x] = 1; scratch[d.place + x] = model(keyStream[d.stream], t.dOff[d.frame] + x); }
        }
    }
    u64 aligned = 0;
    for (const ZlRangeDecode& d : p.decodes) if (d.item == ZL_RANGE_SCRATCH) aligned += (d.size + 15) & ~(u64)15;
    CHECK(aligned == p.scratchBytes);
    for (const ZlRangePiece& q : p.pieces) {
        piecesSeen++;
        CHECK(q.item < n && q.bytes > 0 && !zl_is_error(p.result[q.item]));
        if (q.item >= n || zl_is_error(p.result[q.item]) || q.outOff + q.bytes > out[q.item].size() || q.from + q.bytes > p.scratchBytes) { CHECK(false); continue; }
        for (u64 x = 0; x < q.bytes; x++) { out[q.item][q.outOff + x] = scratch[q.from + x]; cover[q.item][q.outOff + x]++; }
    }
    // every byte of every item written exactly once (no overlap within a dst), with the model's content
    for (size_t i = 0; i < n; i++) {
        itemsChecked++;
        size_t wrong = 0;
        for (u64 x = 0; x < out[i].size(); x++) wrong += cover[i][x] != 1 || out[i][x] != model(keyStream[streamOf[i]], offset[i] + x);
        CHECK(wrong == 0);
    }
    // random failing frames: an item fails exactly when it touches one, with the error of the first in stream order; a frame of the
    // wrong size is corruption_detected
    for (int rep = 0; rep < 4; rep++) {
        std::vector<size_t> dres(p.decodes.size());
        for (size_t id = 0; id < dres.size(); id++) {
            const int r = (int)rndIn(0, rep == 0 ? 0 : 6);
            dres[id] = r == 1 ? ZL_ERROR(checksum_wrong) : r == 2 ? ZL_ERROR(corruption_detected) : r == 3 ? ZL_ERROR(GENERIC)
                     : r == 4 ? (size_t)p.decodes[id].size + 1 : p.decodes[id].size;
        }
        std::vector<size_t> result(n);
        zl_ranges_results(p, dres.data(), result.data(), n);
        for (size_t i = 0; i < n; i++) {
            size_t want = p.result[i];
            for (size_t j = p.touchStart[i]; j < p.touchStart[i + 1]; j++) {
                const size_t r = dres[p.touch[j]];
                if (zl_is_error(r)) { want = r; break; }
                if (r != p.decodes[p.touch[j]].size) { want = ZL_ERROR(corruption_detected); break; }
            }
            CHECK(result[i] == want);
            if (rep == 0) CHECK(result[i] == p.result[i]);
        }
    }
}

// a hand-made case: three ranges over frames of 100 bytes, two sharing frame 1, one covering frame 3 whole
static void fixed()
{
    const std::vector<u8> b = makeStream({20, 20, 20, 20, 20}, {100, 100, 100, 100, 100}, false, false);
    std::vector<ZlSeekTable> t(1);
    std::vector<size_t> err(1, parse(t[0], b));
    CHECK(err[0] == 0);
    const size_t streamOf[3] = {0, 0, 0}, off[3] = {50, 150, 290}, len[3] = {100, 30, 120}, cap[3] = {100, 30, 120};
    void* dst[3] = {(void*)16, (void*)32, (void*)48};
    ZlRangesPlan p;
    zl_ranges_plan(p, t, err, streamOf, off, len, dst, cap, 3);
    // frames 0, 1 (shared by items 0 and 1), 2, 3 (item 2 covers it), 4 (item 2, partly)
    CHECK(p.decodes.size() == 5 && p.result[0] == 100 && p.result[1] == 30 && p.result[2] == 120);
    CHECK(p.decodes[0].item == ZL_RANGE_SCRATCH && p.decodes[1].item == ZL_RANGE_SCRATCH && p.decodes[2].item == ZL_RANGE_SCRATCH);
    CHECK(p.decodes[3].item == 2 && p.decodes[3].place == 10 && p.decodes[4].item == ZL_RANGE_SCRATCH);
    CHECK(p.scratchBytes == 4 * 112 && p.pieces.size() == 5);
}

int main()
{
    fixed();
    for (int it = 0; it < 3000; it++) checkCall(it);
    printf("plans %zu, items %zu, shared frames %zu, direct frames %zu, pieces %zu\n", plansChecked, itemsChecked, sharedSeen, directSeen, piecesSeen);
    CHECK(sharedSeen > 100 && directSeen > 100 && piecesSeen > 100);
    printf("bad=%d\n", bad);
    return bad ? 1 : 0;
}
