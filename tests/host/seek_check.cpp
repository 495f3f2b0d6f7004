// Test infrastructure: checks the seek table and range plan of seekable streams (zstdlite_b200/csrc/zl_seek.h) on the CPU -- tables written
// and parsed back, every malformed table rejected, and range plans over seeded random frame-size lists (zero-size frames included) checked
// against a byte-by-byte model of the decode.  Built and run by tests/test_seek_plan.py; no CUDA call is made.
#include "zl_seek.h"
#include <cstdio>
#include <vector>

static int bad = 0;
#define CHECK(c) do { if (!(c)) { if (bad++ < 20) printf("FAIL line %d: %s\n", __LINE__, #c); } } while (0)

static unsigned long long rngState = 88172645463325252ull;
static unsigned long long rnd() { rngState ^= rngState << 13; rngState ^= rngState >> 7; rngState ^= rngState << 17; return rngState; }
static size_t rndIn(size_t lo, size_t hi) { return lo + (size_t)(rnd() % (hi - lo + 1)); }

// a stream of n made-up frames (cSize[i] bytes of filler each) and its seek table
struct Stream {
    std::vector<u32> cSize, dSize, sums;
    std::vector<u8> bytes;
    size_t tableSize = 0;
    Stream(const std::vector<u32>& c, const std::vector<u32>& d, bool ck) : cSize(c), dSize(d)
    {
        if (ck) for (size_t i = 0; i < c.size(); i++) sums.push_back((u32)rnd());
        for (size_t i = 0; i < c.size(); i++) bytes.insert(bytes.end(), c[i], (u8)i);
        tableSize = zl_seek_table_size(c.size(), ck);
        const size_t at = bytes.size();
        bytes.resize(at + tableSize);
        zl_seek_write(bytes.data() + at, c.size(), c.data(), d.data(), ck ? sums.data() : nullptr);
    }
    size_t parse(ZlSeekTable& t) const
    {
        u32 n = 0; bool ck = false;
        const size_t tail = bytes.size() < ZL_SEEK_FOOTER ? bytes.size() : ZL_SEEK_FOOTER;
        const size_t size = zl_seek_footer(bytes.data() + bytes.size() - tail, bytes.size(), &n, &ck);
        if (zl_is_error(size)) return size;
        return zl_seek_parse(t, bytes.data() + bytes.size() - size, size, bytes.size());
    }
};

static void roundTrips()
{
    for (int it = 0; it < 200; it++) {
        const size_t n = it == 0 ? 0 : rndIn(1, 300);
        const bool ck = it & 1;
        std::vector<u32> c(n), d(n);
        for (size_t i = 0; i < n; i++) { c[i] = (u32)rndIn(9, 200); d[i] = rnd() % 5 == 0 ? 0u : (u32)rnd(); }
        const Stream s(c, d, ck);
        ZlSeekTable t;
        CHECK(s.parse(t) == 0);
        CHECK(t.n == n && t.checksums == ck && t.cSize == c && t.dSize == d && (!ck || t.checksum == s.sums));
        CHECK(s.tableSize == 8 + n * (ck ? 12 : 8) + 9 && t.cOff.size() == n + 1 && t.dOff.size() == n + 1);
        u64 co = 0, dof = 0;
        for (size_t i = 0; i < n; i++) { CHECK(t.cOff[i] == co && t.dOff[i] == dof); co += c[i]; dof += d[i]; }
        CHECK(t.cOff[n] == co && t.dOff[n] == dof && co + s.tableSize == s.bytes.size());
        // the table frame is a skippable frame of Frame_Size bytes after its 8-byte header
        const u8* tf = s.bytes.data() + co;
        CHECK(zl_rd32(tf) == 0x184D2A5Eu && zl_rd32(tf + 4) == s.tableSize - 8);
        CHECK(zl_rd32(s.bytes.data() + s.bytes.size() - 4) == 0x8F92EAB1u && s.bytes[s.bytes.size() - 5] == (ck ? 0x80 : 0));
    }
}

static void rejects()
{
    const Stream good({100, 50, 75}, {1000, 0, 3000}, true);
    ZlSeekTable t;
    CHECK(good.parse(t) == 0);
    const size_t N = good.bytes.size();
    auto with = [&](size_t at, u8 v) { Stream s = good; s.bytes[at] = v; return s; };
    auto word = [&](size_t at, u32 v) { Stream s = good; zl_seek_wr32(s.bytes.data() + at, v); return s; };
    // seekable magic
    CHECK(with(N - 1, 0x00).parse(t) == ZL_ERROR(prefix_unknown));
    CHECK(with(N - 4, 0xB0).parse(t) == ZL_ERROR(prefix_unknown));
    // reserved descriptor bits 6-2, each
    for (int b = 2; b <= 6; b++) CHECK(with(N - 5, (u8)(0x80 | (1 << b))).parse(t) == ZL_ERROR(corruption_detected));
    CHECK(with(N - 5, 0x81).parse(t) == 0 && with(N - 5, 0x82).parse(t) == 0);    // bits 1-0 are unused, not reserved
    // Number_Of_Frames that does not match Frame_Size (or the stream)
    CHECK(word(N - 9, 2).parse(t) == ZL_ERROR(corruption_detected));
    CHECK(word(N - 9, 4).parse(t) == ZL_ERROR(corruption_detected));
    CHECK(word(N - 9, 1000).parse(t) == ZL_ERROR(corruption_detected));
    // Frame_Size, and the skippable magic of the table frame
    CHECK(word(225 + 4, 44).parse(t) == ZL_ERROR(corruption_detected));
    CHECK(word(225 + 4, 46).parse(t) == ZL_ERROR(corruption_detected));
    CHECK(word(225, 0x184D2A50u).parse(t) == ZL_ERROR(corruption_detected));
    // the checksum flag changes the entry size: the same bytes no longer add up
    CHECK(with(N - 5, 0x00).parse(t) == ZL_ERROR(corruption_detected));
    // Compressed_Size values that do not add up to the stream's length
    CHECK(word(225 + 8, 101).parse(t) == ZL_ERROR(corruption_detected));
    CHECK(word(225 + 8, 99).parse(t) == ZL_ERROR(corruption_detected));
    { Stream s = good; s.bytes.insert(s.bytes.begin(), 0); CHECK(s.parse(t) == ZL_ERROR(corruption_detected)); }
    { Stream s = good; s.bytes.erase(s.bytes.begin()); CHECK(s.parse(t) == ZL_ERROR(corruption_detected)); }
    // truncated: a footer of fewer than 9 bytes, a table cut short
    for (size_t keep = 0; keep < 9; keep++) {
        Stream s = good; s.bytes.erase(s.bytes.begin(), s.bytes.end() - keep);
        CHECK(zl_is_error(s.parse(t)));
        if (keep >= 4) CHECK(s.parse(t) == ZL_ERROR(corruption_detected));
    }
    { Stream s = good; s.bytes.erase(s.bytes.begin(), s.bytes.end() - 20); CHECK(s.parse(t) == ZL_ERROR(corruption_detected)); }
    // N > 0x8000000, and N = 0x8000000 with too few bytes
    CHECK(word(N - 9, 0x8000001u).parse(t) == ZL_ERROR(corruption_detected));
    CHECK(word(N - 9, 0xFFFFFFFFu).parse(t) == ZL_ERROR(corruption_detected));
    CHECK(word(N - 9, 0x8000000u).parse(t) == ZL_ERROR(corruption_detected));
    // a stream that is only a table of 0 frames is well-formed, with nothing to read
    const Stream empty({}, {}, false);
    CHECK(empty.parse(t) == 0 && t.n == 0 && t.dOff[0] == 0);
    ZlSeekPlan p;
    CHECK(zl_seek_plan_range(p, t, 0, 10) == 0 && p.bytes == 0 && p.first == p.last);
    CHECK(zl_seek_plan_range(p, t, 1, 0) == ZL_ERROR(parameter_outOfBound));
}

// The plan against a model: frame f's content is the bytes dOff[f] .. dOff[f + 1] - 1 of the stream (as u32 values); decoding the planned
// frames into dst / scratch and copying the edges must give exactly bytes [offset, offset + bytes).
static void checkPlan(const ZlSeekTable& t, u64 offset, u64 length)
{
    const u64 total = t.dOff[t.n];
    ZlSeekPlan p;
    const size_t r = zl_seek_plan_range(p, t, offset, length);
    if (offset > total) { CHECK(r == ZL_ERROR(parameter_outOfBound)); return; }
    CHECK(r == 0);
    const u64 want = length < total - offset ? length : total - offset;
    CHECK(p.bytes == want);
    if (!want) { CHECK(p.first == p.last && p.nEdges == 0 && p.place.empty()); return; }
    const u64 end = offset + want;
    CHECK(p.first < p.last && p.last <= t.n && p.place.size() == p.last - p.first && p.edge.size() == p.place.size());
    // exactly the frames between the first and the last that hold a byte of the range
    for (size_t f = 0; f < t.n; f++) {
        const bool overlaps = t.dOff[f] < end && t.dOff[f + 1] > offset;
        if (overlaps) CHECK(f >= p.first && f < p.last);
        else if (t.dSize[f]) CHECK(f < p.first || f >= p.last);
    }
    CHECK(t.dSize[p.first] && t.dSize[p.last - 1]);
    std::vector<u32> out(want, 0xFFFFFFFFu), scratch(p.scratchBytes, 0xFFFFFFFFu);
    size_t edges = 0;
    for (size_t j = 0; j < p.place.size(); j++) {
        const size_t f = p.first + j;
        const bool edge = t.dOff[f] < offset || t.dOff[f + 1] > end;
        CHECK(p.edge[j] == (edge && t.dSize[f] ? 1 : 0));
        if (p.edge[j]) {
            CHECK((f == p.first || f == p.last - 1) && edges < p.nEdges && p.edges[edges].frame == f && p.edges[edges].scratchOff == p.place[j]);
            edges++;
            CHECK(p.place[j] + t.dSize[f] <= p.scratchBytes && p.place[j] % 16 == 0);
            if (p.place[j] + t.dSize[f] > p.scratchBytes) continue;
            for (u32 k = 0; k < t.dSize[f]; k++) scratch[p.place[j] + k] = (u32)(t.dOff[f] + k);
        } else {
            CHECK(p.place[j] + t.dSize[f] <= want);
            if (p.place[j] + t.dSize[f] > want) continue;
            for (u32 k = 0; k < t.dSize[f]; k++) out[p.place[j] + k] = (u32)(t.dOff[f] + k);
        }
    }
    CHECK(edges == p.nEdges && p.nEdges <= 2);
    for (size_t k = 0; k < p.nEdges; k++) {
        const ZlSeekEdge& e = p.edges[k];
        CHECK(e.skip + e.take <= t.dSize[e.frame] && e.outOff + e.take <= want && e.take > 0);
        if (e.skip + e.take > t.dSize[e.frame] || e.outOff + e.take > want) continue;
        for (u64 i = 0; i < e.take; i++) out[e.outOff + i] = scratch[e.scratchOff + e.skip + i];
    }
    size_t wrong = 0;
    for (u64 i = 0; i < want; i++) wrong += out[i] != (u32)(offset + i);
    CHECK(wrong == 0);
}

static void rangePlans()
{
    size_t plans = 0;
    for (int it = 0; it < 60; it++) {
        const size_t n = rndIn(1, it < 10 ? 4 : 40);
        std::vector<u32> c(n, 20), d(n);
        for (size_t i = 0; i < n; i++) d[i] = rnd() % 4 == 0 ? 0u : (u32)rndIn(1, it % 3 == 0 ? 3 : 300);
        if (it % 7 == 0) d[0] = 0;
        if (it % 5 == 0) d[n - 1] = 0;
        const Stream s(c, d, it & 1);
        ZlSeekTable t;
        CHECK(s.parse(t) == 0);
        const u64 total = t.dOff[n];
        std::vector<u64> offs = {0, total, total + 1, total / 2, total + 1000};
        for (size_t f = 0; f <= n; f++) for (int dd = -1; dd <= 1; dd++) if (t.dOff[f] + dd <= total + 1) offs.push_back(t.dOff[f] + dd);
        for (size_t f = 0; f < n; f++) if (d[f] > 2) offs.push_back(t.dOff[f] + d[f] / 2);
        for (u64 off : offs) {
            std::vector<u64> lens = {0, 1, 2, total - (off < total ? off : total), total + 5, ~0ull, rndIn(1, 50), rndIn(1, 1000)};
            for (size_t f = 0; f <= n; f++) if (t.dOff[f] > off) { lens.push_back(t.dOff[f] - off); lens.push_back(t.dOff[f] - off + 1); }
            for (u64 len : lens) { checkPlan(t, off, len); plans++; }
        }
    }
    printf("range plans checked: %zu\n", plans);
}

int main()
{
    roundTrips();
    rejects();
    rangePlans();
    printf("bad=%d\n", bad);
    return bad ? 1 : 0;
}
