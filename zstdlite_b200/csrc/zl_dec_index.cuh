// zl_dec_index.cuh -- the frame index of a stream in device memory (zl_stream_index.h has the algorithm and the per-thread bodies):
//   zl_k_idx_count / zl_k_idx_scan / zl_k_idx_write   I1: candidates per 64 KiB tile, one scan, then the sorted candidate list
//   zl_k_idx_extent                                   I2: a thread per candidate, at most ZL_IDX_W block steps
//   zl_k_idx_jump                                     I3: one pointer-jumping pass over double-buffered jump arrays
//   zl_k_idx_frontier                                 one thread: the chain's LONG candidate without a cap (or the rest of the chain)
//   zl_k_idx_mark_count / zl_k_idx_scan / zl_k_idx_mark_write   I4: the marked candidates as frame records, and the chain's status
// Loads stay inside the 16-byte-aligned chunks that hold bytes of the stream.
#pragma once
#include "zl_stream_index.h"

#define ZL_IDX_SCAN_THREADS 1024u

// exclusive scan of one value per thread over a CTA of blockDim.x (a multiple of 32, at most 1024) threads; *total: the sum
template <class T>
static __device__ __forceinline__ T zl_idx_block_scan(T v, T* sh, T* total)
{
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    T x = v;
    for (u32 d = 1; d < 32; d <<= 1) { const T y = __shfl_up_sync(0xFFFFFFFFu, x, d); if (lane >= d) x += y; }
    if (lane == 31) sh[warp] = x;
    __syncthreads();
    if (warp == 0) {
        T s = lane < nw ? sh[lane] : (T)0;
        for (u32 d = 1; d < 32; d <<= 1) { const T y = __shfl_up_sync(0xFFFFFFFFu, s, d); if (lane >= d) s += y; }
        if (lane < nw) sh[lane] = s;
    }
    __syncthreads();
    const T before = (warp ? sh[warp - 1] : (T)0) + x - v;
    *total = sh[nw - 1];
    __syncthreads();                                               // (sh is reused by the caller's next scan)
    return before;
}

// I1: the candidate mask of chunk c (16 bytes at the aligned address base + 16c, base = src rounded down to 16; head = src - base)
static __device__ __forceinline__ u32 zl_idx_chunk(const u8* base, u64 head, u64 srcSize, u64 c)
{
    const u64 lastChunk = (head + srcSize - 1) >> 4;
    if (c > lastChunk) return 0;
    u32 w[8];
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(base) + c);
    const uint4 b = c < lastChunk ? __ldg(reinterpret_cast<const uint4*>(base) + c + 1) : make_uint4(0, 0, 0, 0);
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
    const i64 at = (i64)(c << 4) - (i64)head;                      // stream offset of the chunk's first byte
    const i64 lo = -at, hi = (i64)srcSize - 4 - at;
    return zl_idx_chunk_mask(w, lo < 0 ? 0 : (lo > 16 ? 16 : (int)lo), hi > 15 ? 15 : (hi < -1 ? -1 : (int)hi));
}
__global__ void __launch_bounds__(ZL_IDX_TILE_THREADS)
zl_k_idx_count(const u8* __restrict__ base, u64 head, u64 srcSize, u32* __restrict__ tileCount)
{
    __shared__ u32 sh[32];
    u32 cnt = 0;
    for (u32 j = 0; j < ZL_IDX_TILE_CHUNKS; j++)
        cnt += __popc(zl_idx_chunk(base, head, srcSize, ((u64)blockIdx.x * ZL_IDX_TILE_CHUNKS + j) * ZL_IDX_TILE_THREADS + threadIdx.x));
    u32 total;
    zl_idx_block_scan<u32>(cnt, sh, &total);
    if (threadIdx.x == 0) tileCount[blockIdx.x] = total;
}
__global__ void __launch_bounds__(ZL_IDX_TILE_THREADS)
zl_k_idx_write(const u8* __restrict__ base, u64 head, u64 srcSize, const u64* __restrict__ tileOff, u64* __restrict__ cand)
{
    __shared__ u32 sh[32];
    u64 at = tileOff[blockIdx.x];
    for (u32 j = 0; j < ZL_IDX_TILE_CHUNKS; j++) {
        const u64 c = ((u64)blockIdx.x * ZL_IDX_TILE_CHUNKS + j) * ZL_IDX_TILE_THREADS + threadIdx.x;
        u32 m = zl_idx_chunk(base, head, srcSize, c), total;
        u64 w = at + zl_idx_block_scan<u32>(__popc(m), sh, &total);
        while (m) { const u32 q = __ffs(m) - 1; m &= m - 1; cand[w++] = (c << 4) + q - head; }
        at += total;
    }
}
// one CTA: off[i] = count[0] + ... + count[i - 1] for i <= n
__global__ void __launch_bounds__(ZL_IDX_SCAN_THREADS)
zl_k_idx_scan(const u32* __restrict__ count, u64 n, u64* __restrict__ off)
{
    __shared__ u64 sh[32];
    const u64 seg = (n + ZL_IDX_SCAN_THREADS - 1) / ZL_IDX_SCAN_THREADS, a = min(n, threadIdx.x * seg), b = min(n, a + seg);
    u64 s = 0;
    for (u64 i = a; i < b; i++) s += count[i];
    u64 total;
    u64 at = zl_idx_block_scan<u64>(s, sh, &total);
    for (u64 i = a; i < b; i++) { off[i] = at; at += count[i]; }
    if (threadIdx.x == 0) off[n] = total;
}

// I2; also seeds the marks: candidate 0 when it is at offset 0
__global__ void __launch_bounds__(128)
zl_k_idx_extent(const u8* __restrict__ src, u64 srcSize, const u64* __restrict__ cand, u32 n, u32 cap, u32* __restrict__ link,
                u32* __restrict__ errc, u32* __restrict__ nblk, u32* __restrict__ mark)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    zl_idx_extent(src, srcSize, cand, n, i, cap, link, errc, nblk);
    mark[i] = i == 0 && cand[0] == 0 ? 1u : 0u;
}

// I3: pass `pass` of a round; open[pass] counts the marked candidates whose chain is not covered yet (0: the round is done)
__global__ void __launch_bounds__(256)
zl_k_idx_jump(u32 n, const u32* __restrict__ jin, u32* __restrict__ jout, u32* mark, u32* open, u32 pass)
{
    if (pass > 0 && *(volatile u32*)(open + pass - 1) == 0) return;
    const u32 v = blockIdx.x * blockDim.x + threadIdx.x;
    u32 o = v < n ? zl_idx_jump(v, jin, jout, mark) : 0u;
    o = __reduce_add_sync(0xFFFFFFFFu, o);
    if ((threadIdx.x & 31) == 0 && o) atomicAdd(open + pass, o);
}

// the chain's LONG candidate `status->tail`, walked without a cap; serial: and every candidate after it, marking each
__global__ void __launch_bounds__(32)
zl_k_idx_frontier(const u8* __restrict__ src, u64 srcSize, const u64* __restrict__ cand, u32 n, u32* link, u32* errc, u32* nblk, u32* mark,
                  const ZlIdxStatus* __restrict__ status, int serial)
{
    if (threadIdx.x) return;
    u32 v = status->tail;
    for (;;) {
        zl_idx_extent(src, srcSize, cand, n, v, 0, link, errc, nblk);
        const u32 j = link[v];
        if (!serial || j >= ZL_LINK_NODES) return;
        mark[j] = 1; v = j;
    }
}

// I4: frames per tile of ZL_IDX_TILE_NODES candidates; the chain's last candidate (marked, link not a node) and the first candidate's
// offset into *status
__global__ void __launch_bounds__(ZL_IDX_TILE_THREADS)
zl_k_idx_mark_count(const u64* __restrict__ cand, u32 n, const u32* __restrict__ link, const u32* __restrict__ errc, const u32* __restrict__ mark,
                    u32* __restrict__ tileCount, ZlIdxStatus* __restrict__ status)
{
    __shared__ u32 sh[32];
    u32 cnt = 0;
    for (u32 j = 0; j < ZL_IDX_TILE_NODES / ZL_IDX_TILE_THREADS; j++) {
        const u32 v = blockIdx.x * ZL_IDX_TILE_NODES + j * ZL_IDX_TILE_THREADS + threadIdx.x;
        if (v >= n || !mark[v]) continue;
        cnt += link[v] != ZL_LINK_BAD;
        if (link[v] >= ZL_LINK_NODES) { status->tail = v; status->link = link[v]; status->err = errc[v]; }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) status->first = cand[0];
    u32 total;
    zl_idx_block_scan<u32>(cnt, sh, &total);
    if (threadIdx.x == 0) tileCount[blockIdx.x] = total;
}
__global__ void __launch_bounds__(ZL_IDX_TILE_THREADS)
zl_k_idx_mark_write(const u8* __restrict__ src, u64 srcSize, const u64* __restrict__ cand, u32 n, const u32* __restrict__ link,
                    const u32* __restrict__ nblk, const u32* __restrict__ mark, const u64* __restrict__ tileOff, ZlStreamFrame* __restrict__ frames)
{
    __shared__ u32 sh[32];
    u64 at = tileOff[blockIdx.x];
    for (u32 j = 0; j < ZL_IDX_TILE_NODES / ZL_IDX_TILE_THREADS; j++) {
        const u32 v = blockIdx.x * ZL_IDX_TILE_NODES + j * ZL_IDX_TILE_THREADS + threadIdx.x;
        const u32 m = v < n && zl_idx_is_frame(mark, link, v) ? 1u : 0u;
        u32 total;
        const u64 w = at + zl_idx_block_scan<u32>(m, sh, &total);
        if (m) frames[w] = zl_idx_record(src, srcSize, cand, link, nblk, v);
        at += total;
    }
}

// ---- launchers (zl_launch.h) ----
cudaError_t zl_launch_idx_candidates(const u8* src, u64 srcSize, u32 tiles, u32* tileCount, u64* tileOff, u64* cand, cudaStream_t st)
{
    const u8* base = (const u8*)((size_t)src & ~(size_t)15);
    const u64 head = (u64)(src - base);
    if (!cand) {
        zl_k_idx_count<<<tiles, ZL_IDX_TILE_THREADS, 0, st>>>(base, head, srcSize, tileCount);
        zl_k_idx_scan<<<1, ZL_IDX_SCAN_THREADS, 0, st>>>(tileCount, tiles, tileOff);
    } else zl_k_idx_write<<<tiles, ZL_IDX_TILE_THREADS, 0, st>>>(base, head, srcSize, tileOff, cand);
    return cudaGetLastError();
}
cudaError_t zl_launch_idx_extent(const u8* src, u64 srcSize, const u64* cand, u32 n, u32 cap, u32* link, u32* errc, u32* nblk, u32* mark, cudaStream_t st)
{
    zl_k_idx_extent<<<(n + 127) / 128, 128, 0, st>>>(src, srcSize, cand, n, cap, link, errc, nblk, mark);
    return cudaGetLastError();
}
cudaError_t zl_launch_idx_jump(u32 n, u32* j0, u32* j1, u32* mark, u32* open, u32 pass0, u32 passes, cudaStream_t st)
{
    for (u32 p = pass0; p < pass0 + passes; p++)
        zl_k_idx_jump<<<(n + 255) / 256, 256, 0, st>>>(n, p & 1 ? j1 : j0, p & 1 ? j0 : j1, mark, open, p);
    return cudaGetLastError();
}
cudaError_t zl_launch_idx_frontier(const u8* src, u64 srcSize, const u64* cand, u32 n, u32* link, u32* errc, u32* nblk, u32* mark,
                                   const ZlIdxStatus* status, bool serial, cudaStream_t st)
{
    zl_k_idx_frontier<<<1, 32, 0, st>>>(src, srcSize, cand, n, link, errc, nblk, mark, status, serial ? 1 : 0);
    return cudaGetLastError();
}
cudaError_t zl_launch_idx_frames(const u8* src, u64 srcSize, const u64* cand, u32 n, const u32* link, const u32* errc, const u32* nblk,
                                 const u32* mark, u32 tiles, u32* tileCount, u64* tileOff, ZlIdxStatus* status, ZlStreamFrame* frames, cudaStream_t st)
{
    if (!frames) {
        zl_k_idx_mark_count<<<tiles, ZL_IDX_TILE_THREADS, 0, st>>>(cand, n, link, errc, mark, tileCount, status);
        zl_k_idx_scan<<<1, ZL_IDX_SCAN_THREADS, 0, st>>>(tileCount, tiles, tileOff);
    } else zl_k_idx_mark_write<<<tiles, ZL_IDX_TILE_THREADS, 0, st>>>(src, srcSize, cand, n, link, nblk, mark, tileOff, frames);
    return cudaGetLastError();
}
