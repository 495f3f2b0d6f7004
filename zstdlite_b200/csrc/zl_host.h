// zl_host.h -- host-side helpers shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <string.h>
#include <vector>
#include <thread>
#include <mutex>
#include <condition_variable>
#include <atomic>
#include <functional>
#if defined(__linux__)
#include <sched.h>
#endif
#if defined(__x86_64__) || defined(_M_X64)
#include <emmintrin.h>
#define ZL_HAVE_STREAM_COPY 1
#endif
#include "zl_common.cuh"
#include "zl_launch.h"

#define ZL_ERROR(name) ((size_t)0 - (size_t)ZL_E_##name)
static inline bool zl_is_error(size_t r) { return r > (size_t)0 - (size_t)ZL_E_maxCode; }

// grow-only device / pinned-host buffers owned by a context
struct ZlDevBuf {
    void* p = nullptr;
    size_t cap = 0;
    bool reserve(size_t n)
    {
        if (n <= cap) return true;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = n + (n >> 3) + 4096;
        want = (want + 0xFFFFF) & ~(size_t)0xFFFFF;
        if (cudaMalloc(&p, want) != cudaSuccess) { (void)cudaGetLastError(); if (cudaMalloc(&p, n + 256) != cudaSuccess) { (void)cudaGetLastError(); p = nullptr; return false; } want = n + 256; }
        cap = want;
        return true;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};
struct ZlPinBuf {
    void* p = nullptr;
    size_t cap = 0;
    bool reserve(size_t n)
    {
        if (n <= cap) return true;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = n + (n >> 2) + 4096;
        if (cudaMallocHost(&p, want) != cudaSuccess) { (void)cudaGetLastError(); p = nullptr; return false; }
        cap = want;
        return true;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// host copy of the frame header logic (zstd.c:41050-41152); returns 0, an error, or bytes wanted
struct ZlHostFrameHeader {
    unsigned long long contentSize, windowSize;
    unsigned blockSizeMax, skippable, headerSize, dictID, checksumFlag;
};
size_t zl_host_frame_header(ZlHostFrameHeader* h, const void* src, size_t srcSize);
size_t zl_host_find_frame_size(const void* src, size_t srcSize, unsigned* nblocksOut);

// ---- host copy pool ---------------------------------------------------------------------------------------------------
// The reference's C layer hands over PAGEABLE memory (R vectors: src/raw-file.c:166,189).  cudaMemcpyAsync on such memory goes
// through the driver's own staging, synchronously and on one thread (measured: 8.4 GB/s for config 2 end to end against 41 GB/s
// with pinned buffers).  The library stages pageable and scattered buffers through its own pinned memory instead and moves the
// bytes with this pool: a few worker threads (ZL_COPY_THREADS, default 3/4 of the CPUs in the affinity mask, at most 16) that split a list of copies into
// 256 KiB pieces and pull them from a shared counter; the calling thread takes part.  Process-wide, created on first use.
struct ZlCopySeg { void* dst; const void* src; size_t bytes; };
// A piece of a staging copy: plain loads, NON-TEMPORAL stores.  Neither side of these copies is read again by this core -- packed input is
// fetched from DRAM by the copy engine, unpacked output is a gigabyte the caller reads later -- and a 256 KiB memcpy stays below glibc's
// non-temporal threshold, so every destination line was first read for ownership: three DRAM transfers per byte instead of two, with eight
// threads sharing the memory controllers (measured on the development host, 1 GiB in 256 KiB pieces: memcpy 16 - 23 GB/s, this 22 - 36 GB/s).
static inline void zl_copy_stream(void* dstv, const void* srcv, size_t n)
{
#ifdef ZL_HAVE_STREAM_COPY
    char* d = (char*)dstv; const char* s = (const char*)srcv;
    size_t head = (size_t)(16 - ((uintptr_t)d & 15)) & 15;
    if (head > n) head = n;
    memcpy(d, s, head); d += head; s += head; n -= head;
    size_t i = 0;
    for (; i + 128 <= n; i += 128) {
        const __m128i a0 = _mm_loadu_si128((const __m128i*)(s + i)), a1 = _mm_loadu_si128((const __m128i*)(s + i + 16));
        const __m128i a2 = _mm_loadu_si128((const __m128i*)(s + i + 32)), a3 = _mm_loadu_si128((const __m128i*)(s + i + 48));
        const __m128i a4 = _mm_loadu_si128((const __m128i*)(s + i + 64)), a5 = _mm_loadu_si128((const __m128i*)(s + i + 80));
        const __m128i a6 = _mm_loadu_si128((const __m128i*)(s + i + 96)), a7 = _mm_loadu_si128((const __m128i*)(s + i + 112));
        _mm_stream_si128((__m128i*)(d + i), a0); _mm_stream_si128((__m128i*)(d + i + 16), a1);
        _mm_stream_si128((__m128i*)(d + i + 32), a2); _mm_stream_si128((__m128i*)(d + i + 48), a3);
        _mm_stream_si128((__m128i*)(d + i + 64), a4); _mm_stream_si128((__m128i*)(d + i + 80), a5);
        _mm_stream_si128((__m128i*)(d + i + 96), a6); _mm_stream_si128((__m128i*)(d + i + 112), a7);
    }
    _mm_sfence();                                   // the stores are globally visible before the piece counts as done
    memcpy(d + i, s + i, n - i);
#else
    memcpy(dstv, srcv, n);
#endif
}
class ZlCopyPool {
public:
    static ZlCopyPool& get() { static ZlCopyPool p; return p; }
    void run(const std::vector<ZlCopySeg>& segs)
    {
        size_t total = 0;
        for (const ZlCopySeg& s : segs) total += s.bytes;
        if (total < (4u << 20) || workers_.empty()) { for (const ZlCopySeg& s : segs) if (s.bytes) memcpy(s.dst, s.src, s.bytes); return; }
        std::vector<ZlCopySeg> pieces;
        for (const ZlCopySeg& s : segs)
            for (size_t o = 0; o < s.bytes; o += kPiece) pieces.push_back({(char*)s.dst + o, (const char*)s.src + o, s.bytes - o < kPiece ? s.bytes - o : kPiece});
        static const bool plain = getenv("ZL_COPY_PLAIN") != nullptr;              // (development switch: memcpy instead of streaming stores)
        parallel(pieces.size(), [&](size_t i) { if (plain || pieces[i].bytes < 4096) memcpy(pieces[i].dst, pieces[i].src, pieces[i].bytes); else zl_copy_stream(pieces[i].dst, pieces[i].src, pieces[i].bytes); });
    }
    // fn(0) .. fn(n - 1) spread over the pool (and the caller); returns when all are done
    void parallel(size_t n, const std::function<void(size_t)>& fn)
    {
        if (n < 2 || workers_.empty()) { for (size_t i = 0; i < n; i++) fn(i); return; }
        std::lock_guard<std::mutex> serial(runMutex_);            // one job at a time (contexts on different threads share the pool)
        fn_ = &fn; count_ = n;
        next_.store(0); pending_.store((int)workers_.size());
        { std::lock_guard<std::mutex> g(m_); generation_++; }
        cv_.notify_all();
        work();
        std::unique_lock<std::mutex> g(m_);
        done_.wait(g, [&] { return pending_.load() == 0; });
    }
    unsigned threads() const { return (unsigned)workers_.size() + 1; }
private:
    static constexpr size_t kPiece = 256u << 10;
    ZlCopyPool()
    {
        // three quarters of the CPUs this process may run on (its affinity mask: a rank bound to its GPU's share of the box sizes the pool
        // for that share), at most 16.  Measured on a 16-core box, config 2 end to end with malloc'ed buffers: 4 threads 21.6, 8 threads
        // 25.6, 12 threads 27.8, 16 threads 28.3 GB/s.
        unsigned cpus = std::thread::hardware_concurrency();
#if defined(__linux__)
        { cpu_set_t set; CPU_ZERO(&set); if (sched_getaffinity(0, sizeof(set), &set) == 0 && CPU_COUNT(&set) > 0) cpus = (unsigned)CPU_COUNT(&set); }
#endif
        unsigned n = cpus - cpus / 4;
        if (n > 16) n = 16;
        if (const char* e = getenv("ZL_COPY_THREADS")) n = (unsigned)atoi(e);
        if (n < 1) n = 1;
        for (unsigned i = 1; i < n; i++) workers_.emplace_back([this] { loop(); });
    }
    ~ZlCopyPool()
    {
        { std::lock_guard<std::mutex> g(m_); stop_ = true; generation_++; }
        cv_.notify_all();
        for (std::thread& t : workers_) t.join();
    }
    void work()
    {
        for (;;) {
            const size_t i = next_.fetch_add(1);
            if (i >= count_) break;
            (*fn_)(i);
        }
    }
    void loop()
    {
        unsigned long long seen = 0;
        for (;;) {
            { std::unique_lock<std::mutex> g(m_); cv_.wait(g, [&] { return generation_ != seen; }); seen = generation_; if (stop_) return; }
            work();
            if (pending_.fetch_sub(1) == 1) { std::lock_guard<std::mutex> g(m_); done_.notify_all(); }
        }
    }
    std::vector<std::thread> workers_;
    const std::function<void(size_t)>* fn_ = nullptr;
    size_t count_ = 0;
    std::atomic<size_t> next_{0};
    std::atomic<int> pending_{0};
    std::mutex m_, runMutex_;
    std::condition_variable cv_, done_;
    unsigned long long generation_ = 0;
    bool stop_ = false;
};
// true when `p` is ordinary (pageable) host memory: not pinned, not registered, not managed
static inline bool zl_is_pageable(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

// Pinned staging shared by every context of the process, one pool per device (the reference creates a fresh context per call --
// src/raw-file.c:150-189 -- and pinning memory costs ~0.3 s per GB, more than the decode it would serve): grow-only, borrowed
// under a lock for one call.
struct ZlStagePool {
    std::mutex m;
    ZlPinBuf in, out;
    static ZlStagePool& get()
    {
        static ZlStagePool pools[64];
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { (void)cudaGetLastError(); dev = 0; }
        return pools[dev];
    }
};

// ---- devices --------------------------------------------------------------------------------------------------------------
// A context belongs to the device that was current when it was first used; every entry point switches to it and back.
struct ZlDeviceGuard {
    int prev = -1; bool ok = true;
    explicit ZlDeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { (void)cudaGetLastError(); prev = -1; ok = false; return; }
        if (dev >= 0 && dev != prev) ok = cudaSetDevice(dev) == cudaSuccess;
        else prev = -1;                                                // nothing to restore
    }
    ~ZlDeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
static inline int zl_bind_device(int* device)                           // -> the context's device (bound on first use)
{
    if (*device < 0 && cudaGetDevice(device) != cudaSuccess) { (void)cudaGetLastError(); *device = 0; }
    return *device;
}
// GPUs a context may spread a batch of host buffers over: `asked` (0: the ZSTDLITE_GPUS environment variable, default 1; "all" or a
// number), never more than the visible devices
static inline int zl_gpu_count(int asked)
{
    int have = 0;
    if (cudaGetDeviceCount(&have) != cudaSuccess) { (void)cudaGetLastError(); return 1; }
    if (asked <= 0) {
        const char* e = getenv("ZSTDLITE_GPUS");
        asked = !e ? 1 : (!strcmp(e, "all") ? have : atoi(e));
    }
    if (asked < 1) asked = 1;
    return asked < have ? asked : (have > 0 ? have : 1);
}
// contiguous ranges of [0, n) of about equal weight: cut[0] = 0 .. cut[parts] = n
static inline std::vector<size_t> zl_split_ranges(const size_t* weight, size_t n, size_t parts)
{
    std::vector<size_t> cut(parts + 1, n);
    unsigned long long total = 0, acc = 0;
    for (size_t i = 0; i < n; i++) total += weight[i] + 64;
    cut[0] = 0;
    size_t k = 1;
    for (size_t i = 0; i < n && k < parts; i++) {
        acc += weight[i] + 64;
        if (acc * parts >= total * k) cut[k++] = i + 1;
    }
    return cut;
}
