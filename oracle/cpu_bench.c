/*
 * cpu_bench.c -- TEST / BENCH INFRASTRUCTURE ONLY.  Never linked into the product.
 *
 * Frame-parallel CPU baseline over the system's libzstd (libzstd.so.1, linked by oracle/Makefile;
 * the reference vendors the same library at 1.5.6).  No interpreter in the timed
 * region: bench.py hands over packed buffers through ctypes and gets seconds back.
 *
 * Mirrors the reference's call sequences per frame:
 *   decompress  src/raw-file.c:180-189  (ZSTD_createDCtx once per thread, ZSTD_decompressDCtx per frame)
 *   compress    src/raw-file.c:65-74    (ZSTD_createCCtx + level/checksum parameters, ZSTD_compress2)
 * `threads` workers each own a context and pull frames from a shared atomic counter
 * (BASELINE.md section 3, item 3: "frame-parallel x cores"; threads = 1 is item 1).
 * zlb_run_workers is item 2, the reference's own num_threads semantics: ONE frame, ZSTD_c_nbWorkers = n
 * (src/cctx.c:269-277; libzstd only engages its workers above 512 KB of input, zstd.c:28773).
 */
#include <pthread.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

/* prototypes of the libzstd symbols used (src/zstd/zstd.h) */
typedef struct ZSTD_CCtx_s ZSTD_CCtx;
typedef struct ZSTD_DCtx_s ZSTD_DCtx;
ZSTD_CCtx* ZSTD_createCCtx(void);
size_t ZSTD_freeCCtx(ZSTD_CCtx*);
ZSTD_DCtx* ZSTD_createDCtx(void);
size_t ZSTD_freeDCtx(ZSTD_DCtx*);
size_t ZSTD_CCtx_setParameter(ZSTD_CCtx*, int, int);
size_t ZSTD_CCtx_loadDictionary(ZSTD_CCtx*, const void*, size_t);
size_t ZSTD_DCtx_loadDictionary(ZSTD_DCtx*, const void*, size_t);
size_t ZSTD_compress2(ZSTD_CCtx*, void*, size_t, const void*, size_t);
size_t ZSTD_decompressDCtx(ZSTD_DCtx*, void*, size_t, const void*, size_t);
unsigned ZSTD_isError(size_t);

typedef struct {
    int mode;                 /* 0 decompress, 1 compress */
    const uint8_t* src; const size_t* srcOff; const size_t* srcSize;
    uint8_t* dst; const size_t* dstOff; const size_t* dstCap;
    size_t* result; size_t n;
    int level, checksum;
    const void* dict; size_t dictSize;
    volatile size_t next;
    volatile int errors;
    pthread_barrier_t* start;
    double* tBeg; double* tEnd;      /* per-worker timestamps: the pass lasts from the first start to the last end */
    volatile int nextId;
} job_t;

static double now_s(void)
{
    struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t);
    return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec;
}

static void* worker(void* arg)
{
    job_t* j = (job_t*)arg;
    ZSTD_CCtx* c = NULL; ZSTD_DCtx* d = NULL;
    if (j->mode) {
        c = ZSTD_createCCtx();
        ZSTD_CCtx_setParameter(c, 100, j->level);        /* ZSTD_c_compressionLevel */
        ZSTD_CCtx_setParameter(c, 201, j->checksum);     /* ZSTD_c_checksumFlag */
        if (j->dict) ZSTD_CCtx_loadDictionary(c, j->dict, j->dictSize);
    } else {
        d = ZSTD_createDCtx();
        if (j->dict) ZSTD_DCtx_loadDictionary(d, j->dict, j->dictSize);
    }
    const int id = __sync_fetch_and_add(&j->nextId, 1);
    pthread_barrier_wait(j->start);
    j->tBeg[id] = now_s();
    for (;;) {
        size_t i = __sync_fetch_and_add(&j->next, (size_t)16);      /* 16 frames per grab */
        if (i >= j->n) break;
        size_t e = i + 16 < j->n ? i + 16 : j->n;
        for (; i < e; i++) {
            size_t r = j->mode ? ZSTD_compress2(c, j->dst + j->dstOff[i], j->dstCap[i], j->src + j->srcOff[i], j->srcSize[i])
                               : ZSTD_decompressDCtx(d, j->dst + j->dstOff[i], j->dstCap[i], j->src + j->srcOff[i], j->srcSize[i]);
            if (ZSTD_isError(r)) __sync_fetch_and_add(&j->errors, 1);
            if (j->result) j->result[i] = r;
        }
    }
    j->tEnd[id] = now_s();
    pthread_barrier_wait(j->start);
    if (c) ZSTD_freeCCtx(c);
    if (d) ZSTD_freeDCtx(d);
    return NULL;
}

/* One timed pass over all n frames with `threads` workers; returns seconds (contexts are created outside the
 * timed region, which runs from the first worker's start to the last worker's end), or -1 on error. */
double zlb_run(int mode, const void* src, const size_t* srcOff, const size_t* srcSize, void* dst, const size_t* dstOff,
               const size_t* dstCap, size_t* result, size_t n, int level, int checksum, const void* dict, size_t dictSize,
               int threads)
{
    if (threads < 1) threads = 1;
    pthread_barrier_t bar;
    pthread_barrier_init(&bar, NULL, (unsigned)threads + 1);
    job_t j;
    memset(&j, 0, sizeof(j));
    j.mode = mode; j.src = (const uint8_t*)src; j.srcOff = srcOff; j.srcSize = srcSize; j.dst = (uint8_t*)dst;
    j.dstOff = dstOff; j.dstCap = dstCap; j.result = result; j.n = n; j.level = level; j.checksum = checksum;
    j.dict = dictSize ? dict : NULL; j.dictSize = dictSize; j.start = &bar;
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)threads);
    j.tBeg = (double*)calloc((size_t)threads, sizeof(double)); j.tEnd = (double*)calloc((size_t)threads, sizeof(double));
    for (int t = 0; t < threads; t++) pthread_create(&th[t], NULL, worker, &j);
    pthread_barrier_wait(&bar);
    pthread_barrier_wait(&bar);
    for (int t = 0; t < threads; t++) pthread_join(th[t], NULL);
    double t0 = j.tBeg[0], t1 = j.tEnd[0];
    for (int t = 1; t < threads; t++) { if (j.tBeg[t] < t0) t0 = j.tBeg[t]; if (j.tEnd[t] > t1) t1 = j.tEnd[t]; }
    free(j.tBeg); free(j.tEnd);
    free(th);
    pthread_barrier_destroy(&bar);
    return j.errors ? -1.0 : (t1 - t0);
}

/* One buffer -> ONE frame with ZSTD_c_nbWorkers = workers (0: single-threaded ZSTD_compress2), `passes` times; returns the
 * best seconds and the frame size through *outSize, or -1 on error. */
double zlb_run_workers(const void* src, size_t srcSize, void* dst, size_t dstCap, int level, int workers, int passes, size_t* outSize)
{
    ZSTD_CCtx* c = ZSTD_createCCtx();
    if (!c) return -1.0;
    ZSTD_CCtx_setParameter(c, 100, level);               /* ZSTD_c_compressionLevel */
    if (workers > 1 && ZSTD_isError(ZSTD_CCtx_setParameter(c, 400, workers))) { ZSTD_freeCCtx(c); return -1.0; }   /* ZSTD_c_nbWorkers */
    double best = -1.0;
    for (int p = 0; p < passes; p++) {
        const double t0 = now_s();
        const size_t r = ZSTD_compress2(c, dst, dstCap, src, srcSize);
        const double t = now_s() - t0;
        if (ZSTD_isError(r)) { ZSTD_freeCCtx(c); return -1.0; }
        if (outSize) *outSize = r;
        if (best < 0 || t < best) best = t;
    }
    ZSTD_freeCCtx(c);
    return best;
}
