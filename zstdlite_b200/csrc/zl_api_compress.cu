// zl_api_compress.cu -- compression half of the C ABI (include/zstdlite_gpu.h): ZSTD_CCtx lifecycle and parameters
// (call sites: /root/reference/src/cctx.c:205-312,352-354), ZSTD_compressBound / ZSTD_compress2 (src/raw-file.c:52,74;
// src/serialize.c:73,91), and the batch / split extensions.  All compute runs in the kernels of zl_enc_kernels.cu.  The host arithmetic
// of a batch (waves, parts, descriptors, placement of host buffers, gather tables, split chunks) is planned in zl_enc_plan.h; this file
// reserves the buffers and issues the copies and launches the plan describes.
#include <stdio.h>
#include <stdlib.h>
#include <new>
#include <chrono>
#include "../../include/zstdlite_gpu.h"
#include <thread>
#include "zl_enc_plan.h"
#include "zl_enc_dict.h"          // host-side dictionary digest (shared with the CPU emulation in tests/emul)

#define ZL_EXPORT extern "C" __attribute__((visibility("default")))
#define ZL_ALIAS(ret, name, params) extern "C" __attribute__((visibility("default"), alias(#name))) ret zlg_##name params;

#define ZL_MAX_SERVED_LEVEL 5           // levels 4 and 5: the level-3 engine, within 3 % of libzstd at those levels (ZSTD_c_compressionLevel below)

struct ZSTD_CCtx_s {
    int level = 3, nbWorkers = 0, checksumFlag = 0, stableIn = 0, stableOut = 0, windowLog = 0;
    bool levelFallback = false;            // zl_cctx_allow_level_fallback: levels >= 6 run the level-3 engine instead of being refused
    unsigned long long pledged = ZSTD_CONTENTSIZE_UNKNOWN;
    std::vector<u8> dictRaw;
    bool dictDirty = false;                // dictRaw changed (or the engine level did): digest again before the next compression
    int dictLevel = 0;                     // engine level the device tables were built for
    u32 dictID = 0;
    size_t dictErr = 0;                    // error found while digesting, reported by the compress calls (as libzstd does)
    ZlDevBuf dDict, dDictContent, dDictTabS, dDictTabL;
    cudaStream_t stream = nullptr;
    bool ownStream = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t stageEv[ZL_ENC_PARTS][ZL_ENC_STAGES + 1] = {};   // per part of a wave (zl_enc_wave)
    int waveParts = 1;
    cudaEvent_t evDescUp = nullptr;        // pipelined calls: recorded behind a wave's descriptor uploads; the next chunk's input copy waits for it
    double lastKernelMs = 0.0, lastStageMs[ZL_ENC_STAGES] = {};
    unsigned long long launches = 0;
    ZlDevBuf dBlocks, dFrames, dM, dRecs, dLit, dHist, dMetas, dOuts, dPlans, dResults, dXxh, dXxhPtrs, dXxhSizes, dSrc, dDst, dAux, dFar;
    ZlPinBuf hBlocks, hFrames, hResults, hAux;
    // streaming session (ZSTD_compressStream2): input accumulated on the host until ZSTD_e_end, then one frame is produced
    std::vector<u8> sIn, sOut;
    size_t sOutPos = 0;
    bool sFlushing = false;
    cudaStream_t side = nullptr; cudaEvent_t sideFork = nullptr, sideJoin = nullptr;   // sequence coding next to literal coding
    cudaStream_t copyIn = nullptr, copyOut = nullptr;      // zl_compress_split with host buffers: staging pipeline
    cudaEvent_t evIn[2] = {}, evOut[2] = {}, evGather[2] = {};
    struct { bool valid = false; void* dst = nullptr; const void* src = nullptr; size_t bytes = 0; int slot = 0; } pendIn;   // issued by zl_enc_run once its kernels are queued
    ZlDevBuf dOutStage;
    u32* statsDev = nullptr;               // set by the dictionary trainer: parse only, statistics summed here (zl_dict_train.cuh)
    // devices: the context's own (bound on first use) and, for batches of host buffers, the helpers on the other GPUs of the box
    // (num_threads / ZSTD_c_nbWorkers >= 2 asks for that many GPUs; 0 / 1: ZSTDLITE_GPUS, default 1)
    int device = -1;
    unsigned long long dictGen = 0, dictGenSeen = 0;
    std::vector<ZSTD_CCtx_s*> kids;
};

// __constant__ symbols and function attributes are per device: the encoder's code tables are uploaded once for every device a
// context is used on (a process may compress on several devices, and from several threads)
static std::mutex g_constMutex;
static bool g_constReady[64] = {};

static bool zl_cctx_ready(ZSTD_CCtx* c)
{
    if (!c->stream && !c->ownStream) {
        if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { (void)cudaGetLastError(); return false; }
        c->ownStream = true;
    }
    if (!c->ev0) {
        if (cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess) { (void)cudaGetLastError(); return false; }
        for (auto& ps : c->stageEv) for (cudaEvent_t& e : ps) if (cudaEventCreate(&e) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    }
    if (!c->side) {
        if (cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->sideFork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->sideJoin, cudaEventDisableTiming) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    }
    int devId = 0;
    if (cudaGetDevice(&devId) != cudaSuccess || devId < 0 || devId >= 64) { (void)cudaGetLastError(); return false; }
    {
        std::lock_guard<std::mutex> g(g_constMutex);
        if (!g_constReady[devId]) {
            if (zl_enc_upload_const() != cudaSuccess) { (void)cudaGetLastError(); return false; }
            g_constReady[devId] = true;
        }
    }
    return true;
}

ZL_EXPORT ZSTD_CCtx* ZSTD_createCCtx(void) { return new (std::nothrow) ZSTD_CCtx_s(); }
ZL_EXPORT size_t ZSTD_freeCCtx(ZSTD_CCtx* c)
{
    if (!c) return 0;
    for (ZSTD_CCtx_s* k : c->kids) ZSTD_freeCCtx(k);
    c->kids.clear();
    ZlDeviceGuard guard(c->device);
    ZlDevBuf* bufs[] = {&c->dBlocks, &c->dFrames, &c->dM, &c->dRecs, &c->dLit, &c->dHist, &c->dMetas, &c->dOuts, &c->dPlans, &c->dResults,
                        &c->dXxh, &c->dXxhPtrs, &c->dXxhSizes, &c->dSrc, &c->dDst, &c->dAux, &c->dFar,
                        &c->dDict, &c->dDictContent, &c->dDictTabS, &c->dDictTabL};
    for (ZlDevBuf* b : bufs) b->release();
    c->hBlocks.release(); c->hFrames.release(); c->hResults.release(); c->hAux.release();
    if (c->ev0) { cudaEventDestroy(c->ev0); cudaEventDestroy(c->ev1); }
    for (auto& ps : c->stageEv) for (cudaEvent_t e : ps) if (e) cudaEventDestroy(e);
    if (c->side) { cudaStreamDestroy(c->side); cudaEventDestroy(c->sideFork); cudaEventDestroy(c->sideJoin); }
    if (c->evDescUp) cudaEventDestroy(c->evDescUp);
    if (c->copyIn) { cudaStreamDestroy(c->copyIn); cudaStreamDestroy(c->copyOut); for (int i = 0; i < 2; i++) { cudaEventDestroy(c->evIn[i]); cudaEventDestroy(c->evOut[i]); cudaEventDestroy(c->evGather[i]); } }
    c->dOutStage.release();
    if (c->ownStream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return 0;
}
ZL_EXPORT size_t ZSTD_CCtx_reset(ZSTD_CCtx* c, ZSTD_ResetDirective r)          // zstd.c:23872
{
    if (r == ZSTD_reset_session_only || r == ZSTD_reset_session_and_parameters) {
        c->pledged = ZSTD_CONTENTSIZE_UNKNOWN; c->sIn.clear(); c->sOut.clear(); c->sOutPos = 0; c->sFlushing = false;
    }
    if (r == ZSTD_reset_parameters || r == ZSTD_reset_session_and_parameters) {
        c->level = 3; c->nbWorkers = 0; c->checksumFlag = 0; c->stableIn = 0; c->stableOut = 0; c->windowLog = 0; c->dictRaw.clear(); c->dictDirty = true; c->dictErr = 0;
    }
    return 0;
}
ZL_EXPORT size_t ZSTD_CCtx_setParameter(ZSTD_CCtx* c, ZSTD_cParameter p, int v)           // zstd.c:23223 (bounds: 22900-23100)
{
    switch ((int)p) {
    case ZSTD_c_compressionLevel: {                      // clamped like libzstd (ZSTD_cParam_clampBounds); 0 means default
        if (v < -131072) v = -131072;
        if (v > 22) v = 22;
        // Levels 4 and 5 run the level-3 (double-table) engine: with every position inserted and verified its output is within 3 % of
        // libzstd's AT THOSE LEVELS -- measured per family on 4 KB - 8 MiB inputs, with and without a dictionary: at most 1.027x
        // (DESIGN.md section 1, "Levels"; tests/test_emul_encode.py and tests/test_gpu_compress.py hold the bar).
        // Levels 6-22 (lazy / optimal parsers, zstd.c:31546-33746) are not implemented -- the same engine is 1.035x of level 6 and 1.06x
        // of level 9 on 2 MiB of text.  They are REFUSED rather than served under another label (SURVEY.md section 5: "unsupported
        // level" error), unless the caller opts in: ZSTDLITE_GPU_LEVEL_FALLBACK=1 in the environment (or zl_cctx_allow_level_fallback)
        // runs the level-3 engine for them -- valid Zstandard at level-3 ratio -- and says so once on stderr.  Negative ("fast") levels
        // run the level-1 engine: they ask for less ratio than it gives.
        static const bool envFallback = getenv("ZSTDLITE_GPU_LEVEL_FALLBACK") != nullptr && atoi(getenv("ZSTDLITE_GPU_LEVEL_FALLBACK")) != 0;
        if (v > ZL_MAX_SERVED_LEVEL) {
            if (!envFallback && !c->levelFallback) return ZL_ERROR(parameter_unsupported);
            static bool told = false;
            if (!told) { told = true; fprintf(stderr, "zstdlite_gpu: compression level %d is not implemented; running the level-3 engine (ZSTDLITE_GPU_LEVEL_FALLBACK)\n", v); }
        }
        c->level = v == 0 ? 3 : v;
        return 0;
    }
    // Blocks are 128 KiB, so a window below 2^17 cannot be honoured.  17 switches the far candidates of zl_enc_match.cuh off (every match
    // stays inside its block: the fastest setting for one large buffer); 18 and more bound the far offsets (at most 2^24 in any case).
    case ZSTD_c_windowLog: if (v != 0 && (v < 17 || v > 31)) return ZL_ERROR(parameter_outOfBound); c->windowLog = v; return 0;
    case ZSTD_c_nbWorkers: if (v < 0) v = 0; if (v > 256) v = 256; c->nbWorkers = v; return 0;
    case ZSTD_c_checksumFlag: if (v < 0 || v > 1) return ZL_ERROR(parameter_outOfBound); c->checksumFlag = v; return 0;
    case ZSTD_c_stableInBuffer: if (v < 0 || v > 1) return ZL_ERROR(parameter_outOfBound); c->stableIn = v; return 0;
    case ZSTD_c_stableOutBuffer: if (v < 0 || v > 1) return ZL_ERROR(parameter_outOfBound); c->stableOut = v; return 0;
    default: return ZL_ERROR(parameter_unsupported);
    }
}
// extension: accept levels 6-22 on this context and run them on the level-3 engine (see ZSTD_c_compressionLevel above)
ZL_EXPORT size_t zl_cctx_allow_level_fallback(ZSTD_CCtx* c, int on) { if (!c) return ZL_ERROR(GENERIC); c->levelFallback = on != 0; return 0; }
// extension: the engine level (1..3) a context's `level` actually runs
ZL_EXPORT int zl_cctx_engine_level(const ZSTD_CCtx* c) { return c ? (c->level < 1 ? 1 : (c->level > 3 ? 3 : c->level)) : 0; }
ZL_EXPORT size_t ZSTD_CCtx_getParameter(const ZSTD_CCtx* c, ZSTD_cParameter p, int* v)
{
    switch ((int)p) {
    case ZSTD_c_compressionLevel: *v = c->level; return 0;
    case ZSTD_c_windowLog: *v = c->windowLog; return 0;
    case ZSTD_c_nbWorkers: *v = c->nbWorkers; return 0;
    case ZSTD_c_checksumFlag: *v = c->checksumFlag; return 0;
    case ZSTD_c_stableInBuffer: *v = c->stableIn; return 0;
    case ZSTD_c_stableOutBuffer: *v = c->stableOut; return 0;
    default: return ZL_ERROR(parameter_unsupported);
    }
}
ZL_EXPORT size_t ZSTD_CCtx_setPledgedSrcSize(ZSTD_CCtx* c, unsigned long long pledged) { c->pledged = pledged; return 0; }
// Copies the dictionary (zstd.c:23826); it is digested lazily by the first compression that uses it, like the reference's
// ZSTD_initLocalDict (zstd.c:23757), so a corrupted dictionary is reported by the compress call.
ZL_EXPORT size_t ZSTD_CCtx_loadDictionary(ZSTD_CCtx* c, const void* dict, size_t dictSize)
{
    c->dictRaw.clear();
    if (dict && dictSize) c->dictRaw.assign((const u8*)dict, (const u8*)dict + dictSize);
    c->dictDirty = true; c->dictErr = 0; c->dictGen++;
    return 0;
}

static size_t zl_cctx_digest_dict(ZSTD_CCtx* c, const ZlEncParams& P)
{
    ZlEncDictDev* hd = new (std::nothrow) ZlEncDictDev();
    if (!hd) return ZL_ERROR(memory_allocation);
    std::vector<u8> content; std::vector<u32> tabS, tabL;
    const u32 err = zl_dict_digest_host(c->dictRaw.data(), c->dictRaw.size(), P, hd, content, tabS, tabL);
    if (err) { delete hd; return (size_t)0 - (size_t)err; }
    const size_t contentSize = hd->contentSize;
    bool ok = c->dDictContent.reserve(contentSize + 64) && c->dDictTabS.reserve(tabS.size() * 4) && c->dDictTabL.reserve(tabL.size() * 4) &&
              c->dDict.reserve(sizeof(ZlEncDictDev));
    if (ok) {
        hd->content = c->dDictContent.as<u8>(); hd->tabS = c->dDictTabS.as<u32>(); hd->tabL = P.hlogL ? c->dDictTabL.as<u32>() : nullptr;
        ok = cudaMemcpy(c->dDictContent.p, content.data(), contentSize + 64, cudaMemcpyHostToDevice) == cudaSuccess &&
             cudaMemcpy(c->dDictTabS.p, tabS.data(), tabS.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
             cudaMemcpy(c->dDictTabL.p, tabL.data(), tabL.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
             cudaMemcpy(c->dDict.p, hd, sizeof(ZlEncDictDev), cudaMemcpyHostToDevice) == cudaSuccess;
    }
    c->dictID = hd->dictID;
    delete hd;
    if (!ok) { (void)cudaGetLastError(); return ZL_ERROR(memory_allocation); }
    return 0;
}
// null when no dictionary is loaded; sets c->dictErr on failure
static const ZlEncDictDev* zl_cctx_dict(ZSTD_CCtx* c, const ZlEncParams& P)
{
    if (c->dictRaw.empty()) return nullptr;
    if (c->dictDirty || c->dictLevel != (int)P.level) {
        c->dictErr = zl_cctx_digest_dict(c, P);
        c->dictDirty = false; c->dictLevel = (int)P.level;
    }
    return c->dictErr ? nullptr : c->dDict.as<ZlEncDictDev>();
}
ZL_EXPORT size_t zl_cctx_set_stream(ZSTD_CCtx* c, void* s)
{
    if (c->ownStream && c->stream) cudaStreamDestroy(c->stream);
    c->stream = (cudaStream_t)s; c->ownStream = false;
    return 0;
}
ZL_EXPORT unsigned long long zl_cctx_launch_count(const ZSTD_CCtx* c) { return c->launches; }
ZL_EXPORT double zl_cctx_last_kernel_ms(const ZSTD_CCtx* c) { return c->lastKernelMs; }
ZL_EXPORT double zl_cctx_last_stage_ms(const ZSTD_CCtx* c, int stage) { return stage >= 0 && stage < ZL_ENC_STAGES ? c->lastStageMs[stage] : -1.0; }

ZL_EXPORT size_t ZSTD_compressBound(size_t n)                      // zstd.c:22583 / macro 4548
{
    if (n >= 0xFF00FF00FF00FF00ull) return ZL_ERROR(srcSize_wrong);
    return n + (n >> 8) + (n < (128u << 10) ? (((128u << 10) - n) >> 11) : 0);
}
ZL_ALIAS(ZSTD_CCtx*, ZSTD_createCCtx, (void))
ZL_ALIAS(size_t, ZSTD_freeCCtx, (ZSTD_CCtx*))
ZL_ALIAS(size_t, ZSTD_CCtx_reset, (ZSTD_CCtx*, ZSTD_ResetDirective))
ZL_ALIAS(size_t, ZSTD_CCtx_setParameter, (ZSTD_CCtx*, ZSTD_cParameter, int))
ZL_ALIAS(size_t, ZSTD_CCtx_getParameter, (const ZSTD_CCtx*, ZSTD_cParameter, int*))
ZL_ALIAS(size_t, ZSTD_CCtx_setPledgedSrcSize, (ZSTD_CCtx*, unsigned long long))
ZL_ALIAS(size_t, ZSTD_CCtx_loadDictionary, (ZSTD_CCtx*, const void*, size_t))
ZL_ALIAS(size_t, ZSTD_compressBound, (size_t))

// The level selects one of three table layouts (zl_enc_match.cuh).  Levels below 1 run the level-1 engine; levels above 3 are
// served by the level-3 engine (4, 5) or refused by ZSTD_CCtx_setParameter unless the caller opted into it (6+) (DESIGN.md, "levels").
static int zl_engine_level(int level) { return level < 1 ? 1 : (level > 3 ? 3 : level); }

// ---- one wave: frames [f0, f1) with DEVICE src/dst pointers; asynchronous on the context's stream.
// results land in c->dResults[f0..f1).
static size_t zl_enc_wave(ZSTD_CCtx* c, const u8* const* dsrc, const size_t* srcSize, u8* const* ddst, const size_t* dstCap, size_t f0, size_t f1,
                          size_t nbTotalFrames)
{
    static const ZlEncTuning tune = [] {                                  // (development switches)
        ZlEncTuning t;
        if (const char* v = getenv("ZL_ENC_HLOG")) t.hlog = sscanf(v, "%u,%u", &t.hlogS, &t.hlogL) == 2;
        if (const char* v = getenv("ZL_ENC_SIDE")) t.side = atoi(v);
        if (const char* v = getenv("ZL_ENC_PARTS")) t.parts = atoi(v);
        t.noFar = getenv("ZL_ENC_NOFAR") != nullptr;
        return t;
    }();
    cudaStream_t st = c->stream;
    ZlEncParams P = zl_enc_params(zl_engine_level(c->level));
    const ZlEncDictDev* dict = zl_cctx_dict(c, P);
    zl_enc_tune_params(P, dict != nullptr, c->windowLog, tune);
    if (c->dictErr && !c->dictRaw.empty()) return c->dictErr;
    ZlEncWave w;
    if (const size_t e = zl_enc_wave_layout(w, dsrc, srcSize, ddst, dstCap, f0, f1, c->statsDev != nullptr, P, tune)) return e;
    const size_t nb = w.nb, nf = w.nf;
    if (!c->hBlocks.reserve(nb * sizeof(ZlEncBlock)) || !c->hFrames.reserve(nf * sizeof(ZlEncFrame))) return ZL_ERROR(memory_allocation);
    if (!c->dBlocks.reserve(nb * sizeof(ZlEncBlock)) || !c->dFrames.reserve(nf * sizeof(ZlEncFrame)) || !c->dM.reserve(nb * (size_t)w.slotM * 4) ||
        !c->dRecs.reserve(nb * (size_t)w.slotRec * 8) || !c->dLit.reserve(nb * (size_t)w.slotLit) || !c->dHist.reserve(nb * 1024) ||
        !c->dMetas.reserve(nb * sizeof(ZlEncBlockMeta)) || !c->dOuts.reserve(nb * sizeof(ZlEncBlockOut)) || !c->dPlans.reserve(nb * sizeof(ZlEncBlockPlan)) ||
        !c->dResults.reserve(nbTotalFrames * 8))
        return ZL_ERROR(memory_allocation);
    ZlEncBlock* hb = c->hBlocks.as<ZlEncBlock>();
    ZlEncFrame* hf = c->hFrames.as<ZlEncFrame>();
    if (c->checksumFlag && (!c->hAux.reserve(nf * 16) || !c->dXxhPtrs.reserve(nf * 8) || !c->dXxhSizes.reserve(nf * 4) || !c->dXxh.reserve(nf * 8))) return ZL_ERROR(memory_allocation);
    const u8** hp = c->checksumFlag ? c->hAux.as<const u8*>() : nullptr;    // XXH64 of every frame's content (zstd.c:27022-27023)
    u32* hs = c->checksumFlag ? reinterpret_cast<u32*>(hp + nf) : nullptr;
    c->waveParts = (int)w.parts;
    for (size_t part = 0; part < w.parts; part++) {
        const ZlEncPart q = zl_enc_fill_part(w, part, dict ? c->dictID : 0u, (u32)c->checksumFlag, hf, hb, hp, hs);
        const size_t b0 = q.b0, fa = q.fa, pnb = q.nb, pnf = q.fb - q.fa;
        if (w.farEntries) {                                           // (only with parts == 1: frames of several blocks)
            if (!c->dFar.reserve(w.farEntries * 4)) return ZL_ERROR(memory_allocation);
            cudaMemsetAsync(c->dFar.p, 0xFF, w.farEntries * 4, st);
        }
        cudaMemcpyAsync(c->dBlocks.as<ZlEncBlock>() + b0, hb + b0, pnb * sizeof(ZlEncBlock), cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(c->dFrames.as<ZlEncFrame>() + fa, hf + fa, pnf * sizeof(ZlEncFrame), cudaMemcpyHostToDevice, st);
        if (c->evDescUp) cudaEventRecord(c->evDescUp, st);
        const u64* xxh = nullptr;
        if (c->checksumFlag) {
            cudaMemcpyAsync(c->dXxhPtrs.as<const u8*>() + fa, hp + fa, pnf * 8, cudaMemcpyHostToDevice, st);
            cudaMemcpyAsync(c->dXxhSizes.as<u32>() + fa, hs + fa, pnf * 4, cudaMemcpyHostToDevice, st);
            if (zl_launch_xxh64(c->dXxhPtrs.as<const u8*>() + fa, c->dXxhSizes.as<u32>() + fa, c->dXxh.as<u64>() + fa, (u32)pnf, st, q.anyLarge) != cudaSuccess) return ZL_ERROR(GENERIC);
            c->launches += 1;
            xxh = c->dXxh.as<u64>() + fa;
        }
        ZlEncodeLaunch L;
        L.blocks = c->dBlocks.as<ZlEncBlock>() + b0; L.nblocks = (u32)pnb; L.frames = c->dFrames.as<ZlEncFrame>() + fa; L.nframes = (u32)pnf;
        L.params = P; L.dict = dict;
        L.M = c->dM.as<u32>() + b0 * (size_t)w.slotM; L.slotM = w.slotM; L.recs = c->dRecs.as<u64>() + b0 * (size_t)w.slotRec; L.slotRec = w.slotRec;
        L.lit = c->dLit.as<u8>() + b0 * (size_t)w.slotLit; L.slotLit = w.slotLit;
        L.hist = c->dHist.as<u32>() + b0 * 256; L.metas = c->dMetas.as<ZlEncBlockMeta>() + b0; L.outs = c->dOuts.as<ZlEncBlockOut>() + b0;
        L.plans = c->dPlans.as<ZlEncBlockPlan>() + b0;
        L.streamCapWords = w.streamCapWords; L.streamWordsPerBlock = w.streamWordsPerBlock; L.seqCapWords = w.seqCapWords;
        L.far = w.farEntries ? c->dFar.as<u32>() : nullptr;
        L.nSmall = q.nSmall;
        L.results = c->dResults.as<u64>() + f0 + fa; L.xxh = xxh; L.stageEv = c->stageEv[part]; L.stats = c->statsDev; L.maxBlock = w.maxBlock;
        if (zl_enc_side(tune, pnb)) { L.side = c->side; L.sideFork = c->sideFork; L.sideJoin = c->sideJoin; }
        cudaError_t e = zl_launch_encode(L, st);
        c->launches += 6 + (w.farEntries ? 2 : 0) + ((q.nSmall && q.nSmall < pnb) ? 1 : 0);
        if (e != cudaSuccess) { fprintf(stderr, "zstdlite_gpu: kernel launch failed: %s\n", cudaGetErrorString(e)); return ZL_ERROR(GENERIC); }
    }
    return 0;
}

static void zl_copy_pieces(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind, cudaStream_t s);
// all frames, device pointers; synchronises; results in c->hResults
static size_t zl_enc_run(ZSTD_CCtx* c, const u8* const* dsrc, const size_t* srcSize, u8* const* ddst, const size_t* dstCap, size_t n)
{
    if (!c->hResults.reserve(n * 8)) return ZL_ERROR(memory_allocation);
    cudaStream_t st = c->stream;
    size_t waveBlocks = 0;
    if (const size_t e = zl_enc_wave_blocks(srcSize, n, &waveBlocks)) return e;
    double total = 0.0; double stage[ZL_ENC_STAGES] = {};
    auto addTimes = [&]() {                                       // kernel and per-stage times of the wave just finished
        float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1); total += ms;
        for (int q = 0; q < c->waveParts; q++) for (int k = 0; k < ZL_ENC_STAGES; k++) { float t = 0; cudaEventElapsedTime(&t, c->stageEv[q][k], c->stageEv[q][k + 1]); stage[k] += t; }
    };
    for (size_t f0 = 0; f0 < n;) {
        const size_t f1 = zl_enc_wave_end(srcSize, n, f0, waveBlocks);
        if (f0 > 0) {                                             // the wave's host-side descriptor buffers are reused: drain first
            if (cudaStreamSynchronize(st) != cudaSuccess) return ZL_ERROR(GENERIC);
            addTimes();
        }
        cudaEventRecord(c->ev0, st);
        const size_t r = zl_enc_wave(c, dsrc, srcSize, ddst, dstCap, f0, f1, n);
        cudaEventRecord(c->ev1, st);
        if (c->pendIn.valid) {
            // staging copy of the NEXT chunk (zl_compress_split_pipelined): behind this wave's descriptor uploads -- a copy engine serves its
            // requests in submission order, whatever their streams, and the uploads are only submitted once the stream's wait for THIS chunk's
            // input has fired: without the event the next chunk's 1 GiB went first and the kernels of this one waited 19 ms for their descriptors
            if (c->evDescUp) cudaStreamWaitEvent(c->copyIn, c->evDescUp, 0);
            zl_copy_pieces(c->pendIn.dst, c->pendIn.src, c->pendIn.bytes, cudaMemcpyHostToDevice, c->copyIn);
            cudaEventRecord(c->evIn[c->pendIn.slot], c->copyIn);
            c->pendIn.valid = false;
        }
        if (zl_is_error(r)) { cudaStreamSynchronize(st); return r; }
        f0 = f1;
    }
    if (zl_launch_results_out(c->dResults.as<u64>(), c->hResults.as<u64>(), (u32)n, st) != cudaSuccess) return ZL_ERROR(GENERIC);
    c->launches += 1;
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { fprintf(stderr, "zstdlite_gpu: device error: %s\n", cudaGetErrorString(e)); return ZL_ERROR(GENERIC); }
    addTimes();
    c->lastKernelMs = total;
    for (int k = 0; k < ZL_ENC_STAGES; k++) c->lastStageMs[k] = stage[k];
    return 0;
}

static size_t zl_compress_batch_one(ZSTD_CCtx* c, const void* const* src, const size_t* srcSize, void* const* dst, const size_t* dstCap,
                                    size_t* result, size_t n, int dev);
// Batches of HOST buffers spread over the GPUs of the box when the context asks for workers (num_threads = ZSTD_c_nbWorkers >= 2 -> that many
// GPUs) or ZSTDLITE_GPUS says so: contiguous ranges of the frame list of about equal input, one helper context and host thread per device;
// frames are independent, nothing moves between the devices (SURVEY.md 8e)
ZL_EXPORT size_t zl_compress_batch(ZSTD_CCtx* c, const void* const* src, const size_t* srcSize, void* const* dst, const size_t* dstCap,
                                   size_t* result, size_t n, int dev)
{
    if (!c) return ZL_ERROR(GENERIC);
    const int home = zl_bind_device(&c->device);
    size_t G = dev ? 1 : (size_t)zl_gpu_count(c->nbWorkers >= 2 ? c->nbWorkers : 0);
    unsigned long long bytes = 0;
    if (G > 1) for (size_t i = 0; i < n; i++) bytes += srcSize[i];
    if (G > n / 2) G = n / 2;
    if (G < 2 || bytes < ((unsigned long long)64 << 20) || c->statsDev) return zl_compress_batch_one(c, src, srcSize, dst, dstCap, result, n, dev);
    int ndev = 1;
    cudaGetDeviceCount(&ndev);
    while (c->kids.size() + 1 < G) {
        ZSTD_CCtx_s* k = new (std::nothrow) ZSTD_CCtx_s();
        if (!k) return ZL_ERROR(memory_allocation);
        k->device = (home + (int)c->kids.size() + 1) % ndev;
        c->kids.push_back(k);
    }
    const std::vector<size_t> cut = zl_split_ranges(srcSize, n, G);
    std::vector<size_t> rc(G, 0);
    auto work = [&](size_t g) {
        ZSTD_CCtx_s* k = g ? c->kids[g - 1] : c;
        if (g) {
            k->level = c->level; k->checksumFlag = c->checksumFlag; k->windowLog = c->windowLog; k->levelFallback = c->levelFallback; k->nbWorkers = 0;
            if (k->dictGenSeen != c->dictGen) { k->dictRaw = c->dictRaw; k->dictDirty = true; k->dictErr = 0; k->dictGenSeen = c->dictGen; }
        }
        const size_t a = cut[g], cnt = cut[g + 1] - a;
        rc[g] = cnt ? zl_compress_batch_one(k, src + a, srcSize + a, dst + a, dstCap + a, result + a, cnt, 0) : 0;
    };
    std::vector<std::thread> th;
    for (size_t g = 1; g < G; g++) th.emplace_back(work, g);
    work(0);
    for (std::thread& t : th) t.join();
    for (size_t g = 1; g < G; g++) { c->launches += c->kids[g - 1]->launches; c->kids[g - 1]->launches = 0; }
    for (size_t g = 0; g < G; g++) if (zl_is_error(rc[g])) return rc[g];
    return 0;
}
static size_t zl_compress_batch_one(ZSTD_CCtx* c, const void* const* src, const size_t* srcSize, void* const* dst, const size_t* dstCap,
                                    size_t* result, size_t n, int dev)
{
    ZlDeviceGuard guard(zl_bind_device(&c->device));
    if (!guard.ok) return ZL_ERROR(GENERIC);
    if (!c) return ZL_ERROR(GENERIC);
    if (n == 0) return 0;
    if (n > 0x0FFFFFFFull) return ZL_ERROR(memory_allocation);
    if (!zl_cctx_ready(c)) return ZL_ERROR(memory_allocation);
    cudaStream_t st = c->stream;
    if (dev) {
        const size_t r = zl_enc_run(c, (const u8* const*)src, srcSize, (u8* const*)dst, dstCap, n);
        if (zl_is_error(r)) return r;
        const u64* hr = c->hResults.as<u64>();
        for (size_t i = 0; i < n; i++) result[i] = (size_t)hr[i];
        return 0;
    }
    // host pointers: stage contiguous runs to the device, compress, copy the produced bytes back
    ZlEncPlace pl;
    zl_enc_place(pl, src, srcSize, dstCap, n);
    if (!c->dSrc.reserve(pl.srcTotal + 64) || !c->dDst.reserve(pl.dstTotal + 64)) return ZL_ERROR(memory_allocation);
    std::vector<const u8*> dsrc(n); std::vector<u8*> ddst(n);
    zl_enc_place_ptrs(pl, src, dstCap, n, c->dSrc.as<u8>(), c->dDst.as<u8>(), dsrc.data(), ddst.data());
    const bool staged = zl_enc_staged(pl, n, [&] { return zl_is_pageable(pl.runs[0].hbase); });
    ZlStagePool& sp = ZlStagePool::get();
    std::unique_lock<std::mutex> stageLock(sp.m, std::defer_lock);
    if (staged) {
        stageLock.lock();
        if (!sp.in.reserve(pl.srcTotal + 64)) return ZL_ERROR(memory_allocation);
        u8* hs = sp.in.as<u8>();
        for (const ZlUpload& u : zl_enc_stage_uploads(pl, hs)) {
            ZlCopyPool::get().run(u.segs);
            cudaMemcpyAsync(c->dSrc.as<u8>() + u.from, hs + u.from, u.to - u.from, cudaMemcpyHostToDevice, st);
        }
    } else
    for (const ZlRun& r : pl.runs) if (r.bytes) cudaMemcpyAsync(c->dSrc.as<u8>() + r.devOff, r.hbase, r.bytes, cudaMemcpyHostToDevice, st);
    const size_t r = zl_enc_run(c, dsrc.data(), srcSize, ddst.data(), dstCap, n);
    if (zl_is_error(r)) return r;
    const u64* hr = c->hResults.as<u64>();
    if (staged) {
        if (!c->hAux.reserve(n * 24) || !c->dAux.reserve(n * 24)) return ZL_ERROR(memory_allocation);
        u64* hsz = c->hAux.as<u64>();
        for (size_t i = 0; i < n; i++) result[i] = (size_t)hr[i];
        const size_t total = zl_enc_gather_table(hsz, hr, ddst.data(), n);
        if (!c->dOutStage.reserve(total + 64) || !sp.out.reserve(total + 64)) return ZL_ERROR(memory_allocation);
        cudaMemcpyAsync(c->dAux.p, hsz, n * 24, cudaMemcpyHostToDevice, st);
        const u64* dsz = c->dAux.as<u64>();
        if (zl_launch_gather(reinterpret_cast<const u8* const*>(dsz + 2 * n), dsz, dsz + n, c->dOutStage.as<u8>(), (u32)n, st) != cudaSuccess) return ZL_ERROR(GENERIC);
        c->launches += 1;
        if (total) cudaMemcpyAsync(sp.out.p, c->dOutStage.p, total, cudaMemcpyDeviceToHost, st);
        if (cudaStreamSynchronize(st) != cudaSuccess) { (void)cudaGetLastError(); return ZL_ERROR(GENERIC); }
        const u8* ho = sp.out.as<u8>();
        std::vector<ZlCopySeg> osegs;
        for (size_t i = 0; i < n; i++) if (hsz[i]) osegs.push_back({dst[i], ho + hsz[n + i], (size_t)hsz[i]});
        ZlCopyPool::get().run(osegs);
        return 0;
    }
    for (size_t i = 0; i < n; i++) {
        result[i] = (size_t)hr[i];
        if (!zl_is_error(result[i]) && result[i]) cudaMemcpyAsync(dst[i], ddst[i], result[i], cudaMemcpyDeviceToHost, st);
    }
    if (cudaStreamSynchronize(st) != cudaSuccess) { (void)cudaGetLastError(); return ZL_ERROR(GENERIC); }
    return 0;
}

// zstd.c:28949 ZSTD_compress2: one input -> one frame (of independent <= 128 KiB blocks) whose header records the content size
ZL_EXPORT size_t ZSTD_compress2(ZSTD_CCtx* c, void* dst, size_t dstCap, const void* src, size_t srcSize)
{
    if (!c) return ZL_ERROR(GENERIC);
    if (!dst && dstCap) return ZL_ERROR(dstBuffer_null);
    const void* sp = src; void* dp = dst; size_t res = 0;
    static const u8 empty = 0;
    if (!sp) { if (srcSize) return ZL_ERROR(srcSize_wrong); sp = &empty; }
    const size_t r = zl_compress_batch(c, &sp, &srcSize, &dp, &dstCap, &res, 1, 0);
    c->pledged = ZSTD_CONTENTSIZE_UNKNOWN;                                  // session reset, zstd.c:28956
    return zl_is_error(r) ? r : res;
}
ZL_ALIAS(size_t, ZSTD_compress2, (ZSTD_CCtx*, void*, size_t, const void*, size_t))

// zstd.c:28828 ZSTD_compressStream2 over the one-shot engine: ZSTD_e_continue / ZSTD_e_flush only accumulate (a flush cannot
// close a frame whose header must record the content size); ZSTD_e_end compresses everything as one frame and hands it out
// in the caller's chunk sizes.  Return value as libzstd: bytes still to be flushed (0 = this frame is complete).
ZL_EXPORT size_t ZSTD_compressStream2(ZSTD_CCtx* c, ZSTD_outBuffer* out, ZSTD_inBuffer* in, ZSTD_EndDirective end)
{
    if (!c || !out || !in) return ZL_ERROR(GENERIC);
    if (out->pos > out->size) return ZL_ERROR(dstSize_tooSmall);
    if (in->pos > in->size) return ZL_ERROR(srcSize_wrong);
    if ((int)end < 0 || (int)end > 2) return ZL_ERROR(parameter_outOfBound);
    if (!c->sFlushing) {
        if (in->size > in->pos) c->sIn.insert(c->sIn.end(), (const u8*)in->src + in->pos, (const u8*)in->src + in->size);
        in->pos = in->size;
        if (end != ZSTD_e_end) return 0;
        if (c->pledged != ZSTD_CONTENTSIZE_UNKNOWN && c->pledged != c->sIn.size()) {           // zstd.c:27190 (pledged size check)
            c->sIn.clear(); c->pledged = ZSTD_CONTENTSIZE_UNKNOWN;
            return ZL_ERROR(srcSize_wrong);
        }
        const size_t n = c->sIn.size(), cap = ZSTD_compressBound(n);
        if (zl_is_error(cap)) return cap;
        c->sOut.resize(cap ? cap : 1);
        const size_t r = ZSTD_compress2(c, c->sOut.data(), cap, c->sIn.data(), n);
        std::vector<u8>().swap(c->sIn);
        if (zl_is_error(r)) { c->sOut.clear(); return r; }
        c->sOut.resize(r); c->sOutPos = 0; c->sFlushing = true;
    } else if (in->size > in->pos) return ZL_ERROR(stage_wrong);                                // new input while a frame is being flushed
    const size_t room = out->size - out->pos, left = c->sOut.size() - c->sOutPos, k = room < left ? room : left;
    if (k) memcpy((u8*)out->dst + out->pos, c->sOut.data() + c->sOutPos, k);
    out->pos += k; c->sOutPos += k;
    const size_t remaining = c->sOut.size() - c->sOutPos;
    if (!remaining) { std::vector<u8>().swap(c->sOut); c->sOutPos = 0; c->sFlushing = false; }
    return remaining;
}
ZL_ALIAS(size_t, ZSTD_compressStream2, (ZSTD_CCtx*, ZSTD_outBuffer*, ZSTD_inBuffer*, ZSTD_EndDirective))

// One buffer -> concatenated independent frames of `frameSize` content bytes (a standard multi-frame zstd stream).
// host buffers, many frames: chunks of frames are staged, compressed and copied back in a pipeline -- the host-to-device copy of
// chunk k+1 and the device-to-host copy of chunk k-1 run (on their own streams) while chunk k is compressed
// large staging copies go out in pieces of 16 MiB (bounded latency for small copies submitted behind them)
static void zl_copy_pieces(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind, cudaStream_t s)
{
    const size_t piece = (size_t)16 << 20;
    for (size_t o = 0; o < bytes; o += piece)
        cudaMemcpyAsync((u8*)dst + o, (const u8*)src + o, bytes - o < piece ? bytes - o : piece, kind, s);
}
static size_t zl_compress_split_pipelined(ZSTD_CCtx* c, void* dst, size_t dstCap, const u8* src, size_t srcSize, size_t frameSize,
                                          size_t* frameSizes, const ZlSplitPlan& sp, size_t slot)
{
    cudaStream_t st = c->stream;
    if (!c->copyIn) {
        if (cudaStreamCreateWithFlags(&c->copyIn, cudaStreamNonBlocking) != cudaSuccess || cudaStreamCreateWithFlags(&c->copyOut, cudaStreamNonBlocking) != cudaSuccess) { (void)cudaGetLastError(); return ZL_ERROR(memory_allocation); }
        if (cudaEventCreateWithFlags(&c->evDescUp, cudaEventDisableTiming) != cudaSuccess) { (void)cudaGetLastError(); return ZL_ERROR(memory_allocation); }
        for (int i = 0; i < 2; i++)
            if (cudaEventCreateWithFlags(&c->evIn[i], cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&c->evOut[i], cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&c->evGather[i], cudaEventDisableTiming) != cudaSuccess) { (void)cudaGetLastError(); return ZL_ERROR(memory_allocation); }
    }
    const size_t chunkFrames = sp.chunkFrames, chunkBytes = chunkFrames * frameSize;
    const size_t inHalf = (chunkBytes + 255) & ~(size_t)255, outHalf = (chunkFrames * slot + 255) & ~(size_t)255;
    if (!c->dSrc.reserve(2 * inHalf + 64) || !c->dDst.reserve(chunkFrames * slot + 64) || !c->dOutStage.reserve(2 * outHalf + 64) ||
        !c->hAux.reserve(chunkFrames * 24) || !c->dAux.reserve(chunkFrames * 24)) return ZL_ERROR(memory_allocation);
    const size_t nchunks = sp.cstart.size() - 1;
    std::vector<const u8*> dsrc(chunkFrames); std::vector<u8*> ddst(chunkFrames); std::vector<size_t> ssz(chunkFrames), caps(chunkFrames, slot);
    auto chunkBytesOf = [&](size_t k) { return std::min(sp.cstart[k + 1] * frameSize, srcSize) - sp.cstart[k] * frameSize; };
    size_t total = 0, err = 0;
    static const bool trace = getenv("ZL_ENC_TRACE") != nullptr;      // (development: host timeline of the chunks on stderr)
    const auto t00 = std::chrono::steady_clock::now();
    auto nowMs = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t00).count(); };
    zl_copy_pieces(c->dSrc.p, src, chunkBytesOf(0), cudaMemcpyHostToDevice, c->copyIn);
    cudaEventRecord(c->evIn[0], c->copyIn);
    for (size_t k = 0; k < nchunks && !err; k++) {
        const size_t f0 = sp.cstart[k], cnt = sp.cstart[k + 1] - f0;
        if (k + 1 < nchunks) {                                   // next chunk's input (its half was last read by chunk k-1, finished)
            c->pendIn.valid = true; c->pendIn.dst = c->dSrc.as<u8>() + ((k + 1) & 1) * inHalf; c->pendIn.src = src + sp.cstart[k + 1] * frameSize;
            c->pendIn.bytes = chunkBytesOf(k + 1); c->pendIn.slot = (int)((k + 1) & 1);
        }
        cudaStreamWaitEvent(st, c->evIn[k & 1], 0);
        zl_enc_split_frames(c->dSrc.as<u8>() + (k & 1) * inHalf, chunkBytesOf(k), frameSize, c->dDst.as<u8>(), slot, cnt, dsrc.data(), ssz.data(), ddst.data());
        const double tA = nowMs();
        const size_t r = zl_enc_run(c, dsrc.data(), ssz.data(), ddst.data(), caps.data(), cnt);
        if (zl_is_error(r)) { err = r; break; }
        if (trace) fprintf(stderr, "chunk %zu: compress call %.1f -> %.1f ms (kernels %.1f ms: match %.1f parse %.1f literals %.1f sequences %.1f assemble %.1f)\n", k, tA, nowMs(),
                           c->lastKernelMs, c->lastStageMs[0], c->lastStageMs[1], c->lastStageMs[2], c->lastStageMs[3], c->lastStageMs[4]);
        const u64* hr = c->hResults.as<u64>();
        for (size_t i = 0; i < cnt && !err; i++) {
            if (zl_is_error((size_t)hr[i])) err = (size_t)hr[i];
            else if (frameSizes) frameSizes[f0 + i] = (size_t)hr[i];
        }
        if (err) break;
        u64* hsz = c->hAux.as<u64>();
        const size_t ctotal = zl_enc_gather_table(hsz, hr, ddst.data(), cnt);
        if (total + ctotal > dstCap) { err = ZL_ERROR(dstSize_tooSmall); break; }
        // the gather reads its sizes / offsets / pointers straight from the pinned (device-mapped) host array: as a cudaMemcpyAsync these
        // 24 bytes per frame queued up behind the NEXT chunk's input on the host-to-device copy engine (measured: 1.3 and 4.2 ms of idle
        // device before the 512 MiB and 1 GiB chunks of a 4 GiB call)
        u8* stage = c->dOutStage.as<u8>() + (k & 1) * outHalf;
        if (k >= 2) cudaStreamWaitEvent(st, c->evOut[k & 1], 0);  // the copy back of chunk k-2 has left this half
        const u64* dsz = hsz;
        if (zl_launch_gather(reinterpret_cast<const u8* const*>(dsz + 2 * cnt), dsz, dsz + cnt, stage, (u32)cnt, st) != cudaSuccess) { err = ZL_ERROR(GENERIC); break; }
        c->launches += 1;
        cudaEventRecord(c->evGather[k & 1], st);
        cudaStreamWaitEvent(c->copyOut, c->evGather[k & 1], 0);
        if (ctotal) zl_copy_pieces((u8*)dst + total, stage, ctotal, cudaMemcpyDeviceToHost, c->copyOut);
        cudaEventRecord(c->evOut[k & 1], c->copyOut);
        const double tB = nowMs();
        if (cudaStreamSynchronize(st) != cudaSuccess) { (void)cudaGetLastError(); err = ZL_ERROR(GENERIC); break; }   // hAux / dAux are reused by the next chunk
        if (trace) fprintf(stderr, "chunk %zu: gather + copy back queued at %.1f, gather done at %.1f ms (%zu bytes out)\n", k, tB, nowMs(), ctotal);
        total += ctotal;
    }
    if (trace) fprintf(stderr, "chunks done at %.1f ms\n", nowMs());
    const bool ok = cudaStreamSynchronize(c->copyIn) == cudaSuccess && cudaStreamSynchronize(c->copyOut) == cudaSuccess;
    if (trace) fprintf(stderr, "copies done at %.1f ms\n", nowMs());
    if (err) return err;
    if (!ok) { (void)cudaGetLastError(); return ZL_ERROR(GENERIC); }
    return total;
}

ZL_EXPORT size_t zl_compress_split(ZSTD_CCtx* c, void* dst, size_t dstCap, const void* src, size_t srcSize, size_t frameSize,
                                   size_t* frameSizes, int dev)
{
    if (!c || !frameSize) return ZL_ERROR(GENERIC);
    ZlDeviceGuard guard(zl_bind_device(&c->device));
    if (!guard.ok) return ZL_ERROR(GENERIC);
    if (!zl_cctx_ready(c)) return ZL_ERROR(memory_allocation);
    cudaStream_t st = c->stream;
    const ZlSplitPlan sp = zl_enc_split_plan(srcSize, frameSize, dev != 0);
    const size_t nf = sp.nf;
    const size_t slot = (ZSTD_compressBound(frameSize) + 4 + 15) & ~(size_t)15;
    if (sp.pipelined) return zl_compress_split_pipelined(c, dst, dstCap, (const u8*)src, srcSize, frameSize, frameSizes, sp, slot);
    const u8* dsrcBase = (const u8*)src;
    if (!dev) {
        if (!c->dSrc.reserve(srcSize + 64)) return ZL_ERROR(memory_allocation);
        if (srcSize) cudaMemcpyAsync(c->dSrc.p, src, srcSize, cudaMemcpyHostToDevice, st);
        dsrcBase = c->dSrc.as<u8>();
    }
    if (!c->dDst.reserve(nf * slot + 64)) return ZL_ERROR(memory_allocation);
    std::vector<const u8*> dsrc(nf); std::vector<u8*> ddst(nf); std::vector<size_t> ssz(nf), caps(nf, slot);
    zl_enc_split_frames(dsrcBase, srcSize, frameSize, c->dDst.as<u8>(), slot, nf, dsrc.data(), ssz.data(), ddst.data());
    const size_t r = zl_enc_run(c, dsrc.data(), ssz.data(), ddst.data(), caps.data(), nf);
    if (zl_is_error(r)) return r;
    const u64* hr = c->hResults.as<u64>();
    // exclusive scan of the frame sizes (host: nf integers), then one gather launch
    if (!c->hAux.reserve(nf * 24) || !c->dAux.reserve(nf * 24)) return ZL_ERROR(memory_allocation);
    for (size_t i = 0; i < nf; i++) {
        if (zl_is_error((size_t)hr[i])) return (size_t)hr[i];
        if (frameSizes) frameSizes[i] = (size_t)hr[i];
    }
    u64* hsz = c->hAux.as<u64>();
    const size_t total = zl_enc_gather_table(hsz, hr, ddst.data(), nf);
    if (total > dstCap) return ZL_ERROR(dstSize_tooSmall);
    cudaMemcpyAsync(c->dAux.p, hsz, nf * 24, cudaMemcpyHostToDevice, st);
    u8* out = (u8*)dst;
    if (!dev) { if (!c->dSrc.reserve(total + 64)) return ZL_ERROR(memory_allocation); out = c->dSrc.as<u8>(); }   // the staged input is no longer needed
    const u64* dsz = c->dAux.as<u64>();
    if (zl_launch_gather(reinterpret_cast<const u8* const*>(dsz + 2 * nf), dsz, dsz + nf, out, (u32)nf, st) != cudaSuccess) return ZL_ERROR(GENERIC);
    c->launches += 1;
    if (!dev && total) cudaMemcpyAsync(dst, out, total, cudaMemcpyDeviceToHost, st);
    if (cudaStreamSynchronize(st) != cudaSuccess) { (void)cudaGetLastError(); return ZL_ERROR(GENERIC); }
    return total;
}

#include "zl_dict_train.cuh"
