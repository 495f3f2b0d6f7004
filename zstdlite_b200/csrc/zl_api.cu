// zl_api.cu -- the C ABI (include/zstdlite_gpu.h): error/version helpers, frame introspection, the
// decompression context and the batched decode driver.  Compression entry points are in zl_api_compress.cu.
#include <stdio.h>
#include <stdlib.h>
#include <new>
#include <chrono>
#include <vector>
#include <thread>
#include "../../include/zstdlite_gpu.h"
#include "zl_batch_plan.h"            // (and zl_host.h)
#include "zl_dec_entropy.cuh"     // ZL_HD table builders reused to digest dictionaries on the host (zstd.c:42053)

#define ZL_EXPORT extern "C" __attribute__((visibility("default")))
#define ZL_ALIAS(ret, name, params) extern "C" __attribute__((visibility("default"), alias(#name))) ret zlg_##name params;

// ---------------------------------------------------------------------------------------------- errors
ZL_EXPORT unsigned ZSTD_isError(size_t code) { return zl_is_error(code); }
ZL_EXPORT const char* ZSTD_getErrorName(size_t code)
{
    if (!zl_is_error(code)) return "No error detected";
    switch ((unsigned)((size_t)0 - code)) {          // strings: zstd.c:3590-3630
    case ZL_E_GENERIC: return "Error (generic)";
    case ZL_E_prefix_unknown: return "Unknown frame descriptor";
    case ZL_E_version_unsupported: return "Version not supported";
    case ZL_E_frameParameter_unsupported: return "Unsupported frame parameter";
    case ZL_E_frameParameter_windowTooLarge: return "Frame requires too much memory for decoding";
    case ZL_E_corruption_detected: return "Data corruption detected";
    case ZL_E_checksum_wrong: return "Restored data doesn't match checksum";
    case ZL_E_literals_headerWrong: return "Header of Literals' block doesn't respect format specification";
    case ZL_E_parameter_unsupported: return "Unsupported parameter";
    case ZL_E_parameter_combination_unsupported: return "Unsupported combination of parameters";
    case ZL_E_parameter_outOfBound: return "Parameter is out of bound";
    case ZL_E_init_missing: return "Context should be init first";
    case ZL_E_memory_allocation: return "Allocation error : not enough memory";
    case ZL_E_workSpace_tooSmall: return "workSpace buffer is not large enough";
    case ZL_E_stage_wrong: return "Operation not authorized at current processing stage";
    case ZL_E_tableLog_tooLarge: return "tableLog requires too much memory : unsupported";
    case ZL_E_maxSymbolValue_tooLarge: return "Unsupported max Symbol Value : too large";
    case ZL_E_maxSymbolValue_tooSmall: return "Specified maxSymbolValue is too small";
    case ZL_E_stabilityCondition_notRespected: return "pledged buffer stability condition is not respected";
    case ZL_E_dictionary_corrupted: return "Dictionary is corrupted";
    case ZL_E_dictionary_wrong: return "Dictionary mismatch";
    case ZL_E_dictionaryCreation_failed: return "Cannot create Dictionary from provided samples";
    case ZL_E_dstSize_tooSmall: return "Destination buffer is too small";
    case ZL_E_srcSize_wrong: return "Src size is incorrect";
    case ZL_E_dstBuffer_null: return "Operation on NULL destination buffer";
    case ZL_E_noForwardProgress_destFull: return "Operation made no progress over multiple calls, due to output buffer being full";
    case ZL_E_noForwardProgress_inputEmpty: return "Operation made no progress over multiple calls, due to input being empty";
    default: return "Unspecified error code";
    }
}
ZL_EXPORT const char* ZSTD_versionString(void) { return "1.5.6"; }      // format/ABI level of the reference's libzstd
ZL_EXPORT const char* zl_backend_string(void) { return "zstdlite-b200 0.1 (CUDA sm_100a; no CPU fallback)"; }
ZL_ALIAS(unsigned, ZSTD_isError, (size_t))
ZL_ALIAS(const char*, ZSTD_getErrorName, (size_t))
ZL_ALIAS(const char*, ZSTD_versionString, (void))

// ---------------------------------------------------------------------------------------------- frame introspection (host)
size_t zl_host_frame_header(ZlHostFrameHeader* h, const void* srcv, size_t srcSize)
{
    const u8* ip = (const u8*)srcv;
    memset(h, 0, sizeof(*h));
    if (srcSize > 0 && ip == nullptr) return ZL_ERROR(GENERIC);
    if (srcSize < 5) {                               // zstd.c:41061-41077: a too-short prefix must still look like a magic number
        if (srcSize > 0) {
            u8 m[4] = {0x28, 0xB5, 0x2F, 0xFD};
            u8 sk[4] = {0x50, 0x2A, 0x4D, 0x18};
            bool a = true, b = true;
            for (size_t i = 0; i < srcSize && i < 4; i++) { if (ip[i] != m[i]) a = false; if (i > 0 && ip[i] != sk[i]) b = false; if (i == 0 && (ip[i] & 0xF0) != 0x50) b = false; }
            if (!a && !b) return ZL_ERROR(prefix_unknown);
        }
        return 5;
    }
    u32 magic = zl_rd32(ip);
    if ((magic & 0xFFFFFFF0u) == ZL_MAGIC_SKIP) {
        if (srcSize < 8) return 8;
        h->skippable = 1; h->contentSize = zl_rd32(ip + 4); h->headerSize = 8;
        return 0;
    }
    if (magic != ZL_MAGIC) return ZL_ERROR(prefix_unknown);
    u32 fhd = ip[4], didCode = fhd & 3, single = (fhd >> 5) & 1, fcsID = fhd >> 6;
    u32 didSz = didCode == 3 ? 4 : didCode, fcsSz = fcsID == 0 ? (single ? 1u : 0u) : (1u << fcsID);
    u32 hs = 5 + (single ? 0 : 1) + didSz + fcsSz;
    if (srcSize < hs) return hs;
    h->headerSize = hs;
    if (fhd & 8) return ZL_ERROR(frameParameter_unsupported);
    u32 p = 5; u64 window = 0;
    if (!single) {
        u32 wl = ip[p++], wlog = (wl >> 3) + 10;
        if (wlog > 31) return ZL_ERROR(frameParameter_windowTooLarge);
        window = 1ull << wlog; window += (window >> 3) * (wl & 7);
    }
    u32 did = 0;
    if (didSz == 1) did = ip[p]; else if (didSz == 2) did = zl_rd16(ip + p); else if (didSz == 4) did = zl_rd32(ip + p);
    p += didSz;
    u64 fcs = ZSTD_CONTENTSIZE_UNKNOWN;
    if (fcsID == 0) { if (single) fcs = ip[p]; } else if (fcsID == 1) fcs = zl_rd16(ip + p) + 256; else if (fcsID == 2) fcs = zl_rd32(ip + p); else fcs = zl_rd64(ip + p);
    if (single) window = fcs;
    h->contentSize = fcs; h->windowSize = window;
    h->blockSizeMax = (unsigned)(window < ZL_BLOCKSIZE_MAX ? window : ZL_BLOCKSIZE_MAX);
    h->dictID = did; h->checksumFlag = (fhd >> 2) & 1;
    return 0;
}

size_t zl_host_find_frame_size(const void* srcv, size_t srcSize, unsigned* nblocksOut)
{
    const u8* ip = (const u8*)srcv;
    if (nblocksOut) *nblocksOut = 0;
    if (srcSize >= 8 && (zl_rd32(ip) & 0xFFFFFFF0u) == ZL_MAGIC_SKIP) {         // zstd.c:41188
        u64 sz = (u64)zl_rd32(ip + 4) + 8;
        if (sz > srcSize) return ZL_ERROR(srcSize_wrong);
        return (size_t)sz;
    }
    ZlHostFrameHeader h;
    size_t r = zl_host_frame_header(&h, srcv, srcSize);
    if (zl_is_error(r)) return r;
    if (r > 0) return ZL_ERROR(srcSize_wrong);
    size_t pos = h.headerSize; unsigned nb = 0;
    for (;;) {                                                                   // zstd.c:41370-41384
        if (srcSize - pos < 3) return ZL_ERROR(srcSize_wrong);
        u32 bh = zl_rd24(ip + pos), last = bh & 1, type = (bh >> 1) & 3, cs = bh >> 3;
        if (type == 3) return ZL_ERROR(corruption_detected);
        if (type == 1) cs = 1;
        if (3 + (size_t)cs > srcSize - pos) return ZL_ERROR(srcSize_wrong);
        pos += 3 + cs; nb++;
        if (last) break;
    }
    if (h.checksumFlag) { if (srcSize - pos < 4) return ZL_ERROR(srcSize_wrong); pos += 4; }
    if (nblocksOut) *nblocksOut = nb;
    return pos;
}

ZL_EXPORT size_t ZSTD_getFrameHeader(ZSTD_frameHeader* z, const void* src, size_t srcSize)
{
    ZlHostFrameHeader h;
    size_t r = zl_host_frame_header(&h, src, srcSize);
    if (r != 0) return r;
    memset(z, 0, sizeof(*z));
    z->frameContentSize = h.contentSize; z->windowSize = h.windowSize; z->blockSizeMax = h.blockSizeMax;
    z->frameType = h.skippable ? ZSTD_skippableFrame : ZSTD_frame; z->headerSize = h.headerSize;
    z->dictID = h.dictID; z->checksumFlag = h.checksumFlag;
    return 0;
}
ZL_EXPORT unsigned long long ZSTD_getFrameContentSize(const void* src, size_t srcSize)
{
    ZlHostFrameHeader h;
    if (zl_host_frame_header(&h, src, srcSize) != 0) return ZSTD_CONTENTSIZE_ERROR;
    return h.skippable ? 0ULL : h.contentSize;
}
ZL_EXPORT size_t ZSTD_findFrameCompressedSize(const void* src, size_t srcSize) { return zl_host_find_frame_size(src, srcSize, nullptr); }
// zstd.c:41244: content size of a whole stream of concatenated frames (skippable frames count as 0); SURVEY.md 8f rank 2
ZL_EXPORT unsigned long long ZSTD_findDecompressedSize(const void* srcv, size_t srcSize)
{
    const u8* src = (const u8*)srcv;
    unsigned long long total = 0;
    while (srcSize >= 5) {                                                       // ZSTD_startingInputLength
        if ((zl_rd32(src) & 0xFFFFFFF0u) != ZL_MAGIC_SKIP) {
            const unsigned long long fcs = ZSTD_getFrameContentSize(src, srcSize);
            if (fcs >= ZSTD_CONTENTSIZE_ERROR) return fcs;                       // unknown or error: reported as such
            if (total + fcs < total) return ZSTD_CONTENTSIZE_ERROR;
            total += fcs;
        }
        const size_t fs = zl_host_find_frame_size(src, srcSize, nullptr);
        if (zl_is_error(fs)) return ZSTD_CONTENTSIZE_ERROR;
        src += fs; srcSize -= fs;
    }
    return srcSize ? ZSTD_CONTENTSIZE_ERROR : total;
}
ZL_EXPORT unsigned ZSTD_getDictID_fromFrame(const void* src, size_t srcSize)
{
    ZlHostFrameHeader h;
    if (zl_host_frame_header(&h, src, srcSize) != 0) return 0;
    return h.dictID;
}
ZL_EXPORT unsigned ZSTD_getDictID_fromDict(const void* dict, size_t dictSize)
{
    if (dictSize < 8 || zl_rd32((const u8*)dict) != ZL_MAGIC_DICT) return 0;
    return zl_rd32((const u8*)dict + 4);
}
ZL_EXPORT unsigned ZDICT_getDictID(const void* dict, size_t dictSize) { return ZSTD_getDictID_fromDict(dict, dictSize); }
ZL_ALIAS(size_t, ZSTD_getFrameHeader, (ZSTD_frameHeader*, const void*, size_t))
ZL_ALIAS(unsigned long long, ZSTD_getFrameContentSize, (const void*, size_t))
ZL_ALIAS(size_t, ZSTD_findFrameCompressedSize, (const void*, size_t))
ZL_ALIAS(unsigned long long, ZSTD_findDecompressedSize, (const void*, size_t))
ZL_ALIAS(unsigned, ZSTD_getDictID_fromFrame, (const void*, size_t))
ZL_ALIAS(unsigned, ZSTD_getDictID_fromDict, (const void*, size_t))
ZL_ALIAS(unsigned, ZDICT_getDictID, (const void*, size_t))

// ---------------------------------------------------------------------------------------------- decompression context
struct ZSTD_DCtx_s {
    int forceIgnoreChecksum = 0, stableOut = 0, windowLogMax = 27;
    std::vector<u8> dictRaw;
    ZlDevBuf dDictContent, dDict;          // device copies (content bytes, ZlDictDev)
    bool hasDict = false;
    cudaStream_t stream = nullptr;
    bool ownStream = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t stageEv[ZL_DEC_STAGES + 1] = {};
    double lastKernelMs = 0.0, lastStageMs[ZL_DEC_STAGES] = {};
    unsigned long long launches = 0;
    // slice pipeline: a batch is cut into slices that run on ZL_DEC_LANES internal streams, so that the execute
    // kernel and the PCIe copies of one slice overlap the (shared-memory-bound) entropy kernels of the others
    cudaStream_t lane[ZL_DEC_LANES] = {};
    cudaEvent_t laneDone[ZL_DEC_LANES] = {}, forkEv = nullptr;
    cudaEvent_t inDone[ZL_DEC_LANES] = {};                // host buffers: host-to-device copies of a slice done (they run in slice order)
    cudaStream_t side[ZL_DEC_LANES] = {};                 // per lane: the sequence kernel runs here, next to the literal kernel
    cudaEvent_t sideFork[ZL_DEC_LANES] = {}, sideJoin[ZL_DEC_LANES] = {};
    int profileStages = 0;                 // 1: one slice, one stream, per-kernel events (zl_dctx_last_stage_ms)
    // streaming session (ZSTD_decompressStream): input accumulated on the host until a whole frame is present
    std::vector<u8> sIn, sOut;
    size_t sOutPos = 0;
    ZlDevBuf dRaw, dDescs, dInfos, dResults, dHdr, dRec, dCk, dLit, dNorm, dUnits, dCounters, dLargeIdx, dLb, dLc, dParent, dRemain, dSrc, dDst;
    ZlPinBuf hDescs, hResults, hLargeIdx, hRemain;
    std::vector<cudaEvent_t> sliceDone;    // staged host buffers: the copy back of a slice has landed
    // devices: the context's own (bound on first use) and, for batches of host buffers, the helpers on the other GPUs of the box
    int device = -1, gpus = 0;             // gpus: 0 = ZSTDLITE_GPUS (default 1)
    unsigned long long dictGen = 0, dictGenSeen = 0;
    std::vector<ZSTD_DCtx_s*> kids;        // one per further device, created on demand, owned by this context
};

static bool zl_ctx_stream(cudaStream_t* st, bool* own, cudaEvent_t* e0, cudaEvent_t* e1)
{
    if (!*st && !*own) {
        if (cudaStreamCreateWithFlags(st, cudaStreamNonBlocking) != cudaSuccess) { (void)cudaGetLastError(); return false; }
        *own = true;
    }
    if (!*e0) { if (cudaEventCreate(e0) != cudaSuccess || cudaEventCreate(e1) != cudaSuccess) { (void)cudaGetLastError(); return false; } }
    return true;
}

ZL_EXPORT ZSTD_DCtx* ZSTD_createDCtx(void) { return new (std::nothrow) ZSTD_DCtx_s(); }
ZL_EXPORT size_t ZSTD_freeDCtx(ZSTD_DCtx* c)
{
    if (!c) return 0;
    for (ZSTD_DCtx_s* k : c->kids) ZSTD_freeDCtx(k);
    c->kids.clear();
    ZlDeviceGuard guard(c->device);
    ZlDevBuf* bufs[] = {&c->dDictContent, &c->dDict, &c->dRaw, &c->dDescs, &c->dInfos, &c->dResults, &c->dHdr, &c->dRec, &c->dCk, &c->dLit, &c->dNorm, &c->dUnits, &c->dCounters, &c->dLargeIdx, &c->dLb, &c->dLc, &c->dParent, &c->dRemain, &c->dSrc, &c->dDst};
    for (ZlDevBuf* b : bufs) b->release();
    c->hDescs.release(); c->hResults.release(); c->hLargeIdx.release(); c->hRemain.release();
    for (cudaEvent_t e : c->sliceDone) if (e) cudaEventDestroy(e);
    if (c->ev0) { cudaEventDestroy(c->ev0); cudaEventDestroy(c->ev1); }
    for (cudaEvent_t e : c->stageEv) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : c->laneDone) if (e) cudaEventDestroy(e);
    if (c->forkEv) cudaEventDestroy(c->forkEv);
    for (cudaStream_t l : c->lane) if (l) cudaStreamDestroy(l);
    for (cudaStream_t l : c->side) if (l) cudaStreamDestroy(l);
    for (cudaEvent_t e : c->inDone) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : c->sideFork) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : c->sideJoin) if (e) cudaEventDestroy(e);
    if (c->ownStream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return 0;
}
ZL_EXPORT size_t ZSTD_DCtx_reset(ZSTD_DCtx* c, ZSTD_ResetDirective r)
{
    if (r == ZSTD_reset_session_only || r == ZSTD_reset_session_and_parameters) { c->sIn.clear(); c->sOut.clear(); c->sOutPos = 0; }
    if (r == ZSTD_reset_parameters || r == ZSTD_reset_session_and_parameters) {       // zstd.c:42548-42565
        c->forceIgnoreChecksum = 0; c->stableOut = 0; c->windowLogMax = 27;
        c->hasDict = false; c->dictRaw.clear();
    }
    return 0;
}
ZL_EXPORT size_t ZSTD_DCtx_setParameter(ZSTD_DCtx* c, ZSTD_dParameter p, int v)
{
    switch ((int)p) {
    case ZSTD_d_windowLogMax: if (v == 0) v = 27; if (v < 10 || v > 31) return ZL_ERROR(parameter_outOfBound); c->windowLogMax = v; return 0;
    case ZSTD_d_stableOutBuffer: if (v < 0 || v > 1) return ZL_ERROR(parameter_outOfBound); c->stableOut = v; return 0;
    case ZSTD_d_forceIgnoreChecksum: if (v < 0 || v > 1) return ZL_ERROR(parameter_outOfBound); c->forceIgnoreChecksum = v; return 0;
    default: return ZL_ERROR(parameter_unsupported);
    }
}
ZL_EXPORT size_t ZSTD_DCtx_getParameter(ZSTD_DCtx* c, ZSTD_dParameter p, int* v)
{
    switch ((int)p) {
    case ZSTD_d_windowLogMax: *v = c->windowLogMax; return 0;
    case ZSTD_d_stableOutBuffer: *v = c->stableOut; return 0;
    case ZSTD_d_forceIgnoreChecksum: *v = c->forceIgnoreChecksum; return 0;
    default: return ZL_ERROR(parameter_unsupported);
    }
}
ZL_EXPORT size_t zl_dctx_set_stream(ZSTD_DCtx* c, void* s)
{
    if (c->ownStream && c->stream) cudaStreamDestroy(c->stream);
    c->stream = (cudaStream_t)s; c->ownStream = false;
    if (!s) { c->ownStream = false; c->stream = nullptr; }
    return 0;
}
ZL_EXPORT size_t zl_dctx_set_profile(ZSTD_DCtx* c, int on) { c->profileStages = on ? 1 : 0; return 0; }
ZL_EXPORT unsigned long long zl_dctx_launch_count(const ZSTD_DCtx* c) { return c->launches; }
ZL_EXPORT double zl_dctx_last_kernel_ms(const ZSTD_DCtx* c) { return c->lastKernelMs; }
ZL_EXPORT double zl_dctx_last_stage_ms(const ZSTD_DCtx* c, int stage) { return stage >= 0 && stage < ZL_DEC_STAGES ? c->lastStageMs[stage] : -1.0; }

// Digest a dictionary (zstd.c:42053-42137 ZSTD_loadDEntropy, 42140 insertDictionary) into ZlDictDev.
ZL_EXPORT size_t ZSTD_DCtx_loadDictionary(ZSTD_DCtx* c, const void* dict, size_t dictSize)
{
    ZlDeviceGuard guard(zl_bind_device(&c->device));
    c->hasDict = false; c->dictRaw.clear(); c->dictGen++;
    if (!dict || !dictSize) return 0;
    c->dictRaw.assign((const u8*)dict, (const u8*)dict + dictSize);
    std::vector<u8> pad(dictSize + 16, 0);
    u8* d = pad.data() + 4 - (((size_t)pad.data()) & 3);            // 4-aligned copy for the word reader
    memcpy(d, dict, dictSize);
    ZlDictDev* hd = new (std::nothrow) ZlDictDev();
    if (!hd) return ZL_ERROR(memory_allocation);
    memset(hd, 0, sizeof(*hd));
    size_t contentOff = 0;
    if (dictSize >= 8 && zl_rd32(d) == ZL_MAGIC_DICT) {
        hd->dictID = zl_rd32(d + 4);
        ZlLitSm* f = new (std::nothrow) ZlLitSm();
        if (!f) { delete hd; return ZL_ERROR(memory_allocation); }
        memset(f, 0, sizeof(*f));
        size_t p = 8; bool ok = true;
        u32 th = zl_huf_read_stats(*f, d + p, (u32)(dictSize - p), (const u32*)d, 0, (u32)p);
        if (!th) ok = false;
        if (ok) { for (u32 q = 0; q < 4; q++) zl_huf_fill(*f, q); memcpy(hd->huf, f->huf, sizeof(hd->huf)); hd->hufLog = f->ctl.hufLog; p += th; }
        const u32 order[3] = {1, 2, 0}, maxSym[3] = {35, 31, 52}, maxLog[3] = {9, 8, 9};      // OF, ML, LL in the file
        for (int k = 0; ok && k < 3; k++) {
            u32 t = order[k], ms = maxSym[t], tl; i16 norm[64];
            u32 h = p < dictSize ? zl_read_ncount(d + p, (u32)(dictSize - p), norm, &ms, &tl) : 0;
            if (!h || tl > maxLog[t]) { ok = false; break; }
            u16* tbl = t == 0 ? hd->fseLL : (t == 1 ? hd->fseOF : hd->fseML);
            if (!zl_fse_build(tbl, norm, ms, tl)) { ok = false; break; }
            hd->tlog[t] = tl; p += h;
        }
        if (ok && p + 12 > dictSize) ok = false;
        if (ok) {
            size_t content = dictSize - (p + 12);
            for (int i = 0; i < 3; i++) { u32 r = zl_rd32(d + p + 4 * i); if (r == 0 || r > content) ok = false; hd->rep[i] = r; }
            contentOff = p + 12;
        }
        delete f;
        if (!ok) { delete hd; c->dictRaw.clear(); return ZL_ERROR(dictionary_corrupted); }
        hd->hasEntropy = 1;
    }
    hd->contentSize = (u32)(dictSize - contentOff);
    bool ok = c->dDictContent.reserve(hd->contentSize + 16) && c->dDict.reserve(sizeof(ZlDictDev));
    if (ok) {
        hd->content = c->dDictContent.as<u8>();
        ok = cudaMemcpy(c->dDictContent.p, d + contentOff, hd->contentSize, cudaMemcpyHostToDevice) == cudaSuccess &&
             cudaMemcpy(c->dDict.p, hd, sizeof(ZlDictDev), cudaMemcpyHostToDevice) == cudaSuccess;
    }
    delete hd;
    if (!ok) { (void)cudaGetLastError(); c->dictRaw.clear(); return ZL_ERROR(memory_allocation); }
    c->hasDict = true;
    return 0;
}
ZL_ALIAS(ZSTD_DCtx*, ZSTD_createDCtx, (void))
ZL_ALIAS(size_t, ZSTD_freeDCtx, (ZSTD_DCtx*))
ZL_ALIAS(size_t, ZSTD_DCtx_reset, (ZSTD_DCtx*, ZSTD_ResetDirective))
ZL_ALIAS(size_t, ZSTD_DCtx_setParameter, (ZSTD_DCtx*, ZSTD_dParameter, int))
ZL_ALIAS(size_t, ZSTD_DCtx_getParameter, (ZSTD_DCtx*, ZSTD_dParameter, int*))
ZL_ALIAS(size_t, ZSTD_DCtx_loadDictionary, (ZSTD_DCtx*, const void*, size_t))

// ---------------------------------------------------------------------------------------------- batched decode
static bool zl_dctx_lanes(ZSTD_DCtx* c)
{
    if (c->forkEv) return true;
    for (int i = 0; i < ZL_DEC_LANES; i++) {
        if (cudaStreamCreateWithFlags(&c->lane[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->laneDone[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->inDone[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaStreamCreateWithFlags(&c->side[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->sideFork[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->sideJoin[i], cudaEventDisableTiming) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    }
    if (cudaEventCreateWithFlags(&c->forkEv, cudaEventDisableTiming) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return true;
}

static size_t zl_decompress_batch_impl(ZSTD_DCtx* c, const void* const* src, const size_t* srcSize, void* const* dst,
                                       const size_t* dstCap, size_t* result, size_t n, int dev, bool worst);
static size_t zl_decompress_batch_one(ZSTD_DCtx* c, const void* const* src, const size_t* srcSize, void* const* dst,
                                      const size_t* dstCap, size_t* result, size_t n, int dev);
// extension: GPUs a context spreads batches of HOST buffers over (0: ZSTDLITE_GPUS, default 1); frames are independent, so the
// frame list is cut into contiguous ranges of about equal content, one per device, each decoded by a helper context on its own
// host thread (copies, kernels and staging of the devices overlap); no data moves between the devices
ZL_EXPORT size_t zl_dctx_set_gpus(ZSTD_DCtx* c, int n) { if (!c || n < 0) return ZL_ERROR(parameter_outOfBound); c->gpus = n; return 0; }
ZL_EXPORT size_t zl_decompress_batch(ZSTD_DCtx* c, const void* const* src, const size_t* srcSize, void* const* dst,
                                     const size_t* dstCap, size_t* result, size_t n, int dev)
{
    if (!c) return ZL_ERROR(GENERIC);
    const int home = zl_bind_device(&c->device);
    size_t G = dev ? 1 : (size_t)zl_gpu_count(c->gpus);
    unsigned long long content = 0;
    if (G > 1) for (size_t i = 0; i < n; i++) content += dstCap[i];
    if (G > n / 2) G = n / 2;
    if (G < 2 || content < ((unsigned long long)64 << 20)) return zl_decompress_batch_one(c, src, srcSize, dst, dstCap, result, n, dev);
    int ndev = 1;
    cudaGetDeviceCount(&ndev);
    while (c->kids.size() + 1 < G) {
        ZSTD_DCtx_s* k = new (std::nothrow) ZSTD_DCtx_s();
        if (!k) return ZL_ERROR(memory_allocation);
        k->device = (home + (int)c->kids.size() + 1) % ndev; k->gpus = 1;
        c->kids.push_back(k);
    }
    const std::vector<size_t> cut = zl_split_ranges(dstCap, n, G);
    std::vector<size_t> rc(G, 0);
    auto work = [&](size_t g) {
        ZSTD_DCtx_s* k = g ? c->kids[g - 1] : c;
        if (g) {
            k->forceIgnoreChecksum = c->forceIgnoreChecksum; k->windowLogMax = c->windowLogMax;
            if (k->dictGenSeen != c->dictGen) { rc[g] = ZSTD_DCtx_loadDictionary(k, c->dictRaw.data(), c->dictRaw.size()); k->dictGenSeen = c->dictGen; if (zl_is_error(rc[g])) return; }
        }
        const size_t a = cut[g], cnt = cut[g + 1] - a;
        rc[g] = cnt ? zl_decompress_batch_one(k, src + a, srcSize + a, dst + a, dstCap + a, result + a, cnt, 0) : 0;
    };
    std::vector<std::thread> th;
    for (size_t g = 1; g < G; g++) th.emplace_back(work, g);
    work(0);
    for (std::thread& t : th) t.join();
    for (size_t g = 1; g < G; g++) { c->launches += c->kids[g - 1]->launches; c->kids[g - 1]->launches = 0; if (c->kids[g - 1]->lastKernelMs > c->lastKernelMs) c->lastKernelMs = c->kids[g - 1]->lastKernelMs; }
    for (size_t g = 0; g < G; g++) if (zl_is_error(rc[g])) return rc[g];
    return 0;
}
static size_t zl_decompress_batch_one(ZSTD_DCtx* c, const void* const* src, const size_t* srcSize, void* const* dst,
                                      const size_t* dstCap, size_t* result, size_t n, int dev)
{
    ZlDeviceGuard guard(zl_bind_device(&c->device));
    if (!guard.ok) return ZL_ERROR(GENERIC);
    size_t r = zl_decompress_batch_impl(c, src, srcSize, dst, dstCap, result, n, dev, false);
    if (zl_is_error(r)) return r;
    bool retry = false;
    for (size_t i = 0; i < n; i++) if (result[i] == (size_t)0 - (size_t)ZL_E_INTERNAL_hdrCap) { retry = true; break; }
    if (retry) {                          // a frame with very many small blocks: run again with worst-case block arenas
        r = zl_decompress_batch_impl(c, src, srcSize, dst, dstCap, result, n, dev, true);
        if (zl_is_error(r)) return r;
        for (size_t i = 0; i < n; i++) if (result[i] == (size_t)0 - (size_t)ZL_E_INTERNAL_hdrCap) result[i] = ZL_ERROR(GENERIC);
    }
    return 0;
}
static size_t zl_decompress_batch_impl(ZSTD_DCtx* c, const void* const* src, const size_t* srcSize, void* const* dst,
                                       const size_t* dstCap, size_t* result, size_t n, int dev, bool worst)
{
    if (n == 0) return 0;
    static const ZlDecTuning tune = {getenv("ZL_DEC_SLICES") ? atoi(getenv("ZL_DEC_SLICES")) : 0, getenv("ZL_DEC_GRADE") ? atoi(getenv("ZL_DEC_GRADE")) : 6,
                                     getenv("ZL_DEC_NOGRADE") != nullptr, getenv("ZL_DEC_NODEVBUILD") != nullptr, getenv("ZL_DEC_NOSORT") != nullptr,
                                     getenv("ZL_DEC_NOMID") != nullptr, getenv("ZL_DEC_NOLAZY") != nullptr};      // (development switches)
    const auto hostT0 = std::chrono::steady_clock::now();
    auto hostMs = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - hostT0).count(); };
    ZlDecPlan p;
    if (const size_t r = zl_dec_plan(p, src, srcSize, dst, dstCap, n, dev != 0, worst, c->profileStages != 0, tune)) return r;
    if (!zl_ctx_stream(&c->stream, &c->ownStream, &c->ev0, &c->ev1)) return ZL_ERROR(memory_allocation);
    cudaStream_t st = c->stream;
    if (!c->hDescs.reserve(n * sizeof(ZlFrameDesc)) || !c->hResults.reserve(n * 8)) return ZL_ERROR(memory_allocation);
    ZlFrameDesc* hd = c->hDescs.as<ZlFrameDesc>();
    if (p.nslices > 1 && !zl_dctx_lanes(c)) zl_dec_plan(p, src, srcSize, dst, dstCap, n, dev != 0, worst, true, tune);     // no internal streams
    const size_t nslices = p.nslices;
    if (!dev && (!c->dSrc.reserve(p.srcTotal + 64) || !c->dDst.reserve(p.dstTotal + 64))) return ZL_ERROR(memory_allocation);
    // Scattered host buffers (a list of separately allocated objects: thousands of copy runs): one cudaMemcpyAsync per run would
    // cost more than the decode (~2.5 us each).  The runs of a slice are then packed into / unpacked from pinned staging
    // buffers by the host, and each slice moves with ONE copy per direction.
    // ... and PAGEABLE host buffers (what the reference's C layer passes: R vectors) are staged the same way: cudaMemcpyAsync on pageable
    // memory runs through the driver's staging on one thread (config 2: 8.4 GB/s end to end).  Staging is pipelined with the slices:
    // the host packs slice k+1 (zl_host.h, ZlCopyPool) while the device works on slice k, and unpacks slice k while k+1 is in flight.
    // (small pageable calls stay with the driver's path: its staging is fine below a few MiB)
    const bool stageIn = !dev && (p.sruns.size() > 64 + 2 * nslices || (p.srcTotal >= (4u << 20) && zl_is_pageable(p.sruns[0].hbase)));
    const bool stageOut = !dev && (p.druns.size() > 64 + 2 * nslices || (p.dstTotal >= (4u << 20) && zl_is_pageable(p.druns[0].hbase)));
    ZlStagePool& sp = ZlStagePool::get();
    std::unique_lock<std::mutex> stageLock(sp.m, std::defer_lock);
    if (stageIn || stageOut) stageLock.lock();
    if (stageIn && !sp.in.reserve(p.srcTotal + 64)) return ZL_ERROR(memory_allocation);
    if (stageOut && !sp.out.reserve(p.dstTotal + 64)) return ZL_ERROR(memory_allocation);
    if (stageOut && c->sliceDone.size() < nslices) {
        const size_t have = c->sliceDone.size();
        c->sliceDone.resize(nslices);
        for (size_t k = have; k < nslices; k++) if (cudaEventCreateWithFlags(&c->sliceDone[k], cudaEventDisableTiming) != cudaSuccess) { c->sliceDone.resize(k); return ZL_ERROR(memory_allocation); }
    }
    std::vector<ZlCopySeg> copySegs;
    const double tPlan = hostMs();
    // (filling the descriptors of >= 32,768 frames with the copy pool's threads was measured and lost: 1e5 small frames 2.94 ms against
    //  2.03 ms slice by slice on this thread -- waking the workers costs more than the 0.5 ms of stores they share)
    if (!p.lazyDescs && !p.devBuild) zl_plan_fill_descs(p, 0, n, p.base[0], c->dSrc.as<u8>(), c->dDst.as<u8>(), hd);
    if (p.devBuild && !c->dRaw.reserve(n * 32)) return ZL_ERROR(memory_allocation);
    const ZlArenaSums& tot = p.base[nslices];
    if (!c->dDescs.reserve(n * sizeof(ZlFrameDesc)) || !c->dInfos.reserve(n * sizeof(ZlFrameInfo)) || !c->dResults.reserve(n * 8) ||
        !c->dLit.reserve(tot.lit + 64) || !c->dRec.reserve(tot.rec * 8) ||
        !c->dNorm.reserve(nslices * (size_t)ZL_NORM_SLOTS * 3 * ZL_NORM_STRIDE * sizeof(i16)) ||
        !c->dHdr.reserve(tot.hdr * sizeof(ZlBlockHdr)) || !c->dUnits.reserve(tot.hdr * sizeof(ZlUnit)) || !c->dCounters.reserve(nslices * 16))
        return ZL_ERROR(memory_allocation);
    if (p.nLarge) {                             // scratch of the block-parallel path for large frames (zl_dec_large.cuh)
        if (!c->hLargeIdx.reserve(p.nLarge * 4) || !c->dLargeIdx.reserve(p.nLarge * 4) || !c->dLb.reserve(tot.hdr * sizeof(ZlLBlock)) ||
            !c->dLc.reserve(((tot.rec >> ZL_LCHUNK_LOG) + tot.hdr + 2) * sizeof(ZlLChunk)) ||
            !c->dParent.reserve(tot.par * 4 + 64) || !c->dRemain.reserve(nslices * 64 * sizeof(u32)) || !c->hRemain.reserve(nslices * 64))
            return ZL_ERROR(memory_allocation);
        u32* hLarge = c->hLargeIdx.as<u32>();
        size_t w = 0;
        for (size_t k = 0; k < nslices; k++) for (size_t i = p.cut[k]; i < p.cut[k + 1]; i++) if (hd[i].large) hLarge[w++] = (u32)(i - p.cut[k]);
        cudaMemcpyAsync(c->dLargeIdx.p, hLarge, p.nLarge * 4, cudaMemcpyHostToDevice, st);
    }
    size_t largeSeen = 0;
    const double tPrep = hostMs();
    if (!p.lazyDescs && !p.devBuild) cudaMemcpyAsync(c->dDescs.p, hd, n * sizeof(ZlFrameDesc), cudaMemcpyHostToDevice, st);
    if (!c->stageEv[0]) for (cudaEvent_t& e : c->stageEv) cudaEventCreate(&e);
    cudaEventRecord(c->ev0, st);
    if (nslices > 1) cudaEventRecord(c->forkEv, st);
    cudaError_t e = cudaSuccess;
    // per-kernel events: one slice on one stream, unless the batch is a few (large) frames that are not being profiled
    const bool stageTimed = nslices == 1 && (c->profileStages || n > 16);
    static const bool trace = getenv("ZL_DEC_TRACE") != nullptr;        // (development: per-slice timeline on stderr)
    std::vector<cudaEvent_t> tev;
    if (trace) { tev.resize(3 * nslices + 1); for (cudaEvent_t& x : tev) cudaEventCreate(&x); cudaEventRecord(tev[3 * nslices], st); }
    for (size_t k = 0; k < nslices && e == cudaSuccess; k++) {
        const size_t a = p.cut[k], cnt = p.cut[k + 1] - a;
        if (!cnt) continue;
        cudaStream_t ls = nslices > 1 ? c->lane[k % ZL_DEC_LANES] : st;
        if (nslices > 1 && k < ZL_DEC_LANES) cudaStreamWaitEvent(ls, c->forkEv, 0);
        if (!dev) {
            // host-to-device copies in slice order: each waits for the previous slice's (left alone, the copy engine served the
            // streams 0, 4, 1, 5, ...; a dedicated copy stream aliased a hardware queue with a lane and stalled behind its copy back)
            if (nslices > 1 && k > 0) cudaStreamWaitEvent(ls, c->inDone[(k - 1) % ZL_DEC_LANES], 0);
            const size_t r0 = p.srunCut[k], r1 = p.srunCut[k + 1];
            if (stageIn && r1 > r0) {
                u8* hs = sp.in.as<u8>();
                copySegs.clear();
                for (size_t r = r0; r < r1; r++) if (p.sruns[r].bytes) copySegs.push_back({hs + p.sruns[r].devOff, p.sruns[r].hbase, p.sruns[r].bytes});
                ZlCopyPool::get().run(copySegs);                       // (the device is busy with the slices before this one)
                const size_t o0 = p.sruns[r0].devOff, o1 = p.sruns[r1 - 1].devOff + p.sruns[r1 - 1].bytes;
                if (o1 > o0) cudaMemcpyAsync(c->dSrc.as<u8>() + o0, hs + o0, o1 - o0, cudaMemcpyHostToDevice, ls);
            } else if (!stageIn)
            for (size_t r = r0; r < r1; r++)
                if (p.sruns[r].bytes) cudaMemcpyAsync(c->dSrc.as<u8>() + p.sruns[r].devOff, p.sruns[r].hbase, p.sruns[r].bytes, cudaMemcpyHostToDevice, ls);
            if (nslices > 1) cudaEventRecord(c->inDone[k % ZL_DEC_LANES], ls);
        }
        if (p.devBuild) {
            static_assert(sizeof(size_t) == 8 && sizeof(void*) == 8, "the raw descriptor arrays are copied as u64");
            u64* hraw = reinterpret_cast<u64*>(hd) + 4 * a;                    // (the pinned descriptor buffer holds 80 bytes per frame)
            memcpy(hraw, src + a, cnt * 8); memcpy(hraw + cnt, dst + a, cnt * 8);
            memcpy(hraw + 2 * cnt, srcSize + a, cnt * 8); memcpy(hraw + 3 * cnt, dstCap + a, cnt * 8);
            cudaMemcpyAsync(c->dRaw.as<u64>() + 4 * a, hraw, cnt * 32, cudaMemcpyHostToDevice, ls);
            e = zl_launch_build_descs(c->dRaw.as<u64>() + 4 * a, (u32)cnt, c->dDescs.as<ZlFrameDesc>() + a, p.base[k].lit, p.base[k].rec, p.base[k].hdr, worst, ls);
            c->launches += 1;
            if (e != cudaSuccess) break;
        }
        if (p.lazyDescs) {
            zl_plan_fill_descs(p, a, a + cnt, p.base[k], c->dSrc.as<u8>(), c->dDst.as<u8>(), hd);
            cudaMemcpyAsync(c->dDescs.as<ZlFrameDesc>() + a, hd + a, cnt * sizeof(ZlFrameDesc), cudaMemcpyHostToDevice, ls);
        }
        if (trace) cudaEventRecord(tev[3 * k], ls);
        ZlDecodeLaunch L{};
        L.descs = c->dDescs.as<ZlFrameDesc>() + a; L.infos = c->dInfos.as<ZlFrameInfo>() + a; L.hdrArena = c->dHdr.as<ZlBlockHdr>();
        L.descsAll = c->dDescs.as<ZlFrameDesc>(); L.infosAll = c->dInfos.as<ZlFrameInfo>(); L.frameBase = (u32)a;
        L.recArena = c->dRec.as<u64>(); L.litArena = c->dLit.as<u8>();
        L.normArena = c->dNorm.as<i16>() + k * (size_t)ZL_NORM_SLOTS * 3 * ZL_NORM_STRIDE; L.normSlots = ZL_NORM_SLOTS;
        {   const u64 u0 = p.base[k].hdr, u1 = p.base[k + 1].hdr;                                   // the slice's share of the unit arena
            L.units = c->dUnits.as<ZlUnit>() + u0; L.unitCap = (u32)((u1 - u0) > 0xFFFFFFF0ull ? 0xFFFFFFF0ull : (u1 - u0)); }
        L.counters = c->dCounters.as<u32>() + 4 * k;
        if (p.nLarge) {
            L.largeIdx = c->dLargeIdx.as<u32>() + largeSeen;
            for (size_t i = a; i < a + cnt; i++) if (hd[i].large) {
                L.nLarge++;
                if (hd[i].hdrCap > L.largeMaxBlocks) L.largeMaxBlocks = hd[i].hdrCap;
                if (hd[i].dstCap > L.largeMaxBytes) L.largeMaxBytes = hd[i].dstCap;
            }
            largeSeen += L.nLarge;
            L.lbArena = c->dLb.as<ZlLBlock>(); L.lcArena = c->dLc.as<ZlLChunk>(); L.parentArena = c->dParent.as<u32>();
            L.remain = c->dRemain.as<u32>() + 64 * k; L.remainHost = c->hRemain.as<u32>() + 16 * k;
        }
        L.results = c->dResults.as<u64>() + a;
        L.nframes = (u32)cnt; L.verifyChecksum = !c->forceIgnoreChecksum; L.dict = c->hasDict ? c->dDict.as<ZlDictDev>() : nullptr;
        L.stageEv = stageTimed ? c->stageEv : nullptr;
        // host buffers only: literals next to sequences shortens the chain of a slice, i.e. the wait before its copy back can
        // start (measured 39.9 -> 41.4 GB/s end to end); device-resident batches are throughput-bound and lose (143 -> 125 GB/s)
        // ... and batches of a few (large) frames, whose block units leave most of the device idle: a 16 MiB frame 9.4 -> 6.8 ms
        const bool fewFrames = n <= 16 && nslices == 1 && !stageTimed && zl_dctx_lanes(c);
        if ((nslices > 1 && !dev) || fewFrames) { const int ln = (int)(k % ZL_DEC_LANES); L.side = c->side[ln]; L.sideFork = c->sideFork[ln]; L.sideJoin = c->sideJoin[ln]; }
        L.launched = &c->launches;
        e = zl_launch_decode(L, ls);
        if (trace) cudaEventRecord(tev[3 * k + 1], ls);
        const size_t r0 = p.drunCut[k], r1 = p.drunCut[k + 1];            // (none for device buffers)
        if (!dev && stageOut) {
            if (r1 > r0) {
                const size_t o0 = p.druns[r0].devOff, o1 = p.druns[r1 - 1].devOff + p.druns[r1 - 1].bytes;
                if (o1 > o0) cudaMemcpyAsync(sp.out.as<u8>() + o0, c->dDst.as<u8>() + o0, o1 - o0, cudaMemcpyDeviceToHost, ls);
            }
            cudaMemcpyAsync(c->hResults.as<u64>() + a, c->dResults.as<u64>() + a, cnt * 8, cudaMemcpyDeviceToHost, ls);
            cudaEventRecord(c->sliceDone[k], ls);
        } else
        for (size_t r = r0; r < r1; r++)
            if (p.druns[r].bytes) cudaMemcpyAsync((void*)p.druns[r].hbase, c->dDst.as<u8>() + p.druns[r].devOff, p.druns[r].bytes, cudaMemcpyDeviceToHost, ls);
        if (trace) cudaEventRecord(tev[3 * k + 2], ls);
    }
    if (nslices > 1)
        for (int i = 0; i < ZL_DEC_LANES; i++) { cudaEventRecord(c->laneDone[i], c->lane[i]); cudaStreamWaitEvent(st, c->laneDone[i], 0); }
    cudaEventRecord(c->ev1, st);
    if (e != cudaSuccess) { cudaStreamSynchronize(st); fprintf(stderr, "zstdlite_gpu: kernel launch failed: %s\n", cudaGetErrorString(e)); return ZL_ERROR(GENERIC); }
    const double tLaunch = hostMs();
    if (stageOut && e == cudaSuccess) {
        // unpack slice after slice as its copy back lands, while the later slices are still in flight
        for (size_t k = 0; k < nslices; k++) {
            if (p.cut[k + 1] == p.cut[k]) continue;
            if (cudaEventSynchronize(c->sliceDone[k]) != cudaSuccess) break;
            zl_plan_unstage(p, k, c->hResults.as<u64>(), sp.out.as<u8>(), copySegs);
            ZlCopyPool::get().run(copySegs);
        }
    }
    cudaMemcpyAsync(c->hResults.p, c->dResults.p, n * 8, cudaMemcpyDeviceToHost, st);
    e = cudaStreamSynchronize(st);
    const double tSync = hostMs();
    if (e != cudaSuccess) { fprintf(stderr, "zstdlite_gpu: device error: %s\n", cudaGetErrorString(e)); return ZL_ERROR(GENERIC); }
    float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1); c->lastKernelMs = ms;      // with host buffers this span includes the copies
    if (trace) {
        for (size_t k = 0; k < nslices; k++) {
            float t0 = 0, t1 = 0, t2 = 0;
            cudaEventElapsedTime(&t0, tev[3 * nslices], tev[3 * k]); cudaEventElapsedTime(&t1, tev[3 * nslices], tev[3 * k + 1]); cudaEventElapsedTime(&t2, tev[3 * nslices], tev[3 * k + 2]);
            fprintf(stderr, "slice %zu (%zu frames): h2d done %.2f, kernels done %.2f, d2h done %.2f ms\n", k, p.cut[k + 1] - p.cut[k], t0, t1, t2);
        }
        fprintf(stderr, "total %.2f ms; host: planned %.3f, descriptors ready %.3f, launches issued %.3f, synchronised %.3f ms\n", ms, tPlan, tPrep, tLaunch, tSync);
        for (cudaEvent_t x : tev) cudaEventDestroy(x);
    }
    for (int k = 0; k < ZL_DEC_STAGES; k++) {
        float t = -1.0f;
        if (stageTimed) cudaEventElapsedTime(&t, c->stageEv[k], c->stageEv[k + 1]);
        c->lastStageMs[k] = t;
    }
    const u64* hr = c->hResults.as<u64>();
    if (p.devBuild) memcpy(result, hr, n * 8);                                // (the caller's order was kept)
    else for (size_t pos = 0; pos < n; pos++) result[p.order[pos]] = (size_t)hr[pos];
    return 0;
}

// zstd.c:41798 ZSTD_decompressDCtx -> 41671 ZSTD_decompressMultiFrame: concatenated + skippable frames.
ZL_EXPORT size_t ZSTD_decompressDCtx(ZSTD_DCtx* c, void* dst, size_t dstCap, const void* srcv, size_t srcSize)
{
    const u8* src = (const u8*)srcv;
    std::vector<const void*> fsrc; std::vector<size_t> fsize, fcap, fres; std::vector<void*> fdst;
    size_t op = 0; bool more = false;
    auto flush = [&]() -> size_t {
        if (fsrc.empty()) return 0;
        fres.assign(fsrc.size(), 0);
        size_t r = zl_decompress_batch(c, fsrc.data(), fsize.data(), fdst.data(), fcap.data(), fres.data(), fsrc.size(), 0);
        if (zl_is_error(r)) return r;
        for (size_t k = 0; k < fres.size(); k++) if (zl_is_error(fres[k])) return fres[k];
        size_t last = fres.back();
        fsrc.clear(); fsize.clear(); fdst.clear(); fcap.clear();
        return last;
    };
    while (srcSize >= 5) {                                     // ZSTD_startingInputLength, zstd.c:41681
        if ((zl_rd32(src) & 0xFFFFFFF0u) == ZL_MAGIC_SKIP) {
            size_t sk = zl_host_find_frame_size(src, srcSize, nullptr);
            if (zl_is_error(sk)) return sk;
            src += sk; srcSize -= sk; more = true; continue;
        }
        ZlHostFrameHeader h;
        size_t r = zl_host_frame_header(&h, src, srcSize);
        if (zl_is_error(r)) { if (more && r == ZL_ERROR(prefix_unknown)) return ZL_ERROR(srcSize_wrong); return r; }   // zstd.c:41724-41729
        if (r > 0) return ZL_ERROR(srcSize_wrong);
        size_t fs = zl_host_find_frame_size(src, srcSize, nullptr);
        if (zl_is_error(fs)) return fs;
        if (h.contentSize != ZSTD_CONTENTSIZE_UNKNOWN) {
            if (h.contentSize > dstCap - op) return ZL_ERROR(dstSize_tooSmall);
            fsrc.push_back(src); fsize.push_back(fs); fdst.push_back((u8*)dst + op); fcap.push_back((size_t)h.contentSize);
            op += (size_t)h.contentSize;
        } else {                                               // size only known after decoding: run what we have, then this one alone
            size_t e = flush(); if (zl_is_error(e)) return e;
            fsrc.push_back(src); fsize.push_back(fs); fdst.push_back((u8*)dst + op); fcap.push_back(dstCap - op);
            e = flush(); if (zl_is_error(e)) return e;
            op += e;
        }
        src += fs; srcSize -= fs; more = true;
    }
    if (srcSize) return ZL_ERROR(srcSize_wrong);               // zstd.c:41766
    size_t e = flush(); if (zl_is_error(e)) return e;
    return op;
}
ZL_ALIAS(size_t, ZSTD_decompressDCtx, (ZSTD_DCtx*, void*, size_t, const void*, size_t))

// zstd.c:42687 ZSTD_decompressStream over the one-shot engine: all offered input is taken and kept until a complete frame
// is present (its end is found by walking the block headers, zstd.c:41335), the frame is decoded by the kernels into a
// host buffer and handed out in the caller's chunk sizes.  Returns 0 when a frame has been completely decoded and
// delivered, an error code, or a positive hint (bytes of output still held, or 1 when more input is needed).
ZL_EXPORT size_t ZSTD_decompressStream(ZSTD_DCtx* c, ZSTD_outBuffer* out, ZSTD_inBuffer* in)
{
    if (!c || !out || !in) return ZL_ERROR(GENERIC);
    if (out->pos > out->size) return ZL_ERROR(dstSize_tooSmall);
    if (in->pos > in->size) return ZL_ERROR(srcSize_wrong);
    if (in->size > in->pos) c->sIn.insert(c->sIn.end(), (const u8*)in->src + in->pos, (const u8*)in->src + in->size);
    in->pos = in->size;
    for (;;) {
        if (c->sOutPos < c->sOut.size()) {                        // deliver what is decoded
            const size_t room = out->size - out->pos, left = c->sOut.size() - c->sOutPos, k = room < left ? room : left;
            if (k) memcpy((u8*)out->dst + out->pos, c->sOut.data() + c->sOutPos, k);
            out->pos += k; c->sOutPos += k;
            if (c->sOutPos < c->sOut.size()) return c->sOut.size() - c->sOutPos;
            std::vector<u8>().swap(c->sOut); c->sOutPos = 0;
            if (c->sIn.empty()) return 0;
        }
        if (c->sIn.empty()) return 0;
        if (c->sIn.size() < 5) return 1;                          // not even a magic number + descriptor yet
        const u8* p = c->sIn.data();
        ZlHostFrameHeader h;
        const size_t hr = zl_host_frame_header(&h, p, c->sIn.size());
        if (zl_is_error(hr)) { c->sIn.clear(); return hr; }
        if (hr > 0) return 1;                                     // header incomplete
        unsigned nblocks = 0;
        const size_t fs = zl_host_find_frame_size(p, c->sIn.size(), &nblocks);
        if (fs == ZL_ERROR(srcSize_wrong)) return 1;              // frame incomplete: wait for more input
        if (zl_is_error(fs)) { c->sIn.clear(); return fs; }
        if (h.skippable) { c->sIn.erase(c->sIn.begin(), c->sIn.begin() + (ptrdiff_t)fs); if (c->sIn.empty()) return 0; continue; }
        // zstd.c:42800-42806: a streaming decoder refuses windows beyond ZSTD_d_windowLogMax before it allocates anything
        if (h.windowSize > (1ull << c->windowLogMax)) { c->sIn.clear(); return ZL_ERROR(frameParameter_windowTooLarge); }
        // nor does a header get memory its blocks cannot fill (a block regenerates <= blockSizeMax bytes): such a frame can only
        // end in corruption_detected (zstd.c:41646), so say it before allocating the claimed size on the host and ~8x that on the device
        if (h.contentSize != ZSTD_CONTENTSIZE_UNKNOWN && h.contentSize > (unsigned long long)nblocks * h.blockSizeMax) { c->sIn.clear(); return ZL_ERROR(corruption_detected); }
        const size_t cap = h.contentSize != ZSTD_CONTENTSIZE_UNKNOWN ? (size_t)h.contentSize : (size_t)nblocks * h.blockSizeMax;
        if (cap > 0x7FFFFFF0ull) { c->sIn.clear(); return ZL_ERROR(memory_allocation); }
        c->sOut.resize(cap ? cap : 1);
        const void* fsrc = p; void* fdst = c->sOut.data(); size_t fsz = fs, fcap = cap, fres = 0;
        const size_t r = zl_decompress_batch(c, &fsrc, &fsz, &fdst, &fcap, &fres, 1, 0);
        const size_t err = zl_is_error(r) ? r : (zl_is_error(fres) ? fres : 0);
        c->sIn.erase(c->sIn.begin(), c->sIn.begin() + (ptrdiff_t)fs);
        if (err) { c->sOut.clear(); c->sOutPos = 0; return err; }
        c->sOut.resize(fres); c->sOutPos = 0;
        if (!fres && c->sIn.empty()) return 0;
    }
}
ZL_ALIAS(size_t, ZSTD_decompressStream, (ZSTD_DCtx*, ZSTD_outBuffer*, ZSTD_inBuffer*))
