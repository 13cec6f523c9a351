// lsdgpu.cu -- C ABI (include/lsdgpu.h) over the sm_100a kernels in frame.cuh / track.cuh / depth.cuh.
// Host-side control flow mirrors SE3Tracker::trackFrame (Tracking/SE3Tracker.cpp:280-486) and
// DepthMap::updateKeyframe / createKeyFrame / finalizeKeyFrame (DepthEstimation/DepthMap.cpp:1072-1395).
#include "internal.cuh"
#include "frame.cuh"
#include "track.cuh"
#include "depth.cuh"
#include "seqsum.cuh"
#include "track_persistent.cuh"
#include "perma.cuh"
#include "sim3.cuh"
#include "output.cuh"
#include "mapexport.cuh"

#include <algorithm>
#include <stdlib.h>
#include <new>

#define LAUNCH(ctx) ((ctx)->launches++)

// ------------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------------
extern "C" int lsdgpu_abi_version(void) { return LSDGPU_ABI_VERSION; }

extern "C" void lsdgpu_default_globals(lsdgpu_globals* g)
{
    g->minUseGrad = 5; g->cameraPixelNoise2 = 4 * 4; g->depthSmoothingFactor = 1;
    g->allowNegativeIdepths = 1; g->useSubpixelStereo = 1; g->useAffineLightningEstimation = 1;
}

extern "C" void lsdgpu_default_track_settings(lsdgpu_track_settings* s)
{
    static const int maxIterations[6] = { 5, 20, 50, 100, 100, 100 };
    s->lambdaSuccessFac = 0.5f; s->lambdaFailFac = 2.0f;
    for (int l = 0; l < LSD_LEVELS; l++) {
        s->lambdaInitial[l] = 0; s->stepSizeMin[l] = 1e-8f; s->convergenceEps[l] = 0.999f;
        s->maxItsPerLvl[l] = maxIterations[l];
    }
    s->var_weight = 1.0f; s->huber_d = 3;
}

static size_t alignUp(size_t v, size_t a) { return (v + a - 1) / a * a; }

static void setupCams(lsdgpu_ctx* ctx, const float K[9])
{   // Frame::initialize, DataStructures/Frame.cpp:403-459
    LevelCam& c0 = ctx->cam[0];
    memcpy(c0.K, K, 36);
    c0.w = ctx->w; c0.h = ctx->h;
    c0.fx = K[0]; c0.fy = K[4]; c0.cx = K[2]; c0.cy = K[5];
    lsd::mat3Inverse(c0.K, c0.KInv);
    c0.fxi = c0.KInv[0]; c0.fyi = c0.KInv[4]; c0.cxi = c0.KInv[2]; c0.cyi = c0.KInv[5];
    for (int l = 1; l < LSD_LEVELS; l++) {
        LevelCam& c = ctx->cam[l];
        c.w = ctx->w >> l; c.h = ctx->h >> l;
        c.fx = (float)(ctx->cam[l - 1].fx * 0.5);
        c.fy = (float)(ctx->cam[l - 1].fy * 0.5);
        c.cx = (float)((c0.cx + 0.5) / ((int)1 << l) - 0.5);
        c.cy = (float)((c0.cy + 0.5) / ((int)1 << l) - 0.5);
        float Kl[9] = { c.fx, 0.f, c.cx, 0.f, c.fy, c.cy, 0.f, 0.f, 1.f };
        memcpy(c.K, Kl, 36);
        lsd::mat3Inverse(c.K, c.KInv);
        c.fxi = c.KInv[0]; c.fyi = c.KInv[4]; c.cxi = c.KInv[2]; c.cyi = c.KInv[5];
    }
}

extern "C" int lsdgpu_create(int device, int width, int height, const float K[9], int max_frames, lsdgpu_ctx** out)
{
    if (!out) return -2;
    *out = nullptr;
    if (width <= 0 || height <= 0 || (width % 16) || (height % 16) || max_frames < 2) return -2;   // SlamSystem.cpp:55
    lsdgpu_ctx* ctx = new (std::nothrow) lsdgpu_ctx();
    if (!ctx) return -3;
    *out = ctx;      // returned even on failure so that lsdgpu_last_error can be read
    ctx->device = device; ctx->w = width; ctx->h = height;
    lsdgpu_default_globals(&ctx->g);
    setupCams(ctx, K);
    LSD_CHECK(ctx, cudaSetDevice(device));
    cudaDeviceProp prop;
    LSD_CHECK(ctx, cudaGetDeviceProperties(&prop, device));
    ctx->smCount = prop.multiProcessorCount;
    LSD_CHECK(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));

    const size_t n0 = (size_t)width * height;
    size_t perFrame = 0;
    for (int l = 0; l < LSD_LEVELS; l++) {
        size_t n = n0 >> (2 * l);
        perFrame += alignUp(n * 4, 256) + alignUp(n * 16, 256) + 2 * alignUp(n * 4, 256);
    }
    perFrame += alignUp(n0 * 4, 256) + alignUp(n0 / 4, 256);
    size_t depthBytes = 2 * (alignUp(n0 * 16, 256) * 2) + alignUp(n0 * 4, 256)           // cur/oth hf+hi, integral
                        + 2 * alignUp(n0 * 4, 256) + alignUp(n0 * 16, 256);              // prop head/next/val
    const int maxBlocks = divUp((int)n0, EVAL_THREADS) + 8;
    size_t scratch = alignUp((size_t)maxBlocks * EV_NCH * 4 + 65536, 256) + 4096 + alignUp(sizeof(ObserveParams), 256)
                     + 2 * alignUp(n0, 256) + alignUp(n0 * 32, 256) + alignUp((size_t)maxBlocks * 2 * 8 + 64, 256) + (256 + 2 * alignUp((n0 >> 8) * 16, 256) + 2 * alignUp(n0 * 4, 256) + alignUp(n0, 256)) * (size_t)max_frames + alignUp(n0 * 12, 256) + alignUp(LSD_MAX_PERMA_BATCH * (sizeof(PermaItem) + sizeof(PermaResult)), 256) + 1024 + alignUp(S3_MAX_BATCH * sizeof(Sim3Item), 256) + alignUp(S3_MAX_BATCH * sizeof(Sim3Out), 256)
                     + alignUp(sizeof(TrackState), 256) + alignUp(sizeof(ObserveParams), 256) + 8192 + TP_SYNC_WORDS * 4;
    const int seqRuns = divUp((int)n0, SEQ_RUN);
    scratch += alignUp((size_t)seqRuns * SEQ_NBIN * sizeof(int2), 256) + alignUp((size_t)seqRuns, 256) + alignUp((size_t)seqRuns * 4, 256);
    ctx->arenaBytes = perFrame * max_frames + depthBytes + scratch;
    LSD_CHECK(ctx, cudaMalloc((void**)&ctx->arena, ctx->arenaBytes));
    LSD_CHECK(ctx, cudaMemsetAsync(ctx->arena, 0, ctx->arenaBytes, ctx->stream));
    char* p = ctx->arena;
    auto take = [&](size_t bytes) { char* r = p; p += alignUp(bytes, 256); return r; };
    ctx->slots.resize(max_frames);
    for (auto& s : ctx->slots) {
        for (int l = 0; l < LSD_LEVELS; l++) {
            size_t n = n0 >> (2 * l);
            s.image[l] = (float*)take(n * 4);
            s.grad[l] = (float4*)take(n * 16);
            s.idepth[l] = (float*)take(n * 4);
            s.idepthVar[l] = (float*)take(n * 4);
        }
        s.maxgrad = (float*)take(n0 * 4);
        s.goodMask = (uint8_t*)take(n0 / 4);
        memset(s.thisToParent, 0, sizeof(s.thisToParent));
        s.thisToParent[3] = 1; s.thisToParent[7] = 1;
    }
    // TMA descriptors for the tracker's shared-memory windows (one per slot and level)
    {
        cudaDriverEntryPointQueryResult qres;
        LSD_CHECK(ctx, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ctx->encodeTiled, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !ctx->encodeTiled) return lsd_fail(ctx, "cuTensorMapEncodeTiled not available in this driver");
        typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                     const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
        EncodeFn enc = (EncodeFn)ctx->encodeTiled;
        for (auto& s : ctx->slots)
            for (int l = 0; l < LSD_LEVELS; l++) {
                const cuuint64_t gdim[2] = { (cuuint64_t)4 * (width >> l), (cuuint64_t)(height >> l) };
                const cuuint64_t gstr[1] = { (cuuint64_t)16 * (width >> l) };
                const cuuint32_t box[2] = { 4 * TRK_WIN_W, TRK_WIN_H };
                const cuuint32_t estr[2] = { 1, 1 };
                CUresult cr = enc(&s.gradMap[l], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)s.grad[l], gdim, gstr, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                if (cr != CUDA_SUCCESS) return lsd_fail(ctx, "cuTensorMapEncodeTiled failed");
            }
    }
    ctx->cur.hf = (float4*)take(n0 * 16); ctx->cur.hi = (int4*)take(n0 * 16);
    ctx->oth.hf = (float4*)take(n0 * 16); ctx->oth.hi = (int4*)take(n0 * 16);
    ctx->integral = (int*)take(n0 * 4);
    ctx->propHead = (int*)take(n0 * 4);
    ctx->propNext = (int*)take(n0 * 4);
    ctx->propVal = (float4*)take(n0 * 16);
    ctx->evPartials = (float*)take((size_t)maxBlocks * EV_NCH * 4 + 65536);   // also holds the 2 x 160 x 192 B exchange rows of mode 1
    ctx->evCounter = (unsigned int*)take(256);
    ctx->trkSync = (unsigned int*)take(TP_SYNC_WORDS * 4);
    ctx->dEvOut = (float*)take(EV_NCH * 4);
    ctx->dStageU8[0] = (uint8_t*)take(n0);
    ctx->dStageU8[1] = (uint8_t*)take(n0);
    for (auto& s : ctx->slots) {
        s.dStats = (double*)take(64);
        s.permaPC = (float4*)take((n0 >> 8) * 16);
        s.permaVar = (float*)take((n0 >> 8) * 4);
        s.reactIdepth = (float*)take(n0 * 4);
        s.reactVar = (float*)take(n0 * 4);
        s.reactValidity = (uint8_t*)take(n0);
    }
    ctx->dPacked = (uint32_t*)take(n0 * 12);
    ctx->dPermaItems = take(LSD_MAX_PERMA_BATCH * sizeof(PermaItem));
    ctx->dPermaResults = take(LSD_MAX_PERMA_BATCH * sizeof(PermaResult));
    ctx->dSim3Items = take(S3_MAX_BATCH * sizeof(Sim3Item));
    ctx->dSim3Outs = take(S3_MAX_BATCH * sizeof(Sim3Out));
    ctx->dStageF = (float*)take(n0 * 32);
    ctx->dScalars = (double*)take((size_t)maxBlocks * 2 * 8 + 64);
    ctx->dTrackState = take(sizeof(TrackState));
    ctx->dObs = (ObserveParams*)take(sizeof(ObserveParams));
    ctx->dSkipFlag = (int*)take(256);
    ctx->seqTable = (int2*)take((size_t)seqRuns * SEQ_NBIN * sizeof(int2));
    ctx->seqFlags = (unsigned char*)take((size_t)seqRuns);
    ctx->seqCounts = (int*)take((size_t)seqRuns * 4);
    if ((size_t)(p - ctx->arena) > ctx->arenaBytes) return lsd_fail(ctx, "arena overflow");

    LSD_CHECK(ctx, cudaHostAlloc((void**)&ctx->hEvOut, EV_NCH * 4, cudaHostAllocDefault));
    for (int i = 0; i < 2; i++) {
        LSD_CHECK(ctx, cudaHostAlloc((void**)&ctx->hStage[i], n0, cudaHostAllocDefault));
        LSD_CHECK(ctx, cudaEventCreateWithFlags(&ctx->stageDone[i], cudaEventDisableTiming));
        LSD_CHECK(ctx, cudaEventRecord(ctx->stageDone[i], ctx->stream));
    }
    LSD_CHECK(ctx, cudaHostAlloc((void**)&ctx->hStageF, n0 * 32, cudaHostAllocDefault));
    LSD_CHECK(ctx, cudaHostAlloc((void**)&ctx->hScalars, 64, cudaHostAllocDefault));
    // the tracker writes its result block straight into mapped pinned memory (no D2H copy on the path)
    LSD_CHECK(ctx, cudaHostAlloc((void**)&ctx->hTrackState, sizeof(TrackState), cudaHostAllocMapped));
    // cudaHostAlloc does not clear: a recycled block may still hold the result of a destroyed context, whose doneSeq would satisfy
    // the completion spin of this context's first launches (trackPersistentFinish) before the kernel has written anything
    memset(ctx->hTrackState, 0, sizeof(TrackState));
    memset(ctx->hScalars, 0, 64);
    memset(ctx->hEvOut, 0, EV_NCH * 4);
    LSD_CHECK(ctx, cudaHostGetDevicePointer(&ctx->dTrackStateMapped, ctx->hTrackState, 0));
    for (int i = 0; i < 8; i++) {
        LSD_CHECK(ctx, cudaEventCreate(&ctx->tBegin[i]));
        LSD_CHECK(ctx, cudaEventCreate(&ctx->tEnd[i]));
    }
    LSD_CHECK(ctx, cudaEventCreate(&ctx->kBegin));
    LSD_CHECK(ctx, cudaEventCreate(&ctx->kEnd));
    LSD_CHECK(ctx, trackPersistentSetup(ctx));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

static void peerCloseAll(lsdgpu_ctx* ctx);
static void mapStagingFree(lsdgpu_ctx* ctx);

extern "C" void lsdgpu_destroy(lsdgpu_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    peerCloseAll(ctx);
    mapStagingFree(ctx);
    cudaFree(ctx->arena);
    if (ctx->stageRing) cudaFree(ctx->stageRing);
    if (ctx->dRemapX) cudaFree(ctx->dRemapX);
    if (ctx->dRemapY) cudaFree(ctx->dRemapY);
    if (ctx->dRaw) cudaFree(ctx->dRaw);
    if (ctx->hRaw) cudaFreeHost(ctx->hRaw);
    cudaFreeHost(ctx->hEvOut); cudaFreeHost(ctx->hStage[0]); cudaFreeHost(ctx->hStage[1]); cudaFreeHost(ctx->hStageF);
    cudaEventDestroy(ctx->stageDone[0]); cudaEventDestroy(ctx->stageDone[1]);
    cudaFreeHost(ctx->hScalars); cudaFreeHost(ctx->hTrackState);
    for (int i = 0; i < 8; i++) { if (ctx->tBegin[i]) cudaEventDestroy(ctx->tBegin[i]); if (ctx->tEnd[i]) cudaEventDestroy(ctx->tEnd[i]); }
    if (ctx->kBegin) cudaEventDestroy(ctx->kBegin);
    if (ctx->kEnd) cudaEventDestroy(ctx->kEnd);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char* lsdgpu_last_error(const lsdgpu_ctx* ctx) {   // a copy per calling thread: another thread may fail (and overwrite ctx->err) right after this one
    static thread_local std::string mine;
    if (!ctx) return "null context";
    LSD_LOCK(ctx);
    mine = ctx->err;
    return mine.c_str();
}
extern "C" int lsdgpu_set_globals(lsdgpu_ctx* ctx, const lsdgpu_globals* g) { LSD_LOCK(ctx); ctx->g = *g; return 0; }
extern "C" int lsdgpu_get_globals(const lsdgpu_ctx* ctx, lsdgpu_globals* g) { LSD_LOCK(ctx); *g = ctx->g; return 0; }
extern "C" int lsdgpu_synchronize(lsdgpu_ctx* ctx)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
extern "C" long long lsdgpu_launch_count(const lsdgpu_ctx* ctx) { LSD_LOCK(ctx); return ctx->launches; }

extern "C" int lsdgpu_timer_begin(lsdgpu_ctx* ctx, int slot)
{ LSD_LOCK(ctx);
    if (slot < 0 || slot >= 8) return -2;
    LSD_CHECK(ctx, cudaEventRecord(ctx->tBegin[slot], ctx->stream));
    return 0;
}
extern "C" int lsdgpu_timer_end(lsdgpu_ctx* ctx, int slot)
{ LSD_LOCK(ctx);
    if (slot < 0 || slot >= 8) return -2;
    LSD_CHECK(ctx, cudaEventRecord(ctx->tEnd[slot], ctx->stream));
    return 0;
}
extern "C" int lsdgpu_timer_elapsed_ms(lsdgpu_ctx* ctx, int slot, float* ms)
{ LSD_LOCK(ctx);
    if (slot < 0 || slot >= 8) return -2;
    LSD_CHECK(ctx, cudaEventSynchronize(ctx->tEnd[slot]));
    LSD_CHECK(ctx, cudaEventElapsedTime(ms, ctx->tBegin[slot], ctx->tEnd[slot]));
    return 0;
}
static void flushTrackProfile(lsdgpu_ctx* ctx);
extern "C" int lsdgpu_track_kernel_stats(lsdgpu_ctx* ctx, int reset, double* ms, long long* launches, double* bytes)
{ LSD_LOCK(ctx);
    flushTrackProfile(ctx);
    if (ms) *ms = ctx->trackKernelMs;
    if (launches) *launches = ctx->trackKernelLaunches;
    if (bytes) *bytes = ctx->trackKernelBytes;
    if (reset == 1) { ctx->trackKernelMs = 0; ctx->trackKernelLaunches = 0; ctx->trackKernelBytes = 0; ctx->profileTrackKernel = true; }
    if (reset == 2) ctx->profileTrackKernel = false;
    return 0;
}

// ------------------------------------------------------------------------------------------------------
// frames
// ------------------------------------------------------------------------------------------------------
static FrameSlot* acquireSlot(lsdgpu_ctx* ctx, int id)
{
    FrameSlot* s = findSlot(ctx, id);
    if (s) return s;
    for (auto& c : ctx->slots)
        if (!c.used) {
            FrameSlot fresh = c;          // keep the pointers
            fresh.id = id; fresh.used = true;
            fresh.hasDepth = fresh.idepthPyrValid = fresh.hasGoodMask = false;
            fresh.depthHasBeenUpdatedFlag = false;
            fresh.meanIdepth = 1.f; fresh.numPoints = 0; fresh.statsPending = false;
            memset(fresh.thisToParent, 0, sizeof(fresh.thisToParent));
            fresh.thisToParent[3] = 1; fresh.thisToParent[7] = 1;
            fresh.parentId = -1; fresh.initialTrackedResidual = 0;
            fresh.numFramesTrackedOnThis = fresh.numMappedOnThis = 0;
            fresh.permaNumPts = 0;
            fresh.reactAllocated = false; fresh.reactValid = false;
            c = fresh;
            return &c;
        }
    return nullptr;
}

static int buildFrameFromDeviceU8(lsdgpu_ctx* ctx, FrameSlot* s, const uint8_t* dsrc, bool remap = false);

extern "C" int lsdgpu_frame_upload_u8(lsdgpu_ctx* ctx, int frame_id, const uint8_t* gray)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* s = acquireSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "no free frame slot (release frames or raise max_frames)");
    const size_t n0 = (size_t)ctx->w * ctx->h;
    // double-buffered staging: only wait for the upload issued two frames ago.  A caller buffer that is already
    // page-locked (cudaHostAlloc / cudaHostRegister, e.g. a camera DMA buffer) is copied from directly -- it must then
    // stay untouched until the frame has been consumed; pageable memory goes through the pinned staging copy.
    const int b = ctx->stageIdx;
    ctx->stageIdx ^= 1;
    LSD_CHECK(ctx, cudaEventSynchronize(ctx->stageDone[b]));
    cudaPointerAttributes pa;
    const bool pinned = cudaPointerGetAttributes(&pa, gray) == cudaSuccess && pa.type == cudaMemoryTypeHost;
    if (!pinned) { cudaGetLastError(); memcpy(ctx->hStage[b], gray, n0); }
    LSD_CHECK(ctx, cudaMemcpyAsync(ctx->dStageU8[b], pinned ? gray : ctx->hStage[b], n0, cudaMemcpyHostToDevice, ctx->stream));
    int r = buildFrameFromDeviceU8(ctx, s, ctx->dStageU8[b]);
    LSD_CHECK(ctx, cudaEventRecord(ctx->stageDone[b], ctx->stream));
    return r;
}

extern "C" int lsdgpu_stage_reserve(lsdgpu_ctx* ctx, int n_entries)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    if (n_entries <= 0) return lsd_fail(ctx, "bad ring size");
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->stageRing) { cudaFree(ctx->stageRing); ctx->stageRing = nullptr; ctx->stageEntries = 0; }
    LSD_CHECK(ctx, cudaMalloc((void**)&ctx->stageRing, (size_t)n_entries * ctx->w * ctx->h));
    ctx->stageEntries = n_entries;
    return 0;
}
extern "C" int lsdgpu_stage_put(lsdgpu_ctx* ctx, int index, const uint8_t* gray)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    if (index < 0 || index >= ctx->stageEntries) return lsd_fail(ctx, "bad ring index");
    const size_t n0 = (size_t)ctx->w * ctx->h;
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(ctx->hStage[0], gray, n0);
    LSD_CHECK(ctx, cudaMemcpyAsync(ctx->stageRing + (size_t)index * n0, ctx->hStage[0], n0, cudaMemcpyHostToDevice, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
extern "C" int lsdgpu_frame_from_stage(lsdgpu_ctx* ctx, int frame_id, int index)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    if (index < 0 || index >= ctx->stageEntries) return lsd_fail(ctx, "bad ring index");
    FrameSlot* s = acquireSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "no free frame slot (release frames or raise max_frames)");
    return buildFrameFromDeviceU8(ctx, s, ctx->stageRing + (size_t)index * ctx->w * ctx->h);
}

static int buildFrameFromDeviceU8(lsdgpu_ctx* ctx, FrameSlot* s, const uint8_t* dsrc, bool remap)
{
    const int w = ctx->w, h = ctx->h;
    PyrPtrs pp;
    for (int l = 0; l < LSD_LEVELS; l++) pp.l[l] = s->image[l];
    if (remap) k_image_pyramid<true><<<dim3(w / 16, h / 16), 256, 0, ctx->stream>>>(dsrc, pp, w, h, ctx->dRemapX, ctx->dRemapY, ctx->rawW, nullptr);
    else k_image_pyramid<false><<<dim3(w / 16, h / 16), 256, 0, ctx->stream>>>(dsrc, pp, w, h);
    LAUNCH(ctx);
    GradPtrs gp;
    for (int l = 0; l < LSD_LEVELS; l++) { gp.img[l] = s->image[l]; gp.grad[l] = s->grad[l]; gp.w[l] = w >> l; gp.h[l] = h >> l; }
    gp.maxgrad0 = s->maxgrad;
    // blockIdx.y = level; level 0 runs as 32x8 tiles, levels 1..4 linearly (their block counts are smaller than the tile count)
    LSD_CHECK(ctx, launchPDL(k_gradients, dim3(divUp(w, GR_TW) * divUp(h, GR_TH), LSD_LEVELS), dim3(256), 0, ctx->stream, ctx->optPdl, gp));      // + maxGradients of level 0
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    s->hasDepth = false; s->idepthPyrValid = false; s->hasGoodMask = false;
    return 0;
}

extern "C" int lsdgpu_frame_release(lsdgpu_ctx* ctx, int frame_id)
{ LSD_LOCK(ctx);
    FrameSlot* s = findSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "unknown frame id");
    if (ctx->activeKf == frame_id) return lsd_fail(ctx, "frame is the active keyframe of the depth map");
    s->used = false; s->id = -1;
    return 0;
}

static int ensureIdepthPyramid(lsdgpu_ctx* ctx, FrameSlot* s)
{
    if (!s->hasDepth) return lsd_fail(ctx, "keyframe has no depth");
    if (s->idepthPyrValid) return 0;
    PyrPtrs id, var;
    for (int l = 0; l < LSD_LEVELS; l++) { id.l[l] = s->idepth[l]; var.l[l] = s->idepthVar[l]; }
    k_idepth_pyramid<<<dim3(ctx->w / 16, ctx->h / 16), 256, 0, ctx->stream>>>(id, var, ctx->w, ctx->h);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    s->idepthPyrValid = true;
    return 0;
}

extern "C" int lsdgpu_frame_download(lsdgpu_ctx* ctx, int frame_id, int what, int level, void* out)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* s = findSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "unknown frame id");
    if (level < 0 || level >= LSD_LEVELS) return lsd_fail(ctx, "bad level");
    const size_t n = ((size_t)ctx->w * ctx->h) >> (2 * level);
    const void* src = nullptr;
    size_t bytes = 0;
    switch (what) {
    case LSDGPU_BUF_IMAGE: src = s->image[level]; bytes = n * 4; break;
    case LSDGPU_BUF_GRADIENTS: src = s->grad[level]; bytes = n * 16; break;
    case LSDGPU_BUF_MAXGRAD: if (level != 0) return lsd_fail(ctx, "maxGradients exists at level 0 only"); src = s->maxgrad; bytes = n * 4; break;
    case LSDGPU_BUF_IDEPTH:
    case LSDGPU_BUF_IDEPTH_VAR:
        if (!s->hasDepth) return lsd_fail(ctx, "frame has no depth");
        if (level > 0) { int r = ensureIdepthPyramid(ctx, s); if (r) return r; }
        src = (what == LSDGPU_BUF_IDEPTH) ? s->idepth[level] : s->idepthVar[level]; bytes = n * 4; break;
    case LSDGPU_BUF_GOODMASK:
        if (!s->hasGoodMask) { memset(out, 1, ((size_t)ctx->w * ctx->h) / 4); return 0; }   // Frame.h:433: initialised to true
        src = s->goodMask; bytes = ((size_t)ctx->w * ctx->h) / 4; break;
    default: return lsd_fail(ctx, "bad buffer selector");
    }
    LSD_CHECK(ctx, cudaMemcpyAsync(out, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int lsdgpu_frame_set_depth_gt(lsdgpu_ctx* ctx, int frame_id, const float* depth, float cov_scale)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* s = findSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "unknown frame id");
    const int n = ctx->w * ctx->h;
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(ctx->hStageF, depth, (size_t)n * 4);
    LSD_CHECK(ctx, cudaMemcpyAsync(ctx->dStageF, ctx->hStageF, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    k_set_depth_gt<<<divUp(n, 256), 256, 0, ctx->stream>>>(ctx->dStageF, s->maxgrad, s->idepth[0], s->idepthVar[0], ctx->w, ctx->h,
                                                           ctx->g.minUseGrad, cov_scale);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    s->hasDepth = true; s->idepthPyrValid = false;
    return 0;
}

extern "C" int lsdgpu_frame_set_idepth(lsdgpu_ctx* ctx, int frame_id, const float* idepth, const float* idepthVar)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* s = findSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "unknown frame id");
    const size_t n = (size_t)ctx->w * ctx->h;
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(ctx->hStageF, idepth, n * 4);
    memcpy(ctx->hStageF + n, idepthVar, n * 4);
    LSD_CHECK(ctx, cudaMemcpyAsync(s->idepth[0], ctx->hStageF, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    LSD_CHECK(ctx, cudaMemcpyAsync(s->idepthVar[0], ctx->hStageF + n, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    s->hasDepth = true; s->idepthPyrValid = false;
    return 0;
}

extern "C" int lsdgpu_frame_set_pose(lsdgpu_ctx* ctx, int frame_id, const double qts[8], int parent_id, float itr)
{ LSD_LOCK(ctx);
    FrameSlot* s = findSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "unknown frame id");
    memcpy(s->thisToParent, qts, sizeof(s->thisToParent));
    s->parentId = parent_id; s->initialTrackedResidual = itr;
    return 0;
}
extern "C" int lsdgpu_frame_get_pose(lsdgpu_ctx* ctx, int frame_id, double qts[8], int* parent_id, float* itr)
{ LSD_LOCK(ctx);
    FrameSlot* s = findSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "unknown frame id");
    if (qts) memcpy(qts, s->thisToParent, sizeof(s->thisToParent));
    if (parent_id) *parent_id = s->parentId;
    if (itr) *itr = s->initialTrackedResidual;
    return 0;
}
extern "C" int lsdgpu_frame_get_counters(lsdgpu_ctx* ctx, int frame_id, int* tracked, int* mapped)
{ LSD_LOCK(ctx);
    FrameSlot* s = findSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "unknown frame id");
    if (tracked) *tracked = s->numFramesTrackedOnThis;
    if (mapped) *mapped = s->numMappedOnThis;
    return 0;
}
extern "C" int lsdgpu_frame_set_counters(lsdgpu_ctx* ctx, int frame_id, int tracked, int mapped)
{ LSD_LOCK(ctx);
    FrameSlot* s = findSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "unknown frame id");
    s->numFramesTrackedOnThis = tracked; s->numMappedOnThis = mapped;
    return 0;
}
extern "C" int lsdgpu_frame_get_depth_stats(lsdgpu_ctx* ctx, int frame_id, float* meanIdepth, int* numPoints, int* flag)
{ LSD_LOCK(ctx);
    FrameSlot* s = findSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "unknown frame id");
    if ((meanIdepth || numPoints) && s->statsPending) {      // fetched lazily: keeps updateKeyframe free of host syncs
        LSD_CHECK(ctx, cudaSetDevice(ctx->device));
        LSD_CHECK(ctx, cudaMemcpyAsync(ctx->hScalars, s->dStats, 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
        s->numPoints = (int)ctx->hScalars[1];
        s->meanIdepth = (float)ctx->hScalars[0] / (float)s->numPoints;     // Frame.cpp:234
        s->statsPending = false;
    }
    if (meanIdepth) *meanIdepth = s->meanIdepth;
    if (numPoints) *numPoints = s->numPoints;
    if (flag) *flag = s->depthHasBeenUpdatedFlag ? 1 : 0;
    return 0;
}
extern "C" int lsdgpu_frame_clear_good_mask(lsdgpu_ctx* ctx, int frame_id)
{ LSD_LOCK(ctx);
    FrameSlot* s = findSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "unknown frame id");
    s->hasGoodMask = false;
    return 0;
}

// ------------------------------------------------------------------------------------------------------
// tracking
// ------------------------------------------------------------------------------------------------------
extern "C" int lsdgpu_ref_import(lsdgpu_ctx* ctx, int kf_id)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, kf_id);
    if (!kf) return lsd_fail(ctx, "unknown keyframe id");
    int r = ensureIdepthPyramid(ctx, kf);
    if (r) return r;
    kf->depthHasBeenUpdatedFlag = false;       // SlamSystem.cpp:907-912
    return 0;
}

// Frame::refPixelWasGood(): created on first use, initialised to true (DataStructures/Frame.h:421-437)
static int ensureGoodMask(lsdgpu_ctx* ctx, FrameSlot* fr)
{
    if (fr->hasGoodMask) return 0;
    LSD_CHECK(ctx, cudaMemsetAsync(fr->goodMask, 1, ((size_t)ctx->w * ctx->h) / 4, ctx->stream));
    fr->hasGoodMask = true;
    return 0;
}

static void fillEvalLevel(lsdgpu_ctx* ctx, FrameSlot* kf, FrameSlot* fr, int level, bool writeMask, EvalLevel& L)
{
    const LevelCam& c = ctx->cam[level];
    L.kfIdepth = kf->idepth[level]; L.kfVar = kf->idepthVar[level]; L.kfColor = kf->image[level];
    L.frameGrad = fr->grad[level];
    L.goodMask = writeMask ? fr->goodMask : nullptr;
    L.w = c.w; L.h = c.h;
    L.fx = c.fx; L.fy = c.fy; L.cx = c.cx; L.cy = c.cy;
    L.fxi = c.fxi; L.fyi = c.fyi; L.cxi = c.cxi; L.cyi = c.cyi;
    L.shard = 0; L.nShards = 1;
}

// one evaluation launch + readback of the EV_NCH sums into ctx->hEvOut (synchronous)
static int runEval(lsdgpu_ctx* ctx, const EvalLevel& L, const lsd::SE3<float>& refToFrame, float a, float b,
                   const lsdgpu_track_settings* s)
{
    EvalPose P;
    lsd::quatToMatrix(refToFrame.q, P.R);
    P.t[0] = refToFrame.t[0]; P.t[1] = refToFrame.t[1]; P.t[2] = refToFrame.t[2];
    P.a = a; P.b = b;
    EvalConsts C;
    C.cameraPixelNoise2 = ctx->g.cameraPixelNoise2; C.var_weight = s->var_weight; C.huber_half = s->huber_d / 2;
    const int nBlocks = divUp(L.w * L.h, EVAL_THREADS);
    if (ctx->profileTrackKernel) cudaEventRecord(ctx->kBegin, ctx->stream);
    // last-block counter of its own (word 16): evCounter[0] is the persistent tracker's monotonic barrier counter, which must
    // never be reset or counted on by anybody else (mode-1 and mode-0 / parity-hook calls interleave on one context)
    k_se3_eval<<<nBlocks, EVAL_THREADS, 0, ctx->stream>>>(L, P, C, ctx->evPartials, ctx->evCounter + 16, ctx->dEvOut);
    LAUNCH(ctx);
    if (ctx->profileTrackKernel) cudaEventRecord(ctx->kEnd, ctx->stream);
    LSD_CHECK(ctx, cudaGetLastError());
    LSD_CHECK(ctx, cudaMemcpyAsync(ctx->hEvOut, ctx->dEvOut, EV_NCH * 4, cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->profileTrackKernel) {
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->kBegin, ctx->kEnd);
        ctx->trackKernelMs += ms;
        ctx->trackKernelLaunches++;
        // B_fused(l) = 12 B/px keyframe planes + 16 B/px frame gradients (+1 B/px mask on L1) + EV_NCH*4
        ctx->trackKernelBytes += (double)L.w * L.h * (12.0 + 16.0 + (L.goodMask ? 1.0 : 0.0)) + EV_NCH * 4.0;
    }
    return 0;
}

extern "C" int lsdgpu_se3_eval(lsdgpu_ctx* ctx, int kf_id, int frame_id, int level, const float refToFrame_qt[7],
                               float affine_a, float affine_b, const lsdgpu_track_settings* s, int write_good_mask,
                               lsdgpu_eval_result* out)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, kf_id);
    FrameSlot* fr = findSlot(ctx, frame_id);
    if (!kf || !fr) return lsd_fail(ctx, "unknown frame id");
    if (level < 0 || level >= LSD_LEVELS) return lsd_fail(ctx, "bad level");
    int r = ensureIdepthPyramid(ctx, kf);
    if (r) return r;
    lsdgpu_track_settings ds;
    if (!s) { lsdgpu_default_track_settings(&ds); s = &ds; }
    EvalLevel L;
    const bool wm = write_good_mask && level == SE3TRACKING_MIN_LEVEL;
    if (wm) { r = ensureGoodMask(ctx, fr); if (r) return r; }
    fillEvalLevel(ctx, kf, fr, level, wm, L);
    lsd::SE3<float> T;
    for (int i = 0; i < 4; i++) T.q[i] = refToFrame_qt[i];
    for (int i = 0; i < 3; i++) T.t[i] = refToFrame_qt[4 + i];
    r = runEval(ctx, L, T, affine_a, affine_b, s);
    if (r) return r;
    evalFinish(ctx->hEvOut, out);
    return 0;
}

// SE3Tracker::trackFrame with the LM loop on the host (mode 0): a line-by-line mirror of SE3Tracker.cpp:280-486
static int trackHostLM(lsdgpu_ctx* ctx, FrameSlot* kf, FrameSlot* fr, const double init_qt[7],
                       const lsdgpu_track_settings* st, lsdgpu_track_result* out,
                       int shard = 0, int nShards = 1, lsdgpu_allreduce_fn allreduce = nullptr, void* user = nullptr)
{
    memset(out, 0, sizeof(*out));
    bool diverged = false;
    float affine_a = 1, affine_b = 0;
    lsd::SE3<double> init;
    for (int i = 0; i < 4; i++) init.q[i] = init_qt[i];
    for (int i = 0; i < 3; i++) init.t[i] = init_qt[4 + i];
    lsd::SE3<float> referenceToFrame = lsd::se3Cast<float>(lsd::se3Inverse(init));      // :306
    lsdgpu_eval_result ev, lsq;
    memset(&ev, 0, sizeof(ev));
    float last_residual = 0;
    const int W = ctx->w, H = ctx->h;
    { int r0 = ensureGoodMask(ctx, fr); if (r0) return r0; }

    for (int lvl = SE3TRACKING_MAX_LEVEL - 1; lvl >= SE3TRACKING_MIN_LEVEL && !diverged; lvl--) {
        EvalLevel L;
        fillEvalLevel(ctx, kf, fr, lvl, lvl == SE3TRACKING_MIN_LEVEL, L);
        L.shard = shard; L.nShards = nShards;
        int r = runEval(ctx, L, referenceToFrame, affine_a, affine_b, st);
        if (r) return r;
        if (allreduce) allreduce(user, ctx->hEvOut, EV_NCH);
        evalFinish(ctx->hEvOut, &ev);
        if (ev.warpedSize < 0.01f * (W >> lvl) * (H >> lvl)) { diverged = true; break; }   // :324-329
        if (ctx->g.useAffineLightningEstimation) { affine_a = ev.affine_a_lastIt; affine_b = ev.affine_b_lastIt; }
        // NB: the weights of calcWeightsAndResidual (:336) do not depend on the affine parameters just
        // updated (the residual buffer was filled before), so one fused pass yields lastErr and ls
        float lastErr = ev.meanWeightedRes;
        lsq = ev;
        out->numCalcResidualCalls[lvl]++;
        float LM_lambda = st->lambdaInitial[lvl];

        for (int iteration = 0; iteration < st->maxItsPerLvl[lvl] && !diverged; iteration++) {
            out->numCalcWarpUpdateCalls[lvl]++;         // calculateWarpUpdate(ls): lsq already holds it
            int incTry = 0;
            while (true) {
                float b[6], A[36], inc[6];
                for (int i = 0; i < 6; i++) b[i] = -lsq.b[i];
                memcpy(A, lsq.A, sizeof(A));
                for (int i = 0; i < 6; i++) A[i * 6 + i] *= 1 + LM_lambda;
                lsd::ldlt6Solve(A, b, inc);
                incTry++;
                lsd::SE3<float> new_referenceToFrame = lsd::se3Mul(lsd::se3Exp(inc), referenceToFrame);   // :363
                r = runEval(ctx, L, new_referenceToFrame, affine_a, affine_b, st);
                if (r) return r;
                if (allreduce) allreduce(user, ctx->hEvOut, EV_NCH);
                evalFinish(ctx->hEvOut, &ev);
                if (ev.warpedSize < 0.01f * (W >> lvl) * (H >> lvl)) { diverged = true; break; }
                float error = ev.meanWeightedRes;
                out->numCalcResidualCalls[lvl]++;
                if (error < lastErr) {
                    referenceToFrame = new_referenceToFrame;
                    if (ctx->g.useAffineLightningEstimation) { affine_a = ev.affine_a_lastIt; affine_b = ev.affine_b_lastIt; }
                    if (error / lastErr > st->convergenceEps[lvl]) iteration = st->maxItsPerLvl[lvl];
                    last_residual = lastErr = error;
                    lsq = ev;                         // buffers now belong to the accepted pose
                    if (LM_lambda <= 0.2) LM_lambda = 0;
                    else LM_lambda *= st->lambdaSuccessFac;
                    break;
                } else {
                    float dot = 0;
                    for (int i = 0; i < 6; i++) dot += inc[i] * inc[i];
                    if (!(dot > st->stepSizeMin[lvl])) { iteration = st->maxItsPerLvl[lvl]; break; }
                    if (LM_lambda == 0) LM_lambda = 0.2;
                    else LM_lambda *= pow((double)st->lambdaFailFac, incTry);
                }
            }
        }
    }
    out->pointUsage = ev.pointUsage; out->lastGoodCount = ev.goodCount; out->lastBadCount = ev.badCount;
    out->lastMeanRes = ev.meanRes;
    out->affineEstimation_a = affine_a; out->affineEstimation_b = affine_b;
    if (diverged) {
        out->frameToRef_qt[3] = 1;
        out->diverged = 1; out->trackingWasGood = 0;
        return 0;
    }
    out->lastResidual = last_residual;
    out->trackingWasGood = ev.goodCount / ((W >> SE3TRACKING_MIN_LEVEL) * (H >> SE3TRACKING_MIN_LEVEL)) > 0.04f
                           && ev.goodCount / (ev.goodCount + ev.badCount) > 0.5f;                         // :475-477
    out->initialTrackedResidual = out->lastResidual / out->pointUsage;                                    // :482
    lsd::SE3<double> f2r = lsd::se3Cast<double>(lsd::se3Inverse(referenceToFrame));                        // :483-485
    for (int i = 0; i < 4; i++) out->frameToRef_qt[i] = f2r.q[i];
    for (int i = 0; i < 3; i++) out->frameToRef_qt[4 + i] = f2r.t[i];
    return 0;
}

extern "C" int lsdgpu_se3_track(lsdgpu_ctx* ctx, int kf_id, int frame_id, const double init_qt[7],
                                const lsdgpu_track_settings* s, int mode, lsdgpu_track_result* out)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, kf_id);
    FrameSlot* fr = findSlot(ctx, frame_id);
    if (!kf || !fr) return lsd_fail(ctx, "unknown frame id");
    int r = ensureIdepthPyramid(ctx, kf);      // reference->makePointCloud(lvl), SE3Tracker.cpp:321
    if (r) return r;
    lsdgpu_track_settings ds;
    if (!s) { lsdgpu_default_track_settings(&ds); ds.maxItsPerLvl[4] = 0; s = &ds; }
    if (mode == 1) r = trackPersistent(ctx, kf, fr, init_qt, s, out);
    else r = trackHostLM(ctx, kf, fr, init_qt, s, out);
    if (r) return r;
    if (!out->diverged) {
        if (out->trackingWasGood) kf->numFramesTrackedOnThis++;                   // :479-480
        fr->initialTrackedResidual = out->initialTrackedResidual;                 // :482
        for (int i = 0; i < 7; i++) fr->thisToParent[i] = out->frameToRef_qt[i];  // :483 sim3FromSE3(.., 1)
        fr->thisToParent[7] = 1.0;
        fr->parentId = kf->id;                                                    // :484
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------------
// one stream over several GPUs: peer mapping of the contexts' arenas (BASELINE config 5)
// ------------------------------------------------------------------------------------------------------
static_assert(sizeof(cudaIpcMemHandle_t) == LSDGPU_PEER_HANDLE_BYTES, "ABI constant out of sync with cudaIpcMemHandle_t");

extern "C" int lsdgpu_peer_export(lsdgpu_ctx* ctx, void* handle_out)
{ LSD_LOCK(ctx);
    if (!ctx || !handle_out) return lsd_fail(ctx, "peer_export: null argument");
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    LSD_CHECK(ctx, cudaIpcGetMemHandle(&h, ctx->arena));
    memcpy(handle_out, &h, sizeof(h));
    return 0;
}

static void peerCloseAll(lsdgpu_ctx* ctx)
{
    for (int d = 0; d < 8; d++) {
        if (ctx->peerBase[d] && d != ctx->rank) cudaIpcCloseMemHandle(ctx->peerBase[d]);
        ctx->peerBase[d] = nullptr;
    }
    ctx->nRanks = 1; ctx->rank = 0;
}

extern "C" int lsdgpu_peer_attach(lsdgpu_ctx* ctx, int rank, int n_ranks, const void* handles)
{ LSD_LOCK(ctx);
    if (!ctx) return -2;
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    if (n_ranks < 1 || n_ranks > TP_MAX_RANKS || rank < 0 || rank >= n_ranks) return lsd_fail(ctx, "peer_attach: bad rank / number of ranks");
    if (n_ranks > 1 && !handles) return lsd_fail(ctx, "peer_attach: null handle array");
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    peerCloseAll(ctx);
    if (n_ranks == 1) return 0;
    for (int d = 0; d < n_ranks; d++) {
        if (d == rank) { ctx->peerBase[d] = ctx->arena; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char*)handles + (size_t)d * sizeof(h), sizeof(h));
        void* base = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            ctx->rank = rank;
            peerCloseAll(ctx);
            cudaGetLastError();
            const std::string msg = std::string("peer_attach: cudaIpcOpenMemHandle failed for rank ") + std::to_string(d) + ": " + cudaGetErrorString(e);
            return lsd_fail(ctx, msg.c_str());
        }
        ctx->peerBase[d] = (char*)base;
    }
    ctx->rank = rank; ctx->nRanks = n_ranks;
    // the exchange rows, done slots and the tail counter start from a known state on every rank (the caller synchronises the ranks
    // between attach and the first tracking)
    LSD_CHECK(ctx, cudaMemsetAsync(ctx->trkSync + TP_XCHG_OFFSET, 0, (TP_SYNC_WORDS - 4 - TP_XCHG_OFFSET) * sizeof(unsigned int), ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->trkTailBase = 0;
    return 0;
}

extern "C" int lsdgpu_peer_detach(lsdgpu_ctx* ctx)
{ LSD_LOCK(ctx);
    if (!ctx) return -2;
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    peerCloseAll(ctx);
    return 0;
}

static_assert(LSDGPU_EVAL_NSUMS == EV_NCH, "ABI constant out of sync with the kernel's channel count");

extern "C" int lsdgpu_se3_track_sharded(lsdgpu_ctx* ctx, int kf_id, int frame_id, const double init_qt[7],
                                        const lsdgpu_track_settings* s, int shard, int n_shards,
                                        lsdgpu_allreduce_fn allreduce, void* user, lsdgpu_track_result* out)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, kf_id);
    FrameSlot* fr = findSlot(ctx, frame_id);
    if (!kf || !fr) return lsd_fail(ctx, "unknown frame id");
    if (n_shards < 1 || shard < 0 || shard >= n_shards) return lsd_fail(ctx, "bad shard");
    if (n_shards > 1 && !allreduce) return lsd_fail(ctx, "sharded tracking needs an all-reduce callback");
    int r = ensureIdepthPyramid(ctx, kf);
    if (r) return r;
    lsdgpu_track_settings ds;
    if (!s) { lsdgpu_default_track_settings(&ds); ds.maxItsPerLvl[4] = 0; s = &ds; }
    r = trackHostLM(ctx, kf, fr, init_qt, s, out, shard, n_shards, allreduce, user);
    if (r) return r;
    if (!out->diverged) {
        if (out->trackingWasGood) kf->numFramesTrackedOnThis++;
        fr->initialTrackedResidual = out->initialTrackedResidual;
        for (int i = 0; i < 7; i++) fr->thisToParent[i] = out->frameToRef_qt[i];
        fr->thisToParent[7] = 1.0;
        fr->parentId = kf->id;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------------
// depth map
// ------------------------------------------------------------------------------------------------------
static DepthCam depthCam(const lsdgpu_ctx* ctx)
{
    const LevelCam& c = ctx->cam[0];
    DepthCam d;
    d.w = c.w; d.h = c.h; d.fx = c.fx; d.fy = c.fy; d.cx = c.cx; d.cy = c.cy;
    d.fxi = c.fxi; d.fyi = c.fyi; d.cxi = c.cxi; d.cyi = c.cyi;
    return d;
}
static DepthGlobals depthGlobals(const lsdgpu_ctx* ctx)
{
    DepthGlobals g;
    g.minUseGrad = ctx->g.minUseGrad; g.cameraPixelNoise2 = ctx->g.cameraPixelNoise2;
    g.regDistVar = 0.075f * 0.075f * ctx->g.depthSmoothingFactor * ctx->g.depthSmoothingFactor;   // REG_DIST_VAR, settings.h:139
    g.allowNegativeIdepths = ctx->g.allowNegativeIdepths; g.useSubpixelStereo = ctx->g.useSubpixelStereo;
    return g;
}

extern "C" int lsdgpu_depth_reset(lsdgpu_ctx* ctx)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)ctx->w * ctx->h;
    // isValid = false everywhere (the int4 plane: isValid, blacklisted, validity, nextId)
    LSD_CHECK(ctx, cudaMemsetAsync(ctx->cur.hi, 0, n * 16, ctx->stream));
    LSD_CHECK(ctx, cudaMemsetAsync(ctx->oth.hi, 0, n * 16, ctx->stream));
    return 0;
}
extern "C" int lsdgpu_depth_is_valid(lsdgpu_ctx* ctx) { LSD_LOCK(ctx); return ctx->activeKf >= 0 ? 1 : 0; }
extern "C" int lsdgpu_depth_invalidate(lsdgpu_ctx* ctx) { LSD_LOCK(ctx); ctx->activeKf = -1; return 0; }
extern "C" int lsdgpu_depth_active_keyframe(lsdgpu_ctx* ctx) { LSD_LOCK(ctx); return ctx->activeKf; }

// Frame::setDepth(currentDepthMap) of the active keyframe
static int setDepthOnKeyframe(lsdgpu_ctx* ctx, FrameSlot* kf, const int* skip = nullptr)
{
    const int n = ctx->w * ctx->h;
    const int nb = divUp(n, 256);
    PyrPtrs id, var;
    for (int l = 0; l < LSD_LEVELS; l++) { id.l[l] = kf->idepth[l]; var.l[l] = kf->idepthVar[l]; }
    k_set_depth_pyr<<<(ctx->w / 16) * (ctx->h / 16), 256, 0, ctx->stream>>>(ctx->cur, id, var, ctx->w, ctx->h, ctx->dScalars + 8,
                                                                           ctx->evCounter + 48, kf->dStats, skip);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    kf->statsPending = true;
    kf->hasDepth = true; kf->idepthPyrValid = true;          // levels 1..4 were built by the same kernel
    kf->depthHasBeenUpdatedFlag = true;
    return 0;
}

extern "C" int lsdgpu_depth_init_from_gt(lsdgpu_ctx* ctx, int kf_id)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, kf_id);
    if (!kf) return lsd_fail(ctx, "unknown keyframe id");
    if (!kf->hasDepth) return lsd_fail(ctx, "initializeFromGTDepth: frame has no idepth (call lsdgpu_frame_set_depth_gt)");
    const int n = ctx->w * ctx->h;
    ctx->activeKf = kf_id; ctx->activeKfReactivated = false;
    k_init_from_gt<<<divUp(n, 256), 256, 0, ctx->stream>>>(ctx->cur, kf->idepth[0], n);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    return setDepthOnKeyframe(ctx, kf);
}

static int runRegularize(lsdgpu_ctx* ctx, bool removeOcclusions, int validityTH, const int* skip = nullptr)
{
    DepthCam cam = depthCam(ctx);
    DepthGlobals G = depthGlobals(ctx);
    dim3 grid(divUp(cam.w, 32), divUp(cam.h, 8));
    std::swap(ctx->cur, ctx->oth);         // oth = previous current (the memcpy of :862), cur = output
    if (removeOcclusions) k_regularize<true><<<grid, 256, 0, ctx->stream>>>(ctx->oth, ctx->cur, cam, G, validityTH, skip);
    else k_regularize<false><<<grid, 256, 0, ctx->stream>>>(ctx->oth, ctx->cur, cam, G, validityTH, skip);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    return 0;
}
// regularizeDepthMapFillHoles() + regularizeDepthMap(false, TH) as one kernel (see k_fill_regularize); with
// setDepthOn != nullptr the kernel also does Frame::setDepth + the idepth pyramid of that keyframe
static int runFillRegularize(lsdgpu_ctx* ctx, int validityTH, const int* skip = nullptr, FrameSlot* setDepthOn = nullptr)
{
    FrameSlot* kf = findSlot(ctx, ctx->activeKf);
    if (!kf) return lsd_fail(ctx, "no active keyframe");
    DepthCam cam = depthCam(ctx);
    DepthGlobals G = depthGlobals(ctx);
    const int grid = divUp(cam.w, FR_TW) * divUp(cam.h, FR_TH);
    std::swap(ctx->cur, ctx->oth);
    PyrPtrs id, var;
    for (int l = 0; l < LSD_LEVELS; l++) { id.l[l] = setDepthOn ? setDepthOn->idepth[l] : nullptr; var.l[l] = setDepthOn ? setDepthOn->idepthVar[l] : nullptr; }
    if (setDepthOn) {
        LSD_CHECK(ctx, launchPDL(k_fill_regularize<true>, dim3(grid), dim3(FR_THREADS), 0, ctx->stream, ctx->optPdl, ctx->oth, ctx->cur, cam, G,
                                 (const float*)kf->maxgrad, validityTH, skip, id, var, ctx->dScalars + 8, ctx->evCounter + 48, setDepthOn->dStats));
        setDepthOn->statsPending = true;
        setDepthOn->hasDepth = true; setDepthOn->idepthPyrValid = true;
        setDepthOn->depthHasBeenUpdatedFlag = true;                    // Frame.cpp:242
    } else
        LSD_CHECK(ctx, launchPDL(k_fill_regularize<false>, dim3(grid), dim3(FR_THREADS), 0, ctx->stream, ctx->optPdl, ctx->oth, ctx->cur, cam, G,
                                 (const float*)kf->maxgrad, validityTH, skip, id, var, (double*)nullptr, (unsigned int*)nullptr, (double*)nullptr));
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    return 0;
}

static int runFillHoles(lsdgpu_ctx* ctx, const int* skip = nullptr)
{
    FrameSlot* kf = findSlot(ctx, ctx->activeKf);
    if (!kf) return lsd_fail(ctx, "no active keyframe");
    DepthCam cam = depthCam(ctx);
    DepthGlobals G = depthGlobals(ctx);
    dim3 grid(divUp(cam.w, 32), divUp(cam.h, 8));
    std::swap(ctx->cur, ctx->oth);
    k_fill_holes<<<grid, 256, 0, ctx->stream>>>(ctx->oth, ctx->cur, cam, G, kf->maxgrad, skip);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    return 0;
}

extern "C" int lsdgpu_depth_set_hypotheses(lsdgpu_ctx* ctx, int kf_id, const lsdgpu_hyp* aos, int reactivated, int do_set_depth)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, kf_id);
    if (!kf) return lsd_fail(ctx, "unknown keyframe id");
    const int n = ctx->w * ctx->h;
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(ctx->hStageF, aos, (size_t)n * 32);
    LSD_CHECK(ctx, cudaMemcpyAsync(ctx->dStageF, ctx->hStageF, (size_t)n * 32, cudaMemcpyHostToDevice, ctx->stream));
    k_hyp_from_aos<<<divUp(n, 256), 256, 0, ctx->stream>>>((const lsdgpu_hyp*)ctx->dStageF, ctx->cur, n);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    ctx->activeKf = kf_id; ctx->activeKfReactivated = reactivated != 0;
    if (reactivated) {
        kf->numMappedOnThis = 0; kf->numFramesTrackedOnThis = 0;                   // :932-933
        int r = runRegularize(ctx, false, VAL_SUM_MIN_FOR_KEEP);                   // :961
        if (r) return r;
    }
    if (do_set_depth) return setDepthOnKeyframe(ctx, kf);
    return 0;
}

extern "C" int lsdgpu_depth_download(lsdgpu_ctx* ctx, lsdgpu_hyp* aos_out)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    const int n = ctx->w * ctx->h;
    k_hyp_to_aos<<<divUp(n, 256), 256, 0, ctx->stream>>>(ctx->cur, (lsdgpu_hyp*)ctx->dStageF, n);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    LSD_CHECK(ctx, cudaMemcpyAsync(aos_out, ctx->dStageF, (size_t)n * 32, cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int lsdgpu_depth_download_integral(lsdgpu_ctx* ctx, int32_t* out)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    k_integral_rows<<<divUp(ctx->h, 64), 64, 0, ctx->stream>>>(ctx->cur, ctx->integral, ctx->w, ctx->h);
    LAUNCH(ctx);
    k_integral_cols<<<divUp(ctx->w, 64), 64, 0, ctx->stream>>>(ctx->integral, ctx->w, ctx->h);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    LSD_CHECK(ctx, cudaMemcpyAsync(out, ctx->integral, (size_t)ctx->w * ctx->h * 4, cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

static void prepareForStereoWith(const lsdgpu_ctx* ctx, const FrameSlot* fr, RefConst& rc)
{
    prepareStereoConsts(ctx->cam[0].K, fr->thisToParent, fr->thisToParent + 4, fr->thisToParent[7], rc);
}

static int setupObserve(lsdgpu_ctx* ctx, const lsdgpu_ref_desc* refs, int n_refs, FrameSlot* kf)
{   // DepthMap.cpp:1079-1105
    if (n_refs <= 0 || n_refs > LSD_MAX_REFS) return lsd_fail(ctx, "bad number of reference frames");
    ObserveParams& OP = ctx->hObs;
    OP.nRefs = n_refs;
    OP.byIdSize = 0;
    for (int k = 0; k < n_refs; k++) {
        FrameSlot* fr = findSlot(ctx, refs[k].frame_id);
        if (!fr) return lsd_fail(ctx, "unknown reference frame id");
        RefConst& rc = OP.refs[k];
        if (refs[k].tracked_on_kf) {
            // :1096-1097 refToKf = frame->pose->thisToParent_raw
            if (fr->parentId != kf->id) return lsd_fail(ctx, "reference frame declared tracked_on_kf but its tracking parent is not the active keyframe");
            prepareForStereoWith(ctx, fr, rc);
        } else {
            // :1098-1099 refToKf = activeKeyFrame->getScaledCamToWorld().inverse() * frame->getScaledCamToWorld(): the absolute
            // poses live in the caller's pose graph (FramePoseStruct / KeyFrameGraph), so the caller hands the product over
            const double* q = refs[k].refToKf_qts;
            const double n2 = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
            if (!(n2 > 0.25 && n2 < 4.0) || !(q[7] > 0)) return lsd_fail(ctx, "reference frame not tracked on the active keyframe: refToKf_qts must hold a unit quaternion and a positive scale");
            prepareStereoConsts(ctx->cam[0].K, q, q + 4, q[7], rc);
        }
        rc.initialTrackedResidual = fr->initialTrackedResidual;
        rc.id = fr->id;
        rc.trackedOnActive = refs[k].tracked_on_kf ? 1 : 0;       // gate of the tracking mask, DepthMap.cpp:245 / :322
        rc.image = fr->image[0];
        rc.goodMask = fr->hasGoodMask ? fr->goodMask : nullptr;
        if (k == 0) OP.byIdOffset = fr->id;
        while (OP.byIdSize + OP.byIdOffset <= fr->id) {
            if (OP.byIdSize >= LSD_MAX_ID_SPAN) return lsd_fail(ctx, "reference id span too large");
            OP.byId[OP.byIdSize++] = k;
        }
    }
    OP.oldestIdx = 0; OP.newestIdx = n_refs - 1;
    OP.reactivated = ctx->activeKfReactivated ? 1 : 0;
    OP.kfNumTracked = kf->numFramesTrackedOnThis; OP.kfNumMapped = kf->numMappedOnThis;
    return 0;
}

// ids only: every frame was tracked on the active keyframe (the common case, SlamSystem.cpp:559-575)
static int setupObserve(lsdgpu_ctx* ctx, const int* ref_ids, int n_refs, FrameSlot* kf)
{
    if (n_refs <= 0 || n_refs > LSD_MAX_REFS) return lsd_fail(ctx, "bad number of reference frames");
    lsdgpu_ref_desc d[LSD_MAX_REFS];
    memset(d, 0, sizeof(d));
    for (int k = 0; k < n_refs; k++) {
        d[k].frame_id = ref_ids[k]; d[k].tracked_on_kf = 1;
        const FrameSlot* fr = findSlot(ctx, ref_ids[k]);
        if (fr && fr->parentId != kf->id)
            return lsd_fail(ctx, "reference frame was not tracked on the active keyframe: pass its refToKf through lsdgpu_depth_update_keyframe_refs");
    }
    return setupObserve(ctx, d, n_refs, kf);
}

static int runObserve(lsdgpu_ctx* ctx, const int* ref_ids, int n_refs, bool devParams = false, const int* skip = nullptr, bool hostParamsReady = false)
{
    FrameSlot* kf = findSlot(ctx, ctx->activeKf);
    if (!kf) return lsd_fail(ctx, "no active keyframe");
    if (!devParams && !hostParamsReady) {
        int r = setupObserve(ctx, ref_ids, n_refs, kf);
        if (r) return r;
    }
    DepthCam cam = depthCam(ctx);
    DepthGlobals G = depthGlobals(ctx);
    const int grid = divUp((cam.w - 6) * (cam.h - 6), OBS_PIX_PER_CTA);
    LSD_CHECK(ctx, launchPDL(k_observe, dim3(grid), dim3(OBS_THREADS), 0, ctx->stream, ctx->optPdl, ctx->cur, cam, G, (const float*)kf->image[0],
                             (const float4*)kf->grad[0], (const float*)kf->maxgrad, ctx->hObs, (const ObserveParams*)(devParams ? ctx->dObs : nullptr), skip));
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    return 0;
}

extern "C" int lsdgpu_depth_observe(lsdgpu_ctx* ctx, const int* ref_ids, int n_refs)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    return runObserve(ctx, ref_ids, n_refs);
}
extern "C" int lsdgpu_depth_regularize_fill_holes(lsdgpu_ctx* ctx)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    return runFillHoles(ctx);
}
extern "C" int lsdgpu_depth_regularize(lsdgpu_ctx* ctx, int removeOcclusions, int validityTH)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    return runRegularize(ctx, removeOcclusions != 0, validityTH);
}

extern "C" int lsdgpu_depth_update_keyframe(lsdgpu_ctx* ctx, const int* ref_ids, int n_refs)
{ LSD_LOCK(ctx);   // DepthMap::updateKeyframe :1072-1213
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, ctx->activeKf);
    if (!kf) return lsd_fail(ctx, "updateKeyframe: depth map is not valid (no active keyframe)");
    int r = runObserve(ctx, ref_ids, n_refs);                      // :1127
    if (r) return r;
    r = runFillRegularize(ctx, VAL_SUM_MIN_FOR_KEEP, nullptr,      // :1135 + :1143 (+ setDepth :1150-1157 in the same kernel)
                          kf->depthHasBeenUpdatedFlag ? nullptr : kf);
    if (r) return r;
    kf->numMappedOnThis++;                                         // :1165
    return 0;
}

extern "C" int lsdgpu_depth_update_keyframe_refs(lsdgpu_ctx* ctx, const lsdgpu_ref_desc* refs, int n_refs)
{ LSD_LOCK(ctx);   // DepthMap::updateKeyframe :1072-1213 with the reference-frame set-up of :1085-1101 spelled out by the caller
    if (!ctx || !refs) return lsd_fail(ctx, "update_keyframe_refs: null argument");
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, ctx->activeKf);
    if (!kf) return lsd_fail(ctx, "updateKeyframe: depth map is not valid (no active keyframe)");
    int r = setupObserve(ctx, refs, n_refs, kf);
    if (r) return r;
    r = runObserve(ctx, nullptr, n_refs, false, nullptr, true);    // :1127 (parameters already in ctx->hObs)
    if (r) return r;
    r = runFillRegularize(ctx, VAL_SUM_MIN_FOR_KEEP, nullptr, kf->depthHasBeenUpdatedFlag ? nullptr : kf);
    if (r) return r;
    kf->numMappedOnThis++;                                         // :1165
    return 0;
}

static int runPropagate(lsdgpu_ctx* ctx, FrameSlot* kf, FrameSlot* nk)
{   // DepthMap::propagateDepth :475-653
    const int n = ctx->w * ctx->h;
    lsd::SE3<double> tp;
    for (int i = 0; i < 4; i++) tp.q[i] = nk->thisToParent[i];
    for (int i = 0; i < 3; i++) tp.t[i] = nk->thisToParent[4 + i];
    lsd::quatNormalize(tp.q);                                      // se3FromSim3: SE3(quaternion, translation)
    lsd::SE3<double> oldToNew = lsd::se3Inverse(tp);               // :503
    double Rd[9];
    lsd::quatToMatrix(oldToNew.q, Rd);
    PropParams P;
    for (int i = 0; i < 9; i++) P.R[i] = (float)Rd[i];
    for (int i = 0; i < 3; i++) P.t[i] = (float)oldToNew.t[i];
    P.trackingWasGood = (nk->parentId == kf->id && nk->hasGoodMask) ? nk->goodMask : nullptr;      // :508
    P.activeKFImage = kf->image[0];
    P.newKFMaxGrad = nk->maxgrad;
    P.newKFImage = nk->image[0];
    LSD_CHECK(ctx, cudaMemsetAsync(ctx->propHead, 0xff, (size_t)n * 4, ctx->stream));
    DepthCam cam = depthCam(ctx);
    DepthGlobals G = depthGlobals(ctx);
    k_prop_project<<<divUp(n, 256), 256, 0, ctx->stream>>>(ctx->cur, cam, G, P, ctx->propHead, ctx->propNext, ctx->propVal);
    LAUNCH(ctx);
    k_prop_resolve<<<divUp(n, 256), 256, 0, ctx->stream>>>(ctx->oth, n, ctx->propHead, ctx->propNext, ctx->propVal);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    std::swap(ctx->cur, ctx->oth);                                 // :637
    return 0;
}

extern "C" int lsdgpu_depth_propagate(lsdgpu_ctx* ctx, int new_kf_id)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, ctx->activeKf);
    FrameSlot* nk = findSlot(ctx, new_kf_id);
    if (!kf || !nk) return lsd_fail(ctx, "propagateDepth: unknown keyframe");
    return runPropagate(ctx, kf, nk);
}

extern "C" int lsdgpu_depth_create_keyframe(lsdgpu_ctx* ctx, int new_kf_id, double new_qts[8])
{ LSD_LOCK(ctx);   // DepthMap::createKeyFrame :1222-1327
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, ctx->activeKf);
    FrameSlot* nk = findSlot(ctx, new_kf_id);
    if (!kf) return lsd_fail(ctx, "createKeyFrame: depth map is not valid");
    if (!nk) return lsd_fail(ctx, "createKeyFrame: unknown new keyframe");
    if (nk->parentId < 0) return lsd_fail(ctx, "createKeyFrame: new keyframe has no tracking parent");
    lsd::SE3<double> tp;
    for (int i = 0; i < 4; i++) tp.q[i] = nk->thisToParent[i];
    for (int i = 0; i < 3; i++) tp.t[i] = nk->thisToParent[4 + i];
    lsd::quatNormalize(tp.q);
    lsd::SE3<double> oldToNew = lsd::se3Inverse(tp);               // :1246
    int r = runPropagate(ctx, kf, nk);                             // :1250
    if (r) return r;
    ctx->activeKf = new_kf_id; ctx->activeKfReactivated = false;   // :1255-1258
    r = runRegularize(ctx, true, VAL_SUM_MIN_FOR_KEEP);            // :1263
    if (r) return r;
    r = runFillRegularize(ctx, VAL_SUM_MIN_FOR_KEEP);              // :1270 + :1277
    if (r) return r;
    const int n = ctx->w * ctx->h;
    const int nb = divUp(n, 256);
    // :1286-1294: the reference's sequential `float +=` over the valid hypotheses, reproduced bit for bit (seqsum.cuh)
    const int seqRuns = divUp(n, SEQ_RUN);
    k_seqsum_table<<<divUp(seqRuns, 8), 256, 0, ctx->stream>>>(ctx->cur.hf, ctx->cur.hi, n, seqRuns, ctx->seqTable, ctx->seqFlags, ctx->seqCounts);
    LAUNCH(ctx);
    k_seqsum_walk<<<1, 32, 0, ctx->stream>>>(ctx->cur.hf, ctx->cur.hi, n, seqRuns, ctx->seqTable, ctx->seqFlags, ctx->seqCounts, ctx->dScalars);
    LAUNCH(ctx);
    k_rescale<<<nb, 256, 0, ctx->stream>>>(ctx->cur, n, ctx->dScalars);                          // :1295-1304
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    LSD_CHECK(ctx, cudaMemcpyAsync(ctx->hScalars + 4, ctx->dScalars, 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    const float rescaleFactor = (float)ctx->hScalars[4 + 2];
    lsd::SE3<double> back = lsd::se3Inverse(oldToNew);             // :1305 sim3FromSE3(oldToNew_SE3.inverse(), rescaleFactor)
    for (int i = 0; i < 4; i++) nk->thisToParent[i] = back.q[i];
    for (int i = 0; i < 3; i++) nk->thisToParent[4 + i] = back.t[i];
    nk->thisToParent[7] = rescaleFactor;
    if (new_qts) memcpy(new_qts, nk->thisToParent, sizeof(nk->thisToParent));
    return setDepthOnKeyframe(ctx, nk);                            // :1311
}

__global__ void k_seqsum_pack(const float* __restrict__ x, const unsigned char* __restrict__ valid, int n, float4* hf, int4* hi)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    hf[i] = make_float4(0.f, 0.f, x[i], 0.f);
    hi[i] = make_int4(valid ? (valid[i] != 0) : 1, 0, 0, 0);
}

// The sequential `float sum = 0; for (i) if (valid[i]) sum += x[i];` of DepthMap.cpp:1286-1293 on arbitrary host data, through
// the kernels createKeyFrame uses (seqsum.cuh) -- exposed so the bit-exactness of that reproduction can be tested on adversarial
// inputs (ties, binade crossings, negative / non-finite terms), which real depth maps rarely contain.
extern "C" int lsdgpu_seq_sum_f32(lsdgpu_ctx* ctx, const float* x, const unsigned char* valid, int n, float* sum, int* count)
{ LSD_LOCK(ctx);
    if (!ctx || !x || n < 0 || !sum) return lsd_fail(ctx, "seq_sum_f32: bad arguments");
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    if (n == 0) { *sum = 0.f; if (count) *count = 0; return 0; }
    const int runs = divUp(n, SEQ_RUN);
    char* buf = nullptr;
    const size_t bx = alignUp((size_t)n * 4, 256), bv = alignUp((size_t)n, 256), bf = alignUp((size_t)n * 16, 256),
                 bt = alignUp((size_t)runs * SEQ_NBIN * sizeof(int2), 256), bg = alignUp((size_t)runs, 256), bc = alignUp((size_t)runs * 4, 256);
    LSD_CHECK(ctx, cudaMalloc((void**)&buf, bx + bv + 2 * bf + bt + bg + bc + 256));
    char* p = buf;
    float* dx = (float*)p; p += bx;
    unsigned char* dv = (unsigned char*)p; p += bv;
    float4* hf = (float4*)p; p += bf;
    int4* hi = (int4*)p; p += bf;
    int2* table = (int2*)p; p += bt;
    unsigned char* flags = (unsigned char*)p; p += bg;
    int* counts = (int*)p; p += bc;
    double* out = (double*)p;
    int rc = 0;
    do {
        if (cudaMemcpyAsync(dx, x, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) { rc = 1; break; }
        if (valid && cudaMemcpyAsync(dv, valid, (size_t)n, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) { rc = 1; break; }
        k_seqsum_pack<<<divUp(n, 256), 256, 0, ctx->stream>>>(dx, valid ? dv : nullptr, n, hf, hi);
        k_seqsum_table<<<divUp(runs, 8), 256, 0, ctx->stream>>>(hf, hi, n, runs, table, flags, counts);
        k_seqsum_walk<<<1, 32, 0, ctx->stream>>>(hf, hi, n, runs, table, flags, counts, out);
        double h[3];
        if (cudaMemcpyAsync(h, out, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) { rc = 1; break; }
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) { rc = 1; break; }
        *sum = (float)h[0];
        if (count) *count = (int)h[1];
    } while (0);
    cudaFree(buf);
    if (rc) return lsd_fail(ctx, "seq_sum_f32: CUDA error");
    return 0;
}

// Frame::takeReActivationData(currentDepthMap), Frame.cpp:107-145.  The pool buffers of a fresh Frame are defined as
// zero-filled (SURVEY appendix A.12); later takes of the same frame keep the entries of invalid pixels, as the reference does.
static int takeReactivationData(lsdgpu_ctx* ctx, FrameSlot* kf)
{
    const int n = ctx->w * ctx->h;
    if (!kf->reactAllocated) {
        LSD_CHECK(ctx, cudaMemsetAsync(kf->reactIdepth, 0, (size_t)n * 4, ctx->stream));
        LSD_CHECK(ctx, cudaMemsetAsync(kf->reactVar, 0, (size_t)n * 4, ctx->stream));
        LSD_CHECK(ctx, cudaMemsetAsync(kf->reactValidity, 0, (size_t)n, ctx->stream));
        kf->reactAllocated = true;
    }
    k_take_reactivation<<<divUp(n, 256), 256, 0, ctx->stream>>>(ctx->cur, kf->reactIdepth, kf->reactVar, kf->reactValidity, n);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    kf->reactValid = true;
    return 0;
}

extern "C" int lsdgpu_depth_finalize_keyframe(lsdgpu_ctx* ctx)
{ LSD_LOCK(ctx);   // DepthMap::finalizeKeyFrame :1363-1395
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, ctx->activeKf);
    if (!kf) return lsd_fail(ctx, "finalizeKeyFrame: depth map is not valid");
    int r = runFillRegularize(ctx, VAL_SUM_MIN_FOR_KEEP, nullptr, kf);   // :1373 + :1379 + setDepth :1385
    if (r) return r;
    return takeReactivationData(ctx, kf);                                // :1387 (calculateMeanInformation :1386 returns at once, Frame.cpp:178)
}

extern "C" int lsdgpu_track_and_map(lsdgpu_ctx* ctx, int kf_id, int frame_id, const uint8_t* gray, int stage_index,
                                    const double init_qt[7], const lsdgpu_track_settings* s, int mode,
                                    int keyframe_change, lsdgpu_track_result* out, double new_qts[8])
{ LSD_LOCK(ctx);
    int r = gray ? lsdgpu_frame_upload_u8(ctx, frame_id, gray) : lsdgpu_frame_from_stage(ctx, frame_id, stage_index);
    if (r) return r;
    FrameSlot* kf = findSlot(ctx, kf_id);
    if (!kf) return lsd_fail(ctx, "unknown keyframe id");
    if (kf->depthHasBeenUpdatedFlag) { r = lsdgpu_ref_import(ctx, kf_id); if (r) return r; }     // SlamSystem.cpp:907-912
    FrameSlot* fr = findSlot(ctx, frame_id);
    // LSDGPU_SINGLE_SYNC=1 (opt-in): the whole frame is enqueued back to back and the host synchronises once; the stereo
    // constants of prepareForStereoWith are then computed by the tracking kernel's last thread.  Measured on B200 (A/B on
    // one box, 640x480): 202.6 us per step against 202.0 us for the default (poll the tracking result, constants on the
    // host) -- the 2.2 us of one-thread double-precision work at the kernel's tail cost what the round trip saves.
    const bool singleSync = ctx->optSingleSync == 1;
    if (singleSync && mode == 1 && !keyframe_change && ctx->activeKf == kf_id && fr) {
        // Whole frame enqueued back to back: tracking kernel, device-side prepareForStereoWith, observe, fill holes,
        // regularise, setDepth -- ONE host synchronisation at the end (the mapping kernels read the pose from the
        // tracker's device-resident result and do nothing if tracking diverged).
        lsdgpu_track_settings ds;
        if (!s) { lsdgpu_default_track_settings(&ds); ds.maxItsPerLvl[4] = 0; s = &ds; }
        r = ensureIdepthPyramid(ctx, kf);
        if (r) return r;
        PrepareConsts pc;
        memcpy(pc.K, ctx->cam[0].K, 36);
        pc.frameId = frame_id; pc.reactivated = ctx->activeKfReactivated ? 1 : 0;
        pc.kfNumTracked = kf->numFramesTrackedOnThis; pc.kfNumMapped = kf->numMappedOnThis;
        pc.W1 = ctx->w >> SE3TRACKING_MIN_LEVEL; pc.H1 = ctx->h >> SE3TRACKING_MIN_LEVEL;
        pc.image = fr->image[0]; pc.goodMask = fr->goodMask;
        r = trackPersistentEnqueue(ctx, kf, fr, init_qt, s, &pc);         // the kernel's last thread also writes ctx->dObs / dSkipFlag
        if (r) return r;
        r = runObserve(ctx, &frame_id, 1, true, ctx->dSkipFlag);          // DepthMap.cpp:1127
        if (r) return r;
        const bool didSetDepth = !kf->depthHasBeenUpdatedFlag;            // :1150-1157
        const bool prevPending = kf->statsPending, prevPyr = kf->idepthPyrValid;
        r = runFillRegularize(ctx, VAL_SUM_MIN_FOR_KEEP, ctx->dSkipFlag, didSetDepth ? kf : nullptr);    // :1135 + :1143 (+ setDepth)
        if (r) return r;
        r = trackPersistentFinish(ctx, fr, out);                          // the one synchronisation of the frame
        if (r) return r;
        if (out->diverged) {                 // nothing ran on the device: undo the host-side bookkeeping
            std::swap(ctx->cur, ctx->oth);   // the (skipped) fill+regularise kernel had swapped the ping-pong buffers once
            if (didSetDepth) { kf->depthHasBeenUpdatedFlag = false; kf->statsPending = prevPending; kf->idepthPyrValid = prevPyr; }
            return 0;
        }
        if (out->trackingWasGood) kf->numFramesTrackedOnThis++;           // SE3Tracker.cpp:479-480
        fr->initialTrackedResidual = out->initialTrackedResidual;
        for (int i = 0; i < 7; i++) fr->thisToParent[i] = out->frameToRef_qt[i];
        fr->thisToParent[7] = 1.0;
        fr->parentId = kf->id;
        kf->numMappedOnThis++;                                            // DepthMap.cpp:1165
        return lsdgpu_frame_clear_good_mask(ctx, frame_id);               // SlamSystem.cpp:573
    }
    r = lsdgpu_se3_track(ctx, kf_id, frame_id, init_qt, s, mode, out);
    if (r) return r;
    if (out->diverged) return 0;                 // the caller decides (relocalisation is out of scope)
    if (keyframe_change) {
        r = lsdgpu_depth_finalize_keyframe(ctx);
        if (r) return r;
        return lsdgpu_depth_create_keyframe(ctx, frame_id, new_qts);
    }
    r = lsdgpu_depth_update_keyframe(ctx, &frame_id, 1);
    if (r) return r;
    return lsdgpu_frame_clear_good_mask(ctx, frame_id);
}

// ------------------------------------------------------------------------------------------------------
// permaRef tracking (SURVEY 8f row 2)
// ------------------------------------------------------------------------------------------------------
extern "C" int lsdgpu_frame_set_perma_ref(lsdgpu_ctx* ctx, int kf_id, int* num_points_out)
{ LSD_LOCK(ctx);   // Frame::setPermaRef -> reference->makePointCloud(QUICK_KF_CHECK_LVL) + copy (Frame.cpp:149-174, TrackingReference.cpp:96-147)
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, kf_id);
    if (!kf) return lsd_fail(ctx, "unknown keyframe id");
    int r = ensureIdepthPyramid(ctx, kf);
    if (r) return r;
    const LevelCam& c = ctx->cam[QUICK_KF_CHECK_LVL];
    const int w = c.w, h = c.h, n = w * h;
    std::vector<float> id(n), var(n), col(n);
    LSD_CHECK(ctx, cudaMemcpyAsync(id.data(), kf->idepth[QUICK_KF_CHECK_LVL], n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaMemcpyAsync(var.data(), kf->idepthVar[QUICK_KF_CHECK_LVL], n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaMemcpyAsync(col.data(), kf->image[QUICK_KF_CHECK_LVL], n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    std::vector<float4> pc;
    std::vector<float> pv;
    for (int x = 1; x < w - 1; x++)                    // x outer, y inner: the reference's point order (:128-129)
        for (int y = 1; y < h - 1; y++) {
            const int idx = x + y * w;
            if (var[idx] <= 0 || id[idx] == 0) continue;
            const float sc = 1.0f / id[idx];
            pc.push_back(make_float4(sc * (c.fxi * x + c.cxi), sc * (c.fyi * y + c.cyi), sc * 1, col[idx]));
            pv.push_back(var[idx]);
        }
    kf->permaNumPts = (int)pc.size();
    if (kf->permaNumPts) {
        LSD_CHECK(ctx, cudaMemcpyAsync(kf->permaPC, pc.data(), pc.size() * 16, cudaMemcpyHostToDevice, ctx->stream));
        LSD_CHECK(ctx, cudaMemcpyAsync(kf->permaVar, pv.data(), pv.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    }
    if (num_points_out) *num_points_out = kf->permaNumPts;
    return 0;
}

static int fillPermaItems(lsdgpu_ctx* ctx, int n, const int* kf_ids, const double* qt, std::vector<PermaItem>& items)
{
    if (n <= 0 || n > LSD_MAX_PERMA_BATCH) return lsd_fail(ctx, "bad candidate count");
    items.resize(n);
    for (int i = 0; i < n; i++) {
        FrameSlot* kf = findSlot(ctx, kf_ids[i]);
        if (!kf) return lsd_fail(ctx, "unknown keyframe id");
        if (kf->permaNumPts <= 0) return lsd_fail(ctx, "keyframe has no permaRef (call lsdgpu_frame_set_perma_ref)");
        lsd::SE3<double> T;
        for (int k = 0; k < 4; k++) T.q[k] = qt[7 * i + k];
        for (int k = 0; k < 3; k++) T.t[k] = qt[7 * i + 4 + k];
        const lsd::SE3<float> Tf = lsd::se3Cast<float>(T);                 // referenceToFrameOrg.cast<float>(), :125,168
        items[i].pc = kf->permaPC; items[i].var = kf->permaVar; items[i].n = kf->permaNumPts;
        for (int k = 0; k < 4; k++) items[i].refToFrame[k] = Tf.q[k];
        for (int k = 0; k < 3; k++) items[i].refToFrame[4 + k] = Tf.t[k];
    }
    LSD_CHECK(ctx, cudaMemcpyAsync(ctx->dPermaItems, items.data(), n * sizeof(PermaItem), cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}

extern "C" int lsdgpu_perma_overlap_batch(lsdgpu_ctx* ctx, int n, const int* kf_ids, const double* refToFrame_qt, float* usage_out)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    std::vector<PermaItem> items;
    int r = fillPermaItems(ctx, n, kf_ids, refToFrame_qt, items);
    if (r) return r;
    const LevelCam& c = ctx->cam[QUICK_KF_CHECK_LVL];
    float* dUsage = (float*)ctx->dPermaResults;
    k_perma_overlap<<<n, 128, 0, ctx->stream>>>((const PermaItem*)ctx->dPermaItems, c.fx, c.fy, c.cx, c.cy, c.w - 1, c.h - 1, dUsage);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    LSD_CHECK(ctx, cudaMemcpyAsync(usage_out, dUsage, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int lsdgpu_perma_track_batch(lsdgpu_ctx* ctx, int n, const int* kf_ids, int frame_id, const double* refToFrame_init_qt,
                                        lsdgpu_track_result* results)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* fr = findSlot(ctx, frame_id);
    if (!fr) return lsd_fail(ctx, "unknown frame id");
    std::vector<PermaItem> items;
    int r = fillPermaItems(ctx, n, kf_ids, refToFrame_init_qt, items);
    if (r) return r;
    TrackParams P;
    memset(&P, 0, sizeof(P));
    const LevelCam& c = ctx->cam[QUICK_KF_CHECK_LVL];
    TrackLevelParams& L = P.lvl[QUICK_KF_CHECK_LVL];
    L.frameGrad = fr->grad[QUICK_KF_CHECK_LVL];
    L.w = c.w; L.h = c.h; L.fx = c.fx; L.fy = c.fy; L.cx = c.cx; L.cy = c.cy;
    L.fxi = c.fxi; L.fyi = c.fyi; L.cxi = c.cxi; L.cyi = c.cyi;
    P.W = ctx->w; P.H = ctx->h;
    lsdgpu_track_settings st;
    lsdgpu_default_track_settings(&st);
    // TestTrack settings (util/settings.h:379-382) mapped onto level 4
    st.lambdaInitial[QUICK_KF_CHECK_LVL] = 0; st.stepSizeMin[QUICK_KF_CHECK_LVL] = 1e-3f;
    st.convergenceEps[QUICK_KF_CHECK_LVL] = 0.98f; st.maxItsPerLvl[QUICK_KF_CHECK_LVL] = 5;
    P.st = st;
    P.C.cameraPixelNoise2 = ctx->g.cameraPixelNoise2; P.C.var_weight = st.var_weight; P.C.huber_half = st.huber_d / 2;
    P.useAffine = ctx->g.useAffineLightningEstimation;
    P.minLevel = QUICK_KF_CHECK_LVL;
    P.kmax = 1;                                   // one pose per pass: the candidates are independent CTAs already
    PermaResult* dRes = (PermaResult*)ctx->dPermaResults;
    k_perma_track<<<n, PERMA_THREADS, 0, ctx->stream>>>(P, (const PermaItem*)ctx->dPermaItems, dRes);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    std::vector<PermaResult> hres(n);
    LSD_CHECK(ctx, cudaMemcpyAsync(hres.data(), dRes, n * sizeof(PermaResult), cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < n; i++) {
        lsdgpu_track_result& o = results[i];
        memset(&o, 0, sizeof(o));
        const PermaResult& h = hres[i];
        o.pointUsage = h.pointUsage; o.lastGoodCount = h.goodCount; o.lastBadCount = h.badCount; o.lastMeanRes = h.meanRes;
        o.affineEstimation_a = h.affine_a; o.affineEstimation_b = h.affine_b;
        o.numCalcResidualCalls[QUICK_KF_CHECK_LVL] = h.nRes; o.numCalcWarpUpdateCalls[QUICK_KF_CHECK_LVL] = h.nUpd;
        if (h.diverged) { o.frameToRef_qt[3] = 1; o.diverged = 1; continue; }             // return SE3(), :180-185
        o.lastResidual = h.lastResidual;                                                // :265
        o.trackingWasGood = h.goodCount / (c.w * c.h) > 0.04f && h.goodCount / (h.goodCount + h.badCount) > 0.5f;   // :267-269
        lsd::SE3<float> T;
        for (int k = 0; k < 4; k++) T.q[k] = h.refToFrame[k];
        for (int k = 0; k < 3; k++) T.t[k] = h.refToFrame[4 + k];
        const lsd::SE3<double> Td = lsd::se3Cast<double>(T);                            // toSophus(referenceToFrame), :271
        for (int k = 0; k < 4; k++) o.frameToRef_qt[k] = Td.q[k];
        for (int k = 0; k < 3; k++) o.frameToRef_qt[4 + k] = Td.t[k];
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------------
// Sim3 tracking, batched (SURVEY 8f row 1)
// ------------------------------------------------------------------------------------------------------
static int sim3Launch(lsdgpu_ctx* ctx, int n, const int* ref_ids, const int* frame_ids, const double* qts, bool qtsIsRefToFrame,
                      int startLevel, int finalLevel, const lsdgpu_track_settings* s, int evalOnly, float evalA, float evalB,
                      std::vector<Sim3Out>& hout)
{
    if (n <= 0 || n > S3_MAX_BATCH) return lsd_fail(ctx, "bad problem count");
    if (startLevel < 0 || startLevel >= LSD_LEVELS || finalLevel < 0 || finalLevel > startLevel) return lsd_fail(ctx, "bad level range");
    std::vector<Sim3Item> items(n);
    for (int i = 0; i < n; i++) {
        FrameSlot* kf = findSlot(ctx, ref_ids[i]);
        FrameSlot* fr = findSlot(ctx, frame_ids[i]);
        if (!kf || !fr) return lsd_fail(ctx, "unknown frame id");
        int r = ensureIdepthPyramid(ctx, kf);       // reference->makePointCloud(lvl), Sim3Tracker.cpp:174
        if (r) return r;
        r = ensureIdepthPyramid(ctx, fr);           // frame->idepth(level) / idepthVar(level), :467-468
        if (r) return r;
        for (int l = 0; l < LSD_LEVELS; l++) {
            items[i].kfIdepth[l] = kf->idepth[l]; items[i].kfVar[l] = kf->idepthVar[l]; items[i].kfGrad[l] = kf->grad[l];
            items[i].frGrad[l] = fr->grad[l]; items[i].frIdepth[l] = fr->idepth[l]; items[i].frVar[l] = fr->idepthVar[l];
        }
        lsd::Sim3 T = lsd::sim3FromQts(qts + 8 * i);
        if (!qtsIsRefToFrame) T = lsd::sim3Inverse(T);                  // :161
        for (int k = 0; k < 4; k++) items[i].refToFrame[k] = T.q[k];
        for (int k = 0; k < 3; k++) items[i].refToFrame[4 + k] = T.t[k];
    }
    LSD_CHECK(ctx, cudaMemcpyAsync(ctx->dSim3Items, items.data(), n * sizeof(Sim3Item), cudaMemcpyHostToDevice, ctx->stream));
    Sim3Params P;
    memset(&P, 0, sizeof(P));
    for (int l = 0; l < LSD_LEVELS; l++) {
        const LevelCam& c = ctx->cam[l];
        Sim3Level& L = P.lvl[l];
        L.w = c.w; L.h = c.h; L.fx = c.fx; L.fy = c.fy; L.cx = c.cx; L.cy = c.cy; L.fxi = c.fxi; L.fyi = c.fyi; L.cxi = c.cxi; L.cyi = c.cyi;
    }
    lsdgpu_track_settings ds;
    if (!s) { lsdgpu_default_track_settings(&ds); s = &ds; }
    P.st = *s;
    P.cameraPixelNoise2 = ctx->g.cameraPixelNoise2;
    P.useAffine = ctx->g.useAffineLightningEstimation;
    P.W = ctx->w; P.H = ctx->h;
    P.startLevel = startLevel; P.finalLevel = finalLevel;
    P.evalOnly = evalOnly; P.evalA = evalA; P.evalB = evalB;
    // one cluster per problem: 8 CTAs (the portable maximum) unless the batch alone fills the GPU
    int cs = 8;
    if (const char* e = getenv("LSDGPU_SIM3_CLUSTER")) cs = atoi(e);
    else if (n >= 2 * ctx->smCount) cs = 1;
    else if (n * 8 > 2 * ctx->smCount) cs = (n * 4 > 2 * ctx->smCount) ? ((n * 2 > 2 * ctx->smCount) ? 1 : 2) : 4;
    if (cs != 1 && cs != 2 && cs != 4 && cs != 8) cs = 8;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(n * cs); cfg.blockDim = dim3(S3_THREADS); cfg.dynamicSmemBytes = 0; cfg.stream = ctx->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    LSD_CHECK(ctx, cudaLaunchKernelEx(&cfg, k_sim3_track, P, (const Sim3Item*)ctx->dSim3Items, (Sim3Out*)ctx->dSim3Outs));
    LAUNCH(ctx);
    hout.resize(n);
    LSD_CHECK(ctx, cudaMemcpyAsync(hout.data(), ctx->dSim3Outs, n * sizeof(Sim3Out), cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (getenv("LSDGPU_SIM3_DEBUG")) {
        const Sim3Out& o = hout[0];
        int ev = 0;
        for (int l = 0; l < LSD_LEVELS; l++) ev += o.nRes[l];
        fprintf(stderr, "[sim3] cluster=%d evals=%d cycles: points=%lld ctaReduce=%lld exchange=%lld serialLM=%lld\n", cs, ev, o.cyc[0], o.cyc[1], o.cyc[2], o.cyc[3]);
    }
    return 0;
}

extern "C" int lsdgpu_sim3_eval(lsdgpu_ctx* ctx, int ref_kf_id, int frame_id, int level, const double refToFrame_qts[8],
                                float affine_a, float affine_b, const lsdgpu_track_settings* s, lsdgpu_sim3_eval_result* out)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    std::vector<Sim3Out> h;
    int r = sim3Launch(ctx, 1, &ref_kf_id, &frame_id, refToFrame_qts, true, level, level, s, 1, affine_a, affine_b, h);
    if (r) return r;
    const float* sm = h[0].sums;
    sim3AssembleLGS7(sm, out->A, out->b);
    const Sim3Res res = sim3Finish(sm);
    out->num_constraints = 2 * res.warpedSize;
    out->sumResD = sm[S3_RESD]; out->sumResP = sm[S3_RESP]; out->numTermsD = (int)sm[S3_NUMD]; out->numTermsP = (int)sm[S3_NUMP];
    out->mean = res.mean; out->meanD = res.meanD; out->meanP = res.meanP;
    out->warpedSize = res.warpedSize; out->pointUsage = res.pointUsage;
    out->affine_a_lastIt = res.a_lastIt; out->affine_b_lastIt = res.b_lastIt;
    return 0;
}

extern "C" int lsdgpu_sim3_track_batch(lsdgpu_ctx* ctx, int n, const int* ref_kf_ids, const int* frame_ids, const double* frameToRef_init_qts,
                                       int start_level, int final_level, const lsdgpu_track_settings* s, lsdgpu_sim3_result* results)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    std::vector<Sim3Out> h;
    int r = sim3Launch(ctx, n, ref_kf_ids, frame_ids, frameToRef_init_qts, false, start_level, final_level, s, 0, 1.f, 0.f, h);
    if (r) return r;
    for (int i = 0; i < n; i++) {
        lsdgpu_sim3_result& o = results[i];
        const Sim3Out& d = h[i];
        memset(&o, 0, sizeof(o));
        o.frameToRef_qts[3] = 1; o.frameToRef_qts[7] = 1;                               // Sim3()
        o.pointUsage = d.pointUsage; o.affineEstimation_a = d.affine_a; o.affineEstimation_b = d.affine_b;
        for (int l = 0; l < LSD_LEVELS; l++) { o.numCalcResidualCalls[l] = d.nRes[l]; o.numCalcWarpUpdateCalls[l] = d.nUpd[l]; }
        if (d.early) { o.diverged = (d.early == 1); continue; }                         // :184-187, :212-217, :231-235
        float b7[7];
        sim3AssembleLGS7(d.lgs, o.lastSim3Hessian, b7);                                 // lastSim3Hessian = ls7.A, :360
        lsd::Sim3 T;
        for (int k = 0; k < 4; k++) T.q[k] = d.refToFrame[k];
        for (int k = 0; k < 3; k++) T.t[k] = d.refToFrame[4 + k];
        if (lsd::sim3Scale(T) <= 0) { o.diverged = 1; continue; }                       // :363-367
        o.lastResidual = d.resMean; o.lastDepthResidual = d.resMeanD; o.lastPhotometricResidual = d.resMeanP;   // :369-371
        lsd::sim3ToQts(lsd::sim3Inverse(T), o.frameToRef_qts);                          // :374
    }
    return 0;
}

extern "C" int lsdgpu_sim3_track(lsdgpu_ctx* ctx, int ref_kf_id, int frame_id, const double frameToRef_init_qts[8],
                                 int start_level, int final_level, const lsdgpu_track_settings* s, lsdgpu_sim3_result* out)
{ LSD_LOCK(ctx);
    return lsdgpu_sim3_track_batch(ctx, 1, &ref_kf_id, &frame_id, frameToRef_init_qts, start_level, final_level, s, out);
}

// ------------------------------------------------------------------------------------------------------
// keyframe output formats (SURVEY 8f row 4)
// ------------------------------------------------------------------------------------------------------
extern "C" int lsdgpu_keyframe_pack_pointcloud(lsdgpu_ctx* ctx, int kf_id, int publish_level, lsdgpu_input_point_dense* out)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, kf_id);
    if (!kf) return lsd_fail(ctx, "unknown keyframe id");
    if (publish_level < 0 || publish_level >= LSD_LEVELS) return lsd_fail(ctx, "bad level");
    int r = ensureIdepthPyramid(ctx, kf);                      // f->idepth(publishLvl), ROSOutput3DWrapper.cpp:96-97
    if (r) return r;
    const int n = (ctx->w >> publish_level) * (ctx->h >> publish_level);
    k_pack_pointcloud<<<divUp(3 * n, 256), 256, 0, ctx->stream>>>(kf->idepth[publish_level], kf->idepthVar[publish_level],
                                                                  kf->image[publish_level], n, ctx->dPacked);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    LSD_CHECK(ctx, cudaMemcpyAsync(out, ctx->dPacked, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

// ------------------------------------------------------------------------------------------------------
// map export: KeyFrameDisplay::flushPC over many resident keyframes (mapexport.cuh)
// ------------------------------------------------------------------------------------------------------
// Device staging outside the arena, so that contexts which never export keep the arena layout the peer-sharded tracker
// requires to be identical on every rank.  The record buffers are sized once (two chunks of MAP_CHUNK worst-case
// keyframes); the per-keyframe index arrays are sized for max(max_frames, n_kf) and only grow when a call lists more keyframes.
struct MapStaging {
    int kfCap = 0, bandCap = 0;
    MapKf* dKf = nullptr;
    MapKf* hKf = nullptr;                // pinned
    int* dCta = nullptr;                 // [kfCap * bandCap] per-CTA counts
    long long* dOff = nullptr;           // [kfCap * bandCap] output offsets
    int* dKfCount = nullptr;             // [kfCap]
    long long* dTotal = nullptr;
    int* hKfCount = nullptr;             // pinned [kfCap]
    long long* hTotal = nullptr;         // pinned
    float4* dRec[2] = { nullptr, nullptr };
    cudaStream_t copy = nullptr;         // device-to-host copies of the records, overlapping the next chunk's kernel
    cudaEvent_t kernDone[2] = { nullptr, nullptr }, copyDone[2] = { nullptr, nullptr };
};

static int mapBandRows(int W)
{   // (rows + 2) x W floats of shared memory: at most 48 KB where the width allows it, at most 16 rows
    return std::max(1, std::min(16, 48 * 1024 / (4 * std::max(W, 1)) - 2));
}

static void mapFreeIndex(MapStaging* m)
{
    cudaFree(m->dKf); cudaFree(m->dCta); cudaFree(m->dOff); cudaFree(m->dKfCount);
    cudaFreeHost(m->hKf); cudaFreeHost(m->hKfCount);
    m->dKf = nullptr; m->dCta = nullptr; m->dOff = nullptr; m->dKfCount = nullptr; m->hKf = nullptr; m->hKfCount = nullptr;
    m->kfCap = 0;
}

static void mapStagingFree(lsdgpu_ctx* ctx)
{
    MapStaging* m = ctx->map;
    if (!m) return;
    if (m->copy) cudaStreamSynchronize(m->copy);
    mapFreeIndex(m);
    cudaFree(m->dTotal); cudaFreeHost(m->hTotal);
    cudaFree(m->dRec[0]); cudaFree(m->dRec[1]);
    for (int b = 0; b < 2; b++) {
        if (m->kernDone[b]) cudaEventDestroy(m->kernDone[b]);
        if (m->copyDone[b]) cudaEventDestroy(m->copyDone[b]);
    }
    if (m->copy) cudaStreamDestroy(m->copy);
    delete m;
    ctx->map = nullptr;
}

static int mapReserve(lsdgpu_ctx* ctx, int n_kf)
{
    if (!ctx->map) {
        MapStaging* m = new (std::nothrow) MapStaging();
        if (!m) return lsd_fail(ctx, "out of host memory");
        ctx->map = m;
        int bands = 0;
        for (int l = 0; l < LSD_LEVELS; l++) {
            const int W = ctx->w >> l, H = ctx->h >> l, r = mapBandRows(W);
            if (W >= 3 && H >= 3) bands = std::max(bands, divUp(H - 2, r));
        }
        m->bandCap = std::max(bands, 1);
        const size_t recs = (size_t)MAP_CHUNK * ctx->w * ctx->h;
        LSD_CHECK(ctx, cudaMalloc((void**)&m->dRec[0], recs * sizeof(float4)));
        LSD_CHECK(ctx, cudaMalloc((void**)&m->dRec[1], recs * sizeof(float4)));
        LSD_CHECK(ctx, cudaMalloc((void**)&m->dTotal, sizeof(long long)));
        LSD_CHECK(ctx, cudaHostAlloc((void**)&m->hTotal, sizeof(long long), cudaHostAllocDefault));
        LSD_CHECK(ctx, cudaStreamCreateWithFlags(&m->copy, cudaStreamNonBlocking));
        for (int b = 0; b < 2; b++) {
            LSD_CHECK(ctx, cudaEventCreateWithFlags(&m->kernDone[b], cudaEventDisableTiming));
            LSD_CHECK(ctx, cudaEventCreateWithFlags(&m->copyDone[b], cudaEventDisableTiming));
        }
        const size_t smem = (size_t)(mapBandRows(ctx->w) + 2) * ctx->w * 4;
        if (smem > 48 * 1024) {
            LSD_CHECK(ctx, cudaFuncSetAttribute(k_map_points<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            LSD_CHECK(ctx, cudaFuncSetAttribute(k_map_points<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        }
    }
    MapStaging* m = ctx->map;
    if (n_kf <= m->kfCap) return 0;
    mapFreeIndex(m);
    const int cap = std::max(n_kf, (int)ctx->slots.size());
    const size_t nc = (size_t)cap * m->bandCap;
    LSD_CHECK(ctx, cudaMalloc((void**)&m->dKf, (size_t)cap * sizeof(MapKf)));
    LSD_CHECK(ctx, cudaMalloc((void**)&m->dCta, nc * sizeof(int)));
    LSD_CHECK(ctx, cudaMalloc((void**)&m->dOff, nc * sizeof(long long)));
    LSD_CHECK(ctx, cudaMalloc((void**)&m->dKfCount, (size_t)cap * sizeof(int)));
    LSD_CHECK(ctx, cudaHostAlloc((void**)&m->hKf, (size_t)cap * sizeof(MapKf), cudaHostAllocDefault));
    LSD_CHECK(ctx, cudaHostAlloc((void**)&m->hKfCount, (size_t)cap * sizeof(int), cudaHostAllocDefault));
    m->kfCap = cap;
    return 0;
}

extern "C" int lsdgpu_map_export_points(lsdgpu_ctx* ctx, int n_kf, const int* kf_ids, const double* camToWorld_qts, int publish_level,
                                        const lsdgpu_map_filter* f, lsdgpu_map_point* out, long long capacity, int* counts_out,
                                        long long* total_out)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    if (n_kf < 0 || !f || (n_kf > 0 && (!kf_ids || !camToWorld_qts)) || (out && capacity < 0)) return lsd_fail(ctx, "bad arguments");
    if (publish_level < 0 || publish_level >= LSD_LEVELS) return lsd_fail(ctx, "bad level");
    std::vector<FrameSlot*> kfs(n_kf);
    for (int i = 0; i < n_kf; i++) {
        kfs[i] = findSlot(ctx, kf_ids[i]);
        if (!kfs[i]) return lsd_fail(ctx, "unknown keyframe id");
        if (!kfs[i]->hasDepth) return lsd_fail(ctx, "keyframe has no depth");
    }
    const LevelCam& cam = ctx->cam[publish_level];
    MapParams p;
    p.W = cam.w; p.H = cam.h;
    p.bandRows = mapBandRows(p.W);
    p.nBands = (p.W >= 3 && p.H >= 3) ? divUp(p.H - 2, p.bandRows) : 0;
    p.fxi = 1 / cam.fx; p.fyi = 1 / cam.fy; p.cxi = -cam.cx / cam.fx; p.cyi = -cam.cy / cam.fy;   // KeyFrameDisplay.cpp:75-78
    p.scaledTH = f->scaledDepthVarTH; p.absTH = f->absDepthVarTH; p.minNearSupport = f->minNearSupport;
    if (n_kf == 0 || p.nBands == 0) {
        if (counts_out) for (int i = 0; i < n_kf; i++) counts_out[i] = 0;
        if (total_out) *total_out = 0;
        return 0;
    }
    for (FrameSlot* s : kfs) {                                      // f->idepth(publishLvl), ROSOutput3DWrapper.cpp:96-97
        int r = ensureIdepthPyramid(ctx, s);
        if (r) return r;
    }
    int r = mapReserve(ctx, n_kf);
    if (r) return r;
    MapStaging* m = ctx->map;
    for (int i = 0; i < n_kf; i++) {
        MapKf& k = m->hKf[i];
        k.idepth = kfs[i]->idepth[publish_level]; k.var = kfs[i]->idepthVar[publish_level]; k.img = kfs[i]->image[publish_level];
        // getScaledCamToWorld().cast<float>() (ROSOutput3DWrapper.cpp:85): the Sophus storage, quaternion with |q| = scale
        const double* a = camToWorld_qts + 8 * (size_t)i;
        float q[4];
        for (int j = 0; j < 4; j++) q[j] = (float)(a[j] * a[7]);
        for (int j = 0; j < 3; j++) k.t[j] = (float)a[4 + j];
        k.scale = sqrtf((q[0] * q[0] + q[1] * q[1]) + (q[2] * q[2] + q[3] * q[3]));       // Eigen's tree reduction
        for (int j = 0; j < 4; j++) k.nq[j] = q[j] / k.scale;
    }
    LSD_CHECK(ctx, cudaMemcpyAsync(m->dKf, m->hKf, (size_t)n_kf * sizeof(MapKf), cudaMemcpyHostToDevice, ctx->stream));
    const size_t smem = (size_t)(p.bandRows + 2) * p.W * 4;
    for (int b = 0; b < n_kf; b += 65535) {
        k_map_points<false><<<dim3(p.nBands, std::min(65535, n_kf - b)), MAP_THREADS, smem, ctx->stream>>>(m->dKf, b, p, m->dCta, nullptr, 0, nullptr);
        LAUNCH(ctx);
    }
    k_map_scan<<<1, 1024, 0, ctx->stream>>>(m->dCta, n_kf * p.nBands, p.nBands, m->dOff, m->dKfCount, m->dTotal);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    LSD_CHECK(ctx, cudaMemcpyAsync(m->hKfCount, m->dKfCount, (size_t)n_kf * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaMemcpyAsync(m->hTotal, m->dTotal, sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    const long long total = *m->hTotal;
    if (out && total > capacity) return lsd_fail(ctx, "map export: capacity is smaller than the number of points");
    if (out && total > 0) {
        std::vector<long long> kfOff(n_kf + 1, 0);
        for (int i = 0; i < n_kf; i++) kfOff[i + 1] = kfOff[i] + m->hKfCount[i];
        for (int c = 0, ci = 0; c < n_kf; c += MAP_CHUNK, ci++) {
            const int e = std::min(c + MAP_CHUNK, n_kf), b = ci & 1;
            if (ci >= 2) LSD_CHECK(ctx, cudaStreamWaitEvent(ctx->stream, m->copyDone[b], 0));     // buffer b still being copied out
            k_map_points<true><<<dim3(p.nBands, e - c), MAP_THREADS, smem, ctx->stream>>>(m->dKf, c, p, nullptr, m->dOff, kfOff[c], m->dRec[b]);
            LAUNCH(ctx);
            LSD_CHECK(ctx, cudaGetLastError());
            LSD_CHECK(ctx, cudaEventRecord(m->kernDone[b], ctx->stream));
            LSD_CHECK(ctx, cudaStreamWaitEvent(m->copy, m->kernDone[b], 0));
            const long long n = kfOff[e] - kfOff[c];
            if (n) LSD_CHECK(ctx, cudaMemcpyAsync(out + kfOff[c], m->dRec[b], (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, m->copy));
            LSD_CHECK(ctx, cudaEventRecord(m->copyDone[b], m->copy));
        }
        LSD_CHECK(ctx, cudaStreamSynchronize(m->copy));
        LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    }
    if (counts_out) memcpy(counts_out, m->hKfCount, (size_t)n_kf * sizeof(int));
    if (total_out) *total_out = total;
    return 0;
}

extern "C" int lsdgpu_frame_take_reactivation_data(lsdgpu_ctx* ctx, int kf_id)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, kf_id);
    if (!kf) return lsd_fail(ctx, "unknown keyframe id");
    if (ctx->activeKf != kf_id) return lsd_fail(ctx, "takeReActivationData: the keyframe is not the active one");
    return takeReactivationData(ctx, kf);
}

extern "C" int lsdgpu_frame_download_reactivation_data(lsdgpu_ctx* ctx, int kf_id, float* idepth_reAct, float* idepthVar_reAct, uint8_t* validity_reAct)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, kf_id);
    if (!kf) return lsd_fail(ctx, "unknown keyframe id");
    if (!kf->reactValid) return lsd_fail(ctx, "keyframe has no reactivation data");
    const size_t n = (size_t)ctx->w * ctx->h;
    if (idepth_reAct) LSD_CHECK(ctx, cudaMemcpyAsync(idepth_reAct, kf->reactIdepth, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (idepthVar_reAct) LSD_CHECK(ctx, cudaMemcpyAsync(idepthVar_reAct, kf->reactVar, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (validity_reAct) LSD_CHECK(ctx, cudaMemcpyAsync(validity_reAct, kf->reactValidity, n, cudaMemcpyDeviceToHost, ctx->stream));
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int lsdgpu_depth_set_from_existing_kf(lsdgpu_ctx* ctx, int kf_id)
{ LSD_LOCK(ctx);   // DepthMap::setFromExistingKF :920-962
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* kf = findSlot(ctx, kf_id);
    if (!kf) return lsd_fail(ctx, "unknown keyframe id");
    if (!kf->hasDepth) return lsd_fail(ctx, "setFromExistingKF: keyframe has no depth");          // assert(kf->hasIDepthBeenSet()), :922
    if (!kf->reactValid) return lsd_fail(ctx, "setFromExistingKF: keyframe has no reactivation data");
    const int n = ctx->w * ctx->h;
    k_set_from_existing<<<divUp(n, 256), 256, 0, ctx->stream>>>(kf->reactIdepth, kf->reactVar, kf->reactValidity, ctx->cur, n);
    LAUNCH(ctx);
    LSD_CHECK(ctx, cudaGetLastError());
    ctx->activeKf = kf_id; ctx->activeKfReactivated = true;                                       // :925, :935
    kf->numMappedOnThis = 0; kf->numFramesTrackedOnThis = 0;                                      // :932-933
    return runRegularize(ctx, false, VAL_SUM_MIN_FOR_KEEP);                                       // :961
}

// ------------------------------------------------------------------------------------------------------
// input staging: UndistorterPTAM (SURVEY 8f row 3)
// ------------------------------------------------------------------------------------------------------
// Output camera of UndistorterPTAM for the "crop" / "full" / explicit modes and the remap tables (Undistorter.cpp:171-317).
// The expressions keep the reference's float / double mixing (int and 0.5 literals promote as written there); math calls on
// float arguments use the float overloads.
extern "C" int lsdgpu_undistorter_ptam_prepare(const float ic[5], int iw, int ih, const float ocIn[5], int ow, int oh,
                                               float* remapX, float* remapY, float K_out[9])
{
    if (!ic || !ocIn || iw <= 0 || ih <= 0 || ow <= 0 || oh <= 0) return -2;
    const float dist = ic[4];
    const float d2t = 2.0f * tanf(dist / 2.0f);
    float fx = ic[0] * iw, fy = ic[1] * ih;
    float cx = (float)((double)(ic[2] * iw) - 0.5), cy = (float)((double)(ic[3] * ih) - 0.5);
    // the reference rescales by in_width / in_width == 1.0 in double (:187-192): exact no-ops, including (c + 0.5) - 0.5
    auto undistRadius = [&](float r) { return tanf(r * dist) / d2t; };
    float ofx, ofy, ocx, ocy;
    if (ic[4] == 0) {
        ofx = ic[0] * ow; ofy = ic[1] * oh;
        ocx = (float)((double)(ic[2] * ow) - 0.5); ocy = (float)((double)(ic[3] * oh) - 0.5);
    } else if (ocIn[0] == -1 || ocIn[0] == -2) {
        const float rl = cx / fx, rr = (iw - 1 - cx) / fx, rt = cy / fy, rb = (ih - 1 - cy) / fy;
        const float sx = (float)ow / (float)iw, sy = (float)oh / (float)ih;
        if (ocIn[0] == -1) {            // "crop": the axis-aligned extremes
            const float tl = undistRadius(rl), tr = undistRadius(rr), tt = undistRadius(rt), tb = undistRadius(rb);
            ofy = fy * ((rt + rb) / (tt + tb)) * sy;
            ocy = (tt / rt) * ofy * cy / fy;
            ofx = fx * ((rl + rr) / (tl + tr)) * sx;
            ocx = (tl / rl) * ofx * cx / fx;
        } else {                        // "full": the four corners
            const float c_tl = sqrtf(rl * rl + rt * rt), c_tr = sqrtf(rr * rr + rt * rt);
            const float c_bl = sqrtf(rl * rl + rb * rb), c_br = sqrtf(rr * rr + rb * rb);
            const float u_tl = undistRadius(c_tl), u_tr = undistRadius(c_tr), u_bl = undistRadius(c_bl), u_br = undistRadius(c_br);
            const float hor = fmaxf(c_br, c_tr) + fmaxf(c_bl, c_tl), vert = fmaxf(c_tr, c_tl) + fmaxf(c_bl, c_br);
            const float uhor = fmaxf(u_br, u_tr) + fmaxf(u_bl, u_tl), uvert = fmaxf(u_tr, u_tl) + fmaxf(u_bl, u_br);
            ofy = fy * ((vert) / (uvert)) * sy;
            ocy = fmaxf(u_tl / c_tl, u_tr / c_tr) * ofy * cy / fy;
            ofx = fx * ((hor) / (uhor)) * sx;
            ocx = fmaxf(u_bl / c_bl, u_tl / c_tl) * ofx * cx / fx;
        }
    } else {
        ofx = ocIn[0] * ow; ofy = ocIn[1] * oh;
        ocx = (float)((double)(ocIn[2] * ow) - 0.5); ocy = (float)((double)(ocIn[3] * oh) - 0.5);
    }
    // outputCalibration (:268-272) and K_ as main_on_images.cpp:164-167 reads it back
    const float oc0 = ofx / ow, oc1 = ofy / oh;
    const float oc2 = (float)(((double)ocx + 0.5) / ow), oc3 = (float)(((double)ocy + 0.5) / oh);
    if (K_out) {
        for (int i = 0; i < 9; i++) K_out[i] = 0.f;
        K_out[0] = oc0 * ow; K_out[4] = oc1 * oh;
        K_out[2] = (float)((double)(oc2 * ow) - 0.5); K_out[5] = (float)((double)(oc3 * oh) - 0.5);
        K_out[8] = 1.f;
    }
    if (remapX && remapY)
        for (int y = 0; y < oh; y++)
            for (int x = 0; x < ow; x++) {
                float ix = (x - ocx) / ofx, iy = (y - ocy) / ofy;
                const float r = sqrtf(ix * ix + iy * iy);
                const float fac = (r == 0 || dist == 0) ? 1 : atanf(r * d2t) / (dist * r);
                ix = fx * fac * ix + cx;
                iy = fy * fac * iy + cy;
                // "make rounding resistant" (:299-303; the last line assigns ix in the reference, kept)
                if (ix == 0) ix = (float)0.01;
                if (iy == 0) iy = (float)0.01;
                if (ix == iw - 1) ix = (float)(iw - 1.01);
                if (iy == ih - 1) ix = (float)(ih - 1.01);
                const bool inside = ix > 0 && iy > 0 && ix < iw - 1 && iy < ih - 1;
                remapX[x + y * ow] = inside ? ix : -1.f;
                remapY[x + y * ow] = inside ? iy : -1.f;
            }
    return (ih == oh && iw == ow && ic[4] == 0) ? 1 : 0;
}

extern "C" int lsdgpu_undistorter_validate_tables(int in_width, int in_height, int out_width, int out_height, const float* remapX, const float* remapY)
{
    if (!remapX || !remapY || in_width < 2 || in_height < 2 || out_width <= 0 || out_height <= 0) return -2;
    const long long n = (long long)out_width * out_height;
    for (long long i = 0; i < n; i++) {
        const float x = remapX[i], y = remapY[i];
        if (x < 0) continue;                                               // undistort() writes 0 (Undistorter.cpp:389-390)
        if (!(x >= 0 && y >= 0 && x < in_width - 1 && y < in_height - 1)) return (int)(1 + (i < 0x7ffffffeLL ? i : 0x7ffffffeLL));   // also NaN
    }
    return 0;
}

extern "C" int lsdgpu_set_undistorter(lsdgpu_ctx* ctx, int in_width, int in_height, const float* remapX, const float* remapY)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    if (in_width <= 0 || in_height <= 0) return lsd_fail(ctx, "bad input size");
    const size_t n = (size_t)ctx->w * ctx->h, nr = (size_t)in_width * in_height;
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->dRemapX) { cudaFree(ctx->dRemapX); ctx->dRemapX = nullptr; }
    if (ctx->dRemapY) { cudaFree(ctx->dRemapY); ctx->dRemapY = nullptr; }
    if (ctx->dRaw) { cudaFree(ctx->dRaw); ctx->dRaw = nullptr; }
    if (ctx->hRaw) { cudaFreeHost(ctx->hRaw); ctx->hRaw = nullptr; }
    ctx->undistorterSet = false;
    if (!remapX || !remapY) {
        if (in_width != ctx->w || in_height != ctx->h) return lsd_fail(ctx, "pass-through undistorter needs input size == context size");
    } else {
        if (lsdgpu_undistorter_validate_tables(in_width, in_height, ctx->w, ctx->h, remapX, remapY) != 0)
            return lsd_fail(ctx, "remap table entry outside the input image (lsdgpu_undistorter_validate_tables)");
        LSD_CHECK(ctx, cudaMalloc((void**)&ctx->dRemapX, n * 4));
        LSD_CHECK(ctx, cudaMalloc((void**)&ctx->dRemapY, n * 4));
        LSD_CHECK(ctx, cudaMemcpy(ctx->dRemapX, remapX, n * 4, cudaMemcpyHostToDevice));
        LSD_CHECK(ctx, cudaMemcpy(ctx->dRemapY, remapY, n * 4, cudaMemcpyHostToDevice));
    }
    LSD_CHECK(ctx, cudaMalloc((void**)&ctx->dRaw, nr));
    LSD_CHECK(ctx, cudaHostAlloc((void**)&ctx->hRaw, nr, cudaHostAllocDefault));
    ctx->rawW = in_width; ctx->rawH = in_height;
    ctx->undistorterSet = true;
    return 0;
}

static int uploadRaw(lsdgpu_ctx* ctx, const uint8_t* raw)
{
    if (!ctx->undistorterSet) return lsd_fail(ctx, "no undistorter installed (lsdgpu_set_undistorter)");
    const size_t nr = (size_t)ctx->rawW * ctx->rawH;
    cudaPointerAttributes pa;
    const bool pinned = cudaPointerGetAttributes(&pa, raw) == cudaSuccess && pa.type == cudaMemoryTypeHost;
    if (!pinned) {
        cudaGetLastError();
        LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));          // the previous raw image may still be in flight
        memcpy(ctx->hRaw, raw, nr);
    }
    LSD_CHECK(ctx, cudaMemcpyAsync(ctx->dRaw, pinned ? raw : ctx->hRaw, nr, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}

extern "C" int lsdgpu_undistort_u8(lsdgpu_ctx* ctx, const uint8_t* raw, uint8_t* out)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    int r = uploadRaw(ctx, raw);
    if (r) return r;
    const int n = ctx->w * ctx->h;
    if (!ctx->dRemapX) {                                              // result = image, Undistorter.cpp:370-375
        LSD_CHECK(ctx, cudaMemcpyAsync(out, ctx->dRaw, n, cudaMemcpyDeviceToHost, ctx->stream));
    } else {
        uint8_t* dOut = ctx->dStageU8[ctx->stageIdx];
        LSD_CHECK(ctx, cudaEventSynchronize(ctx->stageDone[ctx->stageIdx]));
        k_undistort<<<divUp(n, 256), 256, 0, ctx->stream>>>(ctx->dRaw, ctx->rawW, ctx->dRemapX, ctx->dRemapY, n, dOut);
        LAUNCH(ctx);
        LSD_CHECK(ctx, cudaGetLastError());
        LSD_CHECK(ctx, cudaMemcpyAsync(out, dOut, n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    LSD_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int lsdgpu_frame_upload_distorted_u8(lsdgpu_ctx* ctx, int frame_id, const uint8_t* raw)
{ LSD_LOCK(ctx);
    LSD_CHECK(ctx, cudaSetDevice(ctx->device));
    FrameSlot* s = acquireSlot(ctx, frame_id);
    if (!s) return lsd_fail(ctx, "no free frame slot (release frames or raise max_frames)");
    int r = uploadRaw(ctx, raw);
    if (r) return r;
    return buildFrameFromDeviceU8(ctx, s, ctx->dRaw, ctx->dRemapX != nullptr);
}
