// internal.cuh -- context, device layouts and launch helpers of liblsdgpu (not part of the ABI).
//
// Data layout in HBM (DESIGN.md section 3):
//   * one arena per context, carved into `max_frames` frame slots + one depth map + tracker scratch;
//   * frame slot: image pyramid f32 planar L0..L4, gradient pyramid float4 (dx,dy,I,0) L0..L4,
//     maxGradients L0 f32, idepth / idepthVar pyramids f32 L0..L4, refPixelWasGood u8 at L1;
//   * depth map: two ping-pong copies (current / other) of the hypothesis field, each as two 16-byte planes
//       hf = float4(idepth, idepth_var, idepth_smoothed, idepth_var_smoothed)
//       hi = int4  (isValid, blacklisted, validity_counter, bits(nextStereoFrameMinID))
//     (the reference's 32-byte AoS record split in halves, so that every access is one 128-bit transaction),
//     plus the int32 validity integral image.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/lsdgpu.h"
#include "hostmath.h"

#define LSD_LEVELS LSDGPU_LEVELS
#define SE3TRACKING_MIN_LEVEL 1
#define SE3TRACKING_MAX_LEVEL 5

struct LevelCam {
    int w, h;
    float fx, fy, cx, cy;
    float fxi, fyi, cxi, cyi;
    float K[9], KInv[9];
};

struct FrameSlot {
    int id = -1;
    bool used = false;
    float* image[LSD_LEVELS];
    float4* grad[LSD_LEVELS];
    float* maxgrad;
    float* idepth[LSD_LEVELS];
    float* idepthVar[LSD_LEVELS];
    uint8_t* goodMask;
    float4* permaPC = nullptr;           // permaRef: (x, y, z, colour) per level-4 point (Frame::setPermaRef)
    float* permaVar = nullptr;
    int permaNumPts = 0;
    float* reactIdepth = nullptr;        // Frame::idepth_reAct / idepthVar_reAct / validity_reAct (Frame.cpp:107-145), device-resident
    float* reactVar = nullptr;
    uint8_t* reactValidity = nullptr;
    bool reactAllocated = false, reactValid = false;
    CUtensorMap gradMap[LSD_LEVELS];     // TMA descriptors of grad[l] (float4 texels as 4 x f32), box = tracker window
    bool hasDepth = false, idepthPyrValid = false, hasGoodMask = false;
    bool depthHasBeenUpdatedFlag = false;
    float meanIdepth = 1.f;
    int numPoints = 0;
    double* dStats = nullptr;            // device: sum(idepth_smoothed), count, rescale (written by setDepth kernels)
    bool statsPending = false;           // meanIdepth / numPoints still have to be fetched from dStats
    double thisToParent[8];
    int parentId = -1;
    float initialTrackedResidual = 0.f;
    int numFramesTrackedOnThis = 0, numMappedOnThis = 0;
};

struct HypField {
    float4* hf;
    int4* hi;
};

// per reference-frame constants of Frame::prepareForStereoWith (Frame.cpp:295-317) + what observeDepth reads
struct RefConst {
    float K_otherToThis_R[9];
    float K_otherToThis_t[3];
    float otherToThis_t[3];
    float thisToOther_t[3];
    float row0[3], row1[3], row2[3];
    float initialTrackedResidual;
    int id;
    int trackedOnActive;          // refFrame->getTrackingParent() == activeKeyFrame
    const float* image;           // level 0
    const uint8_t* goodMask;      // refPixelWasGoodNoCreate() or nullptr
};
#define LSD_MAX_PERMA_BATCH 4096
#define LSD_MAX_REFS 16
#define LSD_MAX_ID_SPAN 64
struct ObserveParams {
    RefConst refs[LSD_MAX_REFS];
    int nRefs;
    int byIdOffset, byIdSize;     // referenceFrameByID_offset / size
    int byId[LSD_MAX_ID_SPAN];    // id - offset -> index into refs
    int oldestIdx, newestIdx;
    int reactivated;
    int kfNumTracked, kfNumMapped;
};

// per-warp shared-memory window of the new frame's gradient level used by the persistent tracker: WIN_W x WIN_H
// float4 texels, loaded by one TMA box copy per warp and level (track_persistent.cuh)
#define TRK_WIN_W 48
#define TRK_WIN_H 17

// number of reduction channels of one tracker evaluation (see track.cuh)
#define EV_NCH 40

struct lsdgpu_ctx {
    // Every entry point of the C ABI holds this for its whole duration (LSD_LOCK): one context may be shared by SlamSystem's
    // tracking and mapping threads (SlamSystem.cpp:111, :206) -- their calls serialise here, as they do on the frame / keyframe
    // locks of the reference (Frame::getActiveLock, SE3Tracker.cpp:286, DepthMap.cpp:1104).  Recursive: the fused entry points
    // (lsdgpu_track_and_map, lsdgpu_sim3_track) call other entry points.
    mutable std::recursive_mutex mu;
    int device = 0;
    int w = 0, h = 0;
    LevelCam cam[LSD_LEVELS];
    lsdgpu_globals g;
    cudaStream_t stream = nullptr;
    std::string err;
    long long launches = 0;
    int smCount = 148;

    char* arena = nullptr;
    size_t arenaBytes = 0;
    std::vector<FrameSlot> slots;

    // depth map
    HypField cur, oth;
    int* integral = nullptr;
    int activeKf = -1;
    bool activeKfReactivated = false;
    ObserveParams hObs;                  // passed to k_observe by value (__grid_constant__)
    int* propHead = nullptr;             // per-target list heads (propagateDepth)
    int* propNext = nullptr;
    float4* propVal = nullptr;           // per-source (new_idepth, new_var, validity, -)
    double* dScalars = nullptr;          // small device scratch for reductions (sum, count)
    double* hScalars = nullptr;          // pinned mirror

    // tracker scratch
    float* evPartials = nullptr;         // [maxBlocks][EV_NCH]
    unsigned int* evCounter = nullptr;
    float* dEvOut = nullptr;             // EV_NCH floats (device)
    float* hEvOut = nullptr;             // pinned host mirror
    void* dTrackState = nullptr;         // persistent-kernel state block (device)
    void* hTrackState = nullptr;         // mapped pinned result block (host view)
    void* dTrackStateMapped = nullptr;   // device view of the same block
    int trackUseTma = 1;
    void* dPermaItems = nullptr;         // batched permaRef tracking: candidate descriptors / results (device)
    void* dPermaResults = nullptr;
    void* dSim3Items = nullptr;          // batched Sim3 tracking: problem descriptors / results (device)
    void* dSim3Outs = nullptr;
    float* dRemapX = nullptr;            // UndistorterPTAM remap tables (separate allocation), raw-image staging
    float* dRemapY = nullptr;
    uint8_t* dRaw = nullptr;
    uint8_t* hRaw = nullptr;
    int rawW = 0, rawH = 0;
    bool undistorterSet = false;
    uint32_t* dPacked = nullptr;         // keyframeMsg.pointcloud staging: w*h InputPointDense records (device)
    struct MapStaging* map = nullptr;    // lsdgpu_map_export_points staging (mapexport.cuh): its own allocation, made at the first export
    int trackGrid = 148;                 // launch shape of the persistent tracker (set by trackPersistentSetup): one CTA per SM
    int trackG[LSD_LEVELS] = { 1, 1, 1, 1, 1 };          // CTAs taking part in the evaluations of each level
    unsigned int* trkSync = nullptr;     // per-level barrier counters + level records of the persistent tracker (TP_SYNC_WORDS)
    unsigned int trkBase[LSD_LEVELS] = { 0, 0, 0, 0, 0 };  // arrivals already counted on each level's counter (never reset)
    unsigned int tmaTimeoutsSeen = 0;
    // one stream sharded over several GPUs (lsdgpu_peer_attach): every rank's arena mapped into this process
    int nRanks = 1, rank = 0;
    char* peerBase[8] = { nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr };
    unsigned int trkTailBase = 0;
    // environment switches, read once at lsdgpu_create
    int optTrackTma = 1, optSingleSync = 0;
    bool optTrackDebug = false;
    int optTrackKmax = 3;
    bool optPdl = true;                  // LSDGPU_PDL=0: plain stream-ordered launches of the dependent kernels
    int2* seqTable = nullptr;            // seqsum.cuh: per-run maps of the sequential fp32 sum, [SEQ_NBIN][runs]
    unsigned char* seqFlags = nullptr;
    int* seqCounts = nullptr;
    int* dSkipFlag = nullptr;            // device flag: the frame's tracking diverged -> its mapping kernels do nothing
    ObserveParams* dObs = nullptr;       // device-resident observe parameters written by k_prepare_observe
    unsigned int trackSeq = 0;           // sequence number of the last tracking launch (TrackState::doneSeq)
    uint8_t* stageRing = nullptr;        // device prefetch ring of raw u8 frames (separate allocation)
    int stageEntries = 0;
    uint8_t* hStage[2] = { nullptr, nullptr };   // double-buffered pinned staging for the u8 frame upload
    uint8_t* dStageU8[2] = { nullptr, nullptr };
    cudaEvent_t stageDone[2];
    int stageIdx = 0;
    float* hStageF = nullptr;            // pinned float staging (depth / idepth uploads)
    float* dStageF = nullptr;

    // timers
    cudaEvent_t tBegin[8], tEnd[8];
    cudaEvent_t kBegin, kEnd;
    double trackKernelMs = 0;
    long long trackKernelLaunches = 0;
    double trackKernelBytes = 0;
    bool profileTrackKernel = false;
    bool trackProfilePending = false;
    void* encodeTiled = nullptr;         // cuTensorMapEncodeTiled, resolved through cudaGetDriverEntryPoint
};

struct CtxLock {
    std::recursive_mutex* m;
    explicit CtxLock(const lsdgpu_ctx* c) : m(c ? &c->mu : nullptr) { if (m) m->lock(); }
    ~CtxLock() { if (m) m->unlock(); }
    CtxLock(const CtxLock&) = delete;
};
#define LSD_LOCK(ctx) CtxLock lsd_lock_(ctx)

#define LSD_CHECK(ctx, expr)                                                                              \
    do {                                                                                                  \
        cudaError_t _e = (expr);                                                                          \
        if (_e != cudaSuccess) {                                                                          \
            char _b[512];                                                                                 \
            snprintf(_b, sizeof(_b), "%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            (ctx)->err = _b;                                                                              \
            return -1;                                                                                    \
        }                                                                                                 \
    } while (0)

// Programmatic dependent launch (sm_90+): a kernel launched with LSD_PDL_LAUNCH may be scheduled while its predecessor in the stream
// is still running; it must not touch the predecessor's output before pdlWait() returns (griddepcontrol.wait: all memory operations
// of the predecessor grid are complete and visible).  With the wait as the kernel's first statement the stream semantics are
// unchanged; what is saved is the launch latency between dependent kernels of a step.
__device__ __forceinline__ void pdlWait()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
}
template <typename... KArgs, typename... Args>
static inline cudaError_t launchPDL(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl, Args&&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

static inline int lsd_fail(lsdgpu_ctx* ctx, const char* msg)
{
    ctx->err = msg;
    return -2;
}

static inline FrameSlot* findSlot(lsdgpu_ctx* ctx, int id)
{
    for (auto& s : ctx->slots)
        if (s.used && s.id == id) return &s;
    return nullptr;
}

static inline int divUp(int a, int b) { return (a + b - 1) / b; }

// ---- device helpers shared by all kernels --------------------------------------------------------------
// util/settings.h:34-35.  UNZERO mixes float and double literals; every use converts back to float.
__device__ __forceinline__ float unzero_f(float val)
{
    double r = (val < 0 ? (val > -1e-10 ? -1e-10 : (double)val) : (val < 1e-10 ? 1e-10 : (double)val));
    return (float)r;
}

// util/globalFuncs.h:43-61 -- weights formed and summed in the reference's order (br, bl, tr, tl)
__device__ __forceinline__ float interpF(const float* __restrict__ mat, float x, float y, int width)
{
    int ix = (int)x, iy = (int)y;
    float dx = x - ix, dy = y - iy;
    float dxdy = dx * dy;
    const float* bp = mat + ix + iy * width;
    return dxdy * __ldg(bp + 1 + width) + (dy - dxdy) * __ldg(bp + width) + (dx - dxdy) * __ldg(bp + 1) + (1 - dx - dy + dxdy) * __ldg(bp);
}

// Frame::prepareForStereoWith, DataStructures/Frame.cpp:295-317 (double -> float like the reference).  Host and
// device: the same IEEE operations, so k_prepare_observe produces bit-identical constants on the GPU.
LSD_HD void prepareStereoConsts(const float K[9], const double q[4], const double t[3], const double s, RefConst& rc)
{
    double qi[4] = { -q[0], -q[1], -q[2], q[3] };
    const double si = 1.0 / s;
    double nt[3] = { t[0] * -1.0, t[1] * -1.0, t[2] * -1.0 }, rt[3];
    lsd::quatRotate(qi, nt, rt);
    const double oTt[3] = { si * rt[0], si * rt[1], si * rt[2] };      // otherToThis.translation()
    double Ri[9], R[9];
    lsd::quatToMatrix(qi, Ri);
    lsd::quatToMatrix(q, R);
    float Rif[9];
    for (int i = 0; i < 9; i++) Rif[i] = (float)Ri[i];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            float kr = (K[i * 3 + 0] * Rif[0 * 3 + j] + K[i * 3 + 1] * Rif[1 * 3 + j]) + K[i * 3 + 2] * Rif[2 * 3 + j];
            rc.K_otherToThis_R[i * 3 + j] = kr * (float)si;
        }
    for (int i = 0; i < 3; i++) rc.otherToThis_t[i] = (float)oTt[i];
    for (int i = 0; i < 3; i++)
        rc.K_otherToThis_t[i] = (K[i * 3 + 0] * rc.otherToThis_t[0] + K[i * 3 + 1] * rc.otherToThis_t[1]) + K[i * 3 + 2] * rc.otherToThis_t[2];
    for (int i = 0; i < 3; i++) rc.thisToOther_t[i] = (float)t[i];
    float tR[9];
    for (int i = 0; i < 9; i++) tR[i] = (float)R[i] * (float)s;       // thisToOther_R
    for (int i = 0; i < 3; i++) { rc.row0[i] = tR[i * 3 + 0]; rc.row1[i] = tR[i * 3 + 1]; rc.row2[i] = tR[i * 3 + 2]; }
}

// Device-side tail of SE3Tracker::trackFrame (SE3Tracker.cpp:473-485) + head of DepthMap::updateKeyframe
// (DepthMap.cpp:1079-1105) for the frame that was just tracked on the active keyframe: turns the tracker's
// device-resident result into the observe parameters, so that the mapping kernels can be enqueued behind the
// tracking kernel without a host round trip.  Runs on the last thread of k_track_persistent.
struct PrepareConsts {
    float K[9];
    int frameId, reactivated, kfNumTracked, kfNumMapped, W1, H1;
    const float* image;
    const uint8_t* goodMask;
};
__device__ __forceinline__ void devicePrepareObserve(const lsd::SE3<float>& T, int diverged, float lastResidual, float pointUsage,
                                                     float goodCount, float badCount, const PrepareConsts& c,
                                                     ObserveParams* __restrict__ OP, int* __restrict__ skip)
{
    *skip = diverged;
    if (diverged) return;
    const lsd::SE3<double> f2r = lsd::se3Cast<double>(lsd::se3Inverse(T));        // SE3Tracker.cpp:483-485
    RefConst& rc = OP->refs[0];
    prepareStereoConsts(c.K, f2r.q, f2r.t, 1.0, rc);
    rc.initialTrackedResidual = lastResidual / pointUsage;                       // :482
    rc.id = c.frameId;
    rc.trackedOnActive = 1;
    rc.image = c.image;
    rc.goodMask = c.goodMask;
    const bool trackingWasGood = goodCount / (c.W1 * c.H1) > 0.04f && goodCount / (goodCount + badCount) > 0.5f;   // :475-477
    OP->nRefs = 1;
    OP->byIdOffset = c.frameId; OP->byIdSize = 1; OP->byId[0] = 0;
    OP->oldestIdx = 0; OP->newestIdx = 0;
    OP->reactivated = c.reactivated;
    OP->kfNumTracked = c.kfNumTracked + (trackingWasGood ? 1 : 0);               // :479-480
    OP->kfNumMapped = c.kfNumMapped;
}

