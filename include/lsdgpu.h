/*
 * lsdgpu.h -- C ABI of the B200-native LSD-SLAM hot path (liblsdgpu.so).
 *
 * The reference has no plugin / FFI layer: the seam is three public C++ methods (SURVEY.md 8b)
 *     SE3  SE3Tracker::trackFrame(TrackingReference*, Frame*, const SE3&)    Tracking/SE3Tracker.h:65-68
 *     void DepthMap::updateKeyframe(std::deque<std::shared_ptr<Frame>>)      DepthEstimation/DepthMap.h:58
 *     void DepthMap::createKeyFrame(Frame*)                                  DepthEstimation/DepthMap.h:63
 * plus the state-touching siblings of DepthMap and the Frame builders below them.  Every entry point
 * here names the reference interface it replaces (paths relative to lsd_slam_core/src/).  The C++
 * adapter classes in lsd_slam_b200/host/ keep the reference's method names on top of this ABI;
 * INTEGRATION.md shows the binding a maintainer adds to lsd_slam_core.
 *
 * Conventions: extern "C", POD only, caller-owned HOST buffers, opaque context, int return
 * (0 = ok, negative = error, text via lsdgpu_last_error), never throws.  One context owns one CUDA
 * stream and all device state of one SlamSystem (one tracker + one depth map); contexts are independent
 * and thread-compatible (SlamSystem runs tracking and mapping on different threads: calls into ONE
 * context must be serialised by the caller, or use two contexts' worth of locking as the adapter does).
 *
 * Poses: SE3 as double qt[7] = (qx,qy,qz,qw, tx,ty,tz) (Eigen coefficient order of Sophus::SE3d);
 *        Sim3 as double qts[8] = qt[7] + scale.
 */
#ifndef LSDGPU_H
#define LSDGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSDGPU_LEVELS 5                 /* PYRAMID_LEVELS, util/settings.h:106 */
/* 2: additive over 1 -- lsdgpu_get_globals, lsdgpu_depth_update_keyframe_refs (lsdgpu_ref_desc), lsdgpu_seq_sum_f32,
 *    lsdgpu_peer_export / _attach / _detach, lsdgpu_map_export_points (lsdgpu_map_filter, lsdgpu_map_point); contexts are
 *    thread-safe (per-context mutex).  No existing signature changed. */
#define LSDGPU_ABI_VERSION 2

typedef struct lsdgpu_ctx lsdgpu_ctx;

/* DepthMapPixelHypothesis, DepthEstimation/DepthMapPixelHypothesis.h:37-61 (sizeof == 32, same field order) */
typedef struct {
    uint8_t isValid;
    uint8_t _pad[3];
    int32_t blacklisted;
    float   nextStereoFrameMinID;
    int32_t validity_counter;
    float   idepth;
    float   idepth_var;
    float   idepth_smoothed;
    float   idepth_var_smoothed;
} lsdgpu_hyp;

/* run-time globals of util/settings.cpp:77-88 that the path reads */
typedef struct {
    float minUseGrad;                   /* 5  */
    float cameraPixelNoise2;            /* 16 */
    float depthSmoothingFactor;         /* 1  */
    int   allowNegativeIdepths;         /* 1  */
    int   useSubpixelStereo;            /* 1  */
    int   useAffineLightningEstimation; /* 1 (settings.cpp:88; cfg/LSDParams.cfg:28 sets 0 under ROS) */
} lsdgpu_globals;

/* DenseDepthTrackerSettings, util/settings.h:355-402 (the fields trackFrame reads) */
typedef struct {
    float lambdaSuccessFac, lambdaFailFac;
    float lambdaInitial[LSDGPU_LEVELS];
    float stepSizeMin[LSDGPU_LEVELS];
    float convergenceEps[LSDGPU_LEVELS];
    int   maxItsPerLvl[LSDGPU_LEVELS];
    float huber_d, var_weight;
} lsdgpu_track_settings;

/* public fields of SE3Tracker after trackFrame, Tracking/SE3Tracker.h:82-93 + the Frame side effects */
typedef struct {
    double frameToRef_qt[7];            /* return value of trackFrame (identity when diverged) */
    float  pointUsage, lastGoodCount, lastBadCount, lastMeanRes, lastResidual;
    float  affineEstimation_a, affineEstimation_b;
    int    diverged, trackingWasGood;
    int    numCalcResidualCalls[LSDGPU_LEVELS];
    int    numCalcWarpUpdateCalls[LSDGPU_LEVELS];
    float  initialTrackedResidual;      /* frame->initialTrackedResidual, SE3Tracker.cpp:482 */
} lsdgpu_track_result;

/* one fused evaluation = calcResidualAndBuffers + calcWeightsAndResidual + calculateWarpUpdate
 * (SE3Tracker.cpp:885-1029, 749-790, 1258-1299 + LGS6, LGSX.h:184-402) at a given pose */
typedef struct {
    float A[36];                        /* row-major, normalised by num_constraints like LGS6::finish */
    float b[6];
    float lsError;
    float meanWeightedRes;              /* calcWeightsAndResidual return value */
    float meanUnweightedRes;            /* calcResidualAndBuffers return value */
    int   warpedSize;                   /* buf_warped_size */
    float pointUsage, goodCount, badCount, meanRes;
    float affine_a_lastIt, affine_b_lastIt;
    float sxx, syy, sx, sy, sw;
} lsdgpu_eval_result;

/* what lsdgpu_frame_download can fetch (parity hooks for the Frame builders) */
enum {
    LSDGPU_BUF_IMAGE = 0,               /* Frame::image(level),        float  w_l*h_l            */
    LSDGPU_BUF_GRADIENTS = 1,           /* Frame::gradients(level),    float4 w_l*h_l (dx,dy,I,0) */
    LSDGPU_BUF_MAXGRAD = 2,             /* Frame::maxGradients(0),     float  w*h  (level 0 only) */
    LSDGPU_BUF_IDEPTH = 3,              /* Frame::idepth(level)                                   */
    LSDGPU_BUF_IDEPTH_VAR = 4,          /* Frame::idepthVar(level)                                */
    LSDGPU_BUF_GOODMASK = 5             /* Frame::refPixelWasGood(), uint8 w_1*h_1                */
};

/* ---- context ------------------------------------------------------------------------------------ */
/* replaces SE3Tracker::SE3Tracker(w,h,K) Tracking/SE3Tracker.cpp:46-94 and DepthMap::DepthMap(w,h,K)
 * DepthEstimation/DepthMap.cpp:41-83.  max_frames = number of frame slots resident in HBM. */
int  lsdgpu_create(int device, int width, int height, const float K[9], int max_frames, lsdgpu_ctx** out);
void lsdgpu_destroy(lsdgpu_ctx* ctx);
const char* lsdgpu_last_error(const lsdgpu_ctx* ctx);
int  lsdgpu_abi_version(void);
int  lsdgpu_set_globals(lsdgpu_ctx* ctx, const lsdgpu_globals* g);      /* util/settings.cpp:77-88 */
int  lsdgpu_get_globals(const lsdgpu_ctx* ctx, lsdgpu_globals* g);      /* the values in force (the reference reads the globals directly) */
void lsdgpu_default_globals(lsdgpu_globals* g);
void lsdgpu_default_track_settings(lsdgpu_track_settings* s);            /* util/settings.h:358-386 */
int  lsdgpu_synchronize(lsdgpu_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches claim) */
long long lsdgpu_launch_count(const lsdgpu_ctx* ctx);
/* CUDA-event timers on the context's stream (bench.py: roofline / per-stage times) */
int  lsdgpu_timer_begin(lsdgpu_ctx* ctx, int slot);
int  lsdgpu_timer_end(lsdgpu_ctx* ctx, int slot);
int  lsdgpu_timer_elapsed_ms(lsdgpu_ctx* ctx, int slot, float* ms);      /* synchronises on the end event */
/* accumulated device time (ms) and launch count of the warp/residual kernel since the last reset */
int  lsdgpu_track_kernel_stats(lsdgpu_ctx* ctx, int reset, double* ms, long long* launches, double* algorithmic_bytes);

/* ---- Frame: DataStructures/Frame.{h,cpp} -------------------------------------------------------- */
/* Frame::Frame(id,w,h,K,ts,const uchar*) Frame.cpp:35-54 + buildImage :491-630 + buildGradients :643-680
 * + buildMaxGradients :690-767, all levels, once per frame.  gray = HOST buffer of w*h bytes. */
int lsdgpu_frame_upload_u8(lsdgpu_ctx* ctx, int frame_id, const uint8_t* gray);
int lsdgpu_frame_release(lsdgpu_ctx* ctx, int frame_id);                 /* Frame::~Frame */
/* Prefetch ring: raw u8 frames parked in HBM ahead of time (camera DMA / dataset prefetch), so that the
 * Frame constructor above can run without touching the host: stage_put copies one HOST frame into ring
 * entry `index`; frame_from_stage builds frame `frame_id` from it (same kernels as lsdgpu_frame_upload_u8). */
int lsdgpu_stage_reserve(lsdgpu_ctx* ctx, int n_entries);
int lsdgpu_stage_put(lsdgpu_ctx* ctx, int index, const uint8_t* gray);
int lsdgpu_frame_from_stage(lsdgpu_ctx* ctx, int frame_id, int index);
int lsdgpu_frame_download(lsdgpu_ctx* ctx, int frame_id, int what, int level, void* out_host);
/* Frame::setDepthFromGroundTruth(depth, cov_scale) Frame.cpp:245-293 */
int lsdgpu_frame_set_depth_gt(lsdgpu_ctx* ctx, int frame_id, const float* depth, float cov_scale);
/* raw level-0 idepth / idepthVar import (Frame::setDepth output of a host-side DepthMap) */
int lsdgpu_frame_set_idepth(lsdgpu_ctx* ctx, int frame_id, const float* idepth, const float* idepthVar);
/* FramePoseStruct::thisToParent_raw / trackingParent + Frame::initialTrackedResidual (written by
 * lsdgpu_se3_track; the setter lets a host pose-graph override them) */
int lsdgpu_frame_set_pose(lsdgpu_ctx* ctx, int frame_id, const double thisToParent_qts[8], int parent_id, float initialTrackedResidual);
int lsdgpu_frame_get_pose(lsdgpu_ctx* ctx, int frame_id, double thisToParent_qts[8], int* parent_id, float* initialTrackedResidual);
/* Frame::numFramesTrackedOnThis / numMappedOnThis (DepthMap.cpp:454, SE3Tracker.cpp:480) */
int lsdgpu_frame_get_counters(lsdgpu_ctx* ctx, int frame_id, int* numFramesTrackedOnThis, int* numMappedOnThis);
int lsdgpu_frame_set_counters(lsdgpu_ctx* ctx, int frame_id, int numFramesTrackedOnThis, int numMappedOnThis);
/* Frame::meanIdepth / numPoints / depthHasBeenUpdatedFlag (Frame.cpp:234-242) */
int lsdgpu_frame_get_depth_stats(lsdgpu_ctx* ctx, int frame_id, float* meanIdepth, int* numPoints, int* depthHasBeenUpdatedFlag);
/* Frame::clear_refPixelWasGood (SlamSystem.cpp:573) */
int lsdgpu_frame_clear_good_mask(lsdgpu_ctx* ctx, int frame_id);

/* ---- Tracking: Tracking/TrackingReference.cpp + Tracking/SE3Tracker.cpp -------------------------- */
/* TrackingReference::importFrame :71-87 (+ the depthHasBeenUpdatedFlag=false of SlamSystem.cpp:907-912):
 * (re)builds the keyframe's idepth pyramids (Frame::buildIDepthAndIDepthVar, Frame.cpp:775-877) that
 * makePointCloud :96-147 reads; the point cloud itself is never materialised on the device. */
int lsdgpu_ref_import(lsdgpu_ctx* ctx, int kf_id);
/* single fused evaluation at `level` for pose refToFrame (float qt[7]); parity hook for hot loops A+B+C */
int lsdgpu_se3_eval(lsdgpu_ctx* ctx, int kf_id, int frame_id, int level, const float refToFrame_qt[7],
                    float affine_a, float affine_b, const lsdgpu_track_settings* s, int write_good_mask,
                    lsdgpu_eval_result* out);
/* SE3Tracker::trackFrame :280-486.  Whole coarse-to-fine LM loop; mode 0 = host-driven LM (one kernel
 * per evaluation, 6x6 solve on the host), mode 1 = device-resident LM (one persistent kernel per frame). */
int lsdgpu_se3_track(lsdgpu_ctx* ctx, int kf_id, int frame_id, const double frameToRef_init_qt[7],
                     const lsdgpu_track_settings* s, int mode, lsdgpu_track_result* out);

/* One frame of the sequential (dataset_slam _hz:=0) loop in a single call -- the order of SlamSystem::trackFrame
 * (SlamSystem.cpp:890-1040) followed by SlamSystem::doMappingIteration (:739-828):
 *   Frame construction (from HOST `gray`, or from prefetch-ring entry `stage_index` when gray == NULL),
 *   lsdgpu_ref_import if the keyframe's depth changed, lsdgpu_se3_track, then
 *   keyframe_change == 0: lsdgpu_depth_update_keyframe({frame_id}) + clear_good_mask        (:571-573)
 *   keyframe_change != 0: lsdgpu_depth_finalize_keyframe + lsdgpu_depth_create_keyframe     (:400, :473)
 * Exactly equivalent to issuing those calls one by one; exists so that a host loop pays one FFI crossing per frame. */
int lsdgpu_track_and_map(lsdgpu_ctx* ctx, int kf_id, int frame_id, const uint8_t* gray, int stage_index,
                         const double frameToRef_init_qt[7], const lsdgpu_track_settings* s, int mode,
                         int keyframe_change, lsdgpu_track_result* out, double new_kf_thisToParent_qts[8]);

/* ---- input staging: UndistorterPTAM fused into the Frame construction (SURVEY 8f row 3) ----------------------------
 * UndistorterPTAM::UndistorterPTAM, util/Undistorter.cpp:171-317, with the four lines of the calibration file already parsed:
 * input_calibration = fx fy cx cy dist (relative to the input size); output_calibration[0] = -1 for "crop", -2 for "full",
 * otherwise fx fy cx cy 0 (relative to the output size).  Host-only (no context needed): fills the two remap tables
 * (out_width*out_height floats each, may be NULL) and K_out (row-major, the matrix main_on_images.cpp:164-169 hands to
 * SlamSystem).  Returns 0 = tables valid, 1 = undistort() passes the image through (:370-375), -2 = invalid arguments.
 * UndistorterOpenCV (:449-567) delegates to cv::initUndistortRectifyMap / cv::remap and stays on the host. */
int lsdgpu_undistorter_ptam_prepare(const float input_calibration[5], int in_width, int in_height, const float output_calibration[5],
                                    int out_width, int out_height, float* remapX, float* remapY, float K_out[9]);
/* host-only check of a pair of remap tables: every entry is either "no source" (x < 0, as Undistorter.cpp:312-316 writes it)
 * or a position whose four bilinear taps lie inside the in_width x in_height image (0 <= x < in_width-1, 0 <= y < in_height-1).
 * Returns 0 if valid, otherwise 1 + the index of the first offending entry (-2 for bad arguments). */
int lsdgpu_undistorter_validate_tables(int in_width, int in_height, int out_width, int out_height, const float* remapX, const float* remapY);
/* install remap tables (host pointers, w*h floats each; w, h = the context's size) for raw images of in_width x in_height;
 * NULL tables = pass-through (then in_width/in_height must equal the context's size).  Tables that fail
 * lsdgpu_undistorter_validate_tables are rejected (the gather kernel does no bounds checks of its own). */
int lsdgpu_set_undistorter(lsdgpu_ctx* ctx, int in_width, int in_height, const float* remapX, const float* remapY);
/* UndistorterPTAM::undistort, util/Undistorter.cpp:355-411: raw (in_width*in_height) -> out (w*h), 8 bit */
int lsdgpu_undistort_u8(lsdgpu_ctx* ctx, const uint8_t* raw, uint8_t* out);
/* undistort + Frame::Frame(id, w, h, K, ts, const uchar*) + buildImage/buildGradients/buildMaxGradients of all levels:
 * the raw image is copied to the device once and the remap feeds the pyramid kernel directly
 * (main_on_images.cpp:238-244: undistorter->undistort(imageDist, image); system->trackFrame(image.data, ...)) */
int lsdgpu_frame_upload_distorted_u8(lsdgpu_ctx* ctx, int frame_id, const uint8_t* raw);

/* ---- keyframe output formats, packed on the device (SURVEY 8f row 4) ----------------------------------------------
 * InputPointDense, IOWrapper/ROS/ROSOutput3DWrapper.h:34-39 = one record of keyframeMsg.pointcloud (lsd_slam_viewer/msg/keyframeMsg.msg:20-22) */
typedef struct { float idepth; float idepth_var; unsigned char color[4]; } lsdgpu_input_point_dense;
/* the packing loop of ROSOutput3DWrapper::publishKeyframe (ROSOutput3DWrapper.cpp:91-110) for level `publish_level`:
 * out receives (w >> level) * (h >> level) records, one device-to-host copy in wire layout */
int lsdgpu_keyframe_pack_pointcloud(lsdgpu_ctx* ctx, int kf_id, int publish_level, lsdgpu_input_point_dense* out);
/* The map as lsd_slam_viewer saves it (pc.ply), for many resident keyframes in one call: the point filter and world-frame transform
 * of KeyFrameDisplay::flushPC (lsd_slam_viewer/src/KeyFrameDisplay.cpp:269-340) applied to what lsdgpu_keyframe_pack_pointcloud
 * would publish for each keyframe (idepth, idepthVar and image of `publish_level`).  camToWorld_qts[8*i..] = the caller's
 * getScaledCamToWorld() of kf_ids[i] (unit quaternion x,y,z,w, translation, scale), cast to the float Sophus storage as
 * ROSOutput3DWrapper.cpp:85 does.  Records follow kf_ids order, then y, then x; counts_out[i] = points of keyframe i.
 * out == NULL: counts only.  Errors (nothing written): unknown id, a keyframe without depth, bad level, total > capacity.
 * sparsifyFactor > 1 (a rand() draw per pixel) is not offered; keyframe selection (cutFirstNKf) is the caller's list. */
/* the point filter of lsd_slam_viewer's KeyFrameDisplay::flushPC (KeyFrameDisplay.cpp:274-307); viewer defaults
 * settings.cpp:36-38 = (1, 1, 5), under ROS cfg/LSDSLAMViewerParams.cfg:20-22 = (10^-3, 10^-1, 7) */
typedef struct { float scaledDepthVarTH, absDepthVarTH; int minNearSupport; } lsdgpu_map_filter;
/* one vertex record of pc.ply (KeyFrameDisplay.cpp:328-333, header KeyFrameGraphDisplay.cpp:75-82) */
typedef struct { float x, y, z, intensity; } lsdgpu_map_point;
int lsdgpu_map_export_points(lsdgpu_ctx* ctx, int n_kf, const int* kf_ids, const double* camToWorld_qts /* 8*n_kf */,
                             int publish_level, const lsdgpu_map_filter* f,
                             lsdgpu_map_point* out /* NULL: counts only */, long long capacity,
                             int* counts_out /* n_kf, may be NULL */, long long* total_out);
/* Frame::takeReActivationData(currentDepthMap), DataStructures/Frame.cpp:107-145: snapshot of the ACTIVE depth map into the
 * keyframe's idepth_reAct / idepthVar_reAct / validity_reAct -- kept on the device.  lsdgpu_depth_finalize_keyframe calls it
 * (DepthMap.cpp:1387); exposed for re-activation bookkeeping outside finalize. */
int lsdgpu_frame_take_reactivation_data(lsdgpu_ctx* ctx, int kf_id);
/* copies of the three reactivation arrays (w*h each), for host consumers and the parity tests; any pointer may be NULL */
int lsdgpu_frame_download_reactivation_data(lsdgpu_ctx* ctx, int kf_id, float* idepth_reAct, float* idepthVar_reAct, uint8_t* validity_reAct);
/* DepthMap::setFromExistingKF(kf), DepthEstimation/DepthMap.cpp:920-962, from the keyframe's device-resident reactivation data */
int lsdgpu_depth_set_from_existing_kf(lsdgpu_ctx* ctx, int kf_id);

/* ---- Sim3Tracker, batched (SURVEY 8f row 1) --------------------------------------------------------------------
 * Sim3 values cross the ABI as qts[8] = unit quaternion (x,y,z,w), translation, scale (like new_kf_thisToParent_qts).
 * Everything SlamSystem::tryTrackSim3 (SlamSystem.cpp:1043-1127) reads from the tracker, Tracking/Sim3Tracker.h:66,127-138. */
typedef struct {
    double frameToRef_qts[8];          /* identity (Sim3()) on the early returns, Sim3Tracker.cpp:184-187, 212-217, 231-235, 363-367 */
    float  lastSim3Hessian[49];        /* ls7.A row-major, NOT divided by num_constraints (:360); zero on the early returns */
    float  lastResidual, lastDepthResidual, lastPhotometricResidual;
    float  pointUsage;
    float  affineEstimation_a, affineEstimation_b;
    int    diverged;
    int    numCalcResidualCalls[LSDGPU_LEVELS];
    int    numCalcWarpUpdateCalls[LSDGPU_LEVELS];
} lsdgpu_sim3_result;
/* one fused evaluation (calcSim3Buffers :414-607 + calcSim3WeightsAndResidual :748-856 + calcSim3LGS :992-1047): parity hook */
typedef struct {
    float A[49], b[7];                 /* LGS7 (LGSX.h:411-443), undivided */
    int   num_constraints;
    float sumResD, sumResP; int numTermsD, numTermsP;
    float mean, meanD, meanP;
    int   warpedSize;
    float pointUsage, affine_a_lastIt, affine_b_lastIt;
} lsdgpu_sim3_eval_result;
int lsdgpu_sim3_eval(lsdgpu_ctx* ctx, int ref_kf_id, int frame_id, int level, const double refToFrame_qts[8],
                     float affine_a, float affine_b, const lsdgpu_track_settings* s, lsdgpu_sim3_eval_result* out);
/* Sim3Tracker::trackFrameSim3(reference, frame, frameToReference_initialEstimate, startLevel, finalLevel) :149-382.
 * Both frames must carry depth (keyframes).  s == NULL: DenseDepthTrackerSettings defaults (util/settings.h:355-386). */
int lsdgpu_sim3_track(lsdgpu_ctx* ctx, int ref_kf_id, int frame_id, const double frameToRef_init_qts[8],
                      int start_level, int final_level, const lsdgpu_track_settings* s, lsdgpu_sim3_result* out);
/* n independent trackings in ONE launch (one thread-block cluster per problem): problem i tracks frame frame_ids[i] on
 * reference keyframe ref_kf_ids[i] from frameToRef_init_qts[8*i..]; n <= 1024. */
int lsdgpu_sim3_track_batch(lsdgpu_ctx* ctx, int n, const int* ref_kf_ids, const int* frame_ids, const double* frameToRef_init_qts,
                            int start_level, int final_level, const lsdgpu_track_settings* s, lsdgpu_sim3_result* results);

/* ---- permaRef tracking, batched (SURVEY 8f row 2) ------------------------------------------------------------
 * Frame::setPermaRef Frame.cpp:149-174: freeze the keyframe's CURRENT level-4 point cloud (positions, colour, variance). */
int lsdgpu_frame_set_perma_ref(lsdgpu_ctx* ctx, int kf_id, int* num_points_out);
/* SE3Tracker::checkPermaRefOverlap SE3Tracker.cpp:121-157 for n candidates in one launch:
 * usage_out[i] = pointUsage of keyframe kf_ids[i] under referenceToFrame refToFrame_qt[7*i..] */
int lsdgpu_perma_overlap_batch(lsdgpu_ctx* ctx, int n, const int* kf_ids, const double* refToFrame_qt, float* usage_out);
/* SE3Tracker::trackFrameOnPermaref SE3Tracker.cpp:162-272 for n candidate keyframes against ONE frame in one launch
 * (one CTA per candidate; TestTrack settings util/settings.h:379-382: 5 iterations, eps 0.98, step-min 1e-3).
 * results[i].frameToRef_qt holds referenceToFrame (the reference returns it un-inverted, :271). */
int lsdgpu_perma_track_batch(lsdgpu_ctx* ctx, int n, const int* kf_ids, int frame_id, const double* refToFrame_init_qt,
                             lsdgpu_track_result* results);

/* ---- one stream over several GPUs (BASELINE.json config 5) ------------------------------------------------------------------
 * The device-resident tracker (lsdgpu_se3_track, mode 1) can split the points of every level over n_ranks GPUs, one process per
 * GPU.  Every rank holds the same frames and the same depth map (all ranks issue the same calls); rank r evaluates every
 * n_ranks-th 32-pixel chunk, and the 40..56 sums of each pass as well as the level-1 refPixelWasGood flags cross NVLink INSIDE
 * the kernel through peer-mapped memory (posted stores + polling of tagged 8-byte slots; no host round trip, no NCCL call on the
 * path), added in rank order on every GPU, so every rank takes identical LM decisions and returns identical results.
 *   lsdgpu_peer_export  CUDA IPC handle (LSDGPU_PEER_HANDLE_BYTES) of this context's arena; the caller gathers the handles of
 *                       all ranks (e.g. torch.distributed.all_gather)
 *   lsdgpu_peer_attach  handles = n_ranks * LSDGPU_PEER_HANDLE_BYTES bytes in rank order; maps the peers and switches the
 *                       tracker to sharded operation.  All contexts must have been created with the same size and max_frames
 *                       (same arena layout).  Synchronise the ranks after attach and before the first tracking.
 *   lsdgpu_peer_detach  back to single-GPU operation (also done by lsdgpu_destroy); synchronise the ranks first. */
#define LSDGPU_PEER_HANDLE_BYTES 64
int lsdgpu_peer_export(lsdgpu_ctx* ctx, void* handle_out);
int lsdgpu_peer_attach(lsdgpu_ctx* ctx, int rank, int n_ranks, const void* handles);
int lsdgpu_peer_detach(lsdgpu_ctx* ctx);

/* Point-sharded tracking across GPUs (SURVEY 8e, BASELINE config 5): rank `shard` of `n_shards` evaluates every
 * n_shards-th 32-pixel chunk of the level; the LSDGPU_EVAL_NSUMS partial sums of every evaluation are handed to
 * `allreduce` (sum over ranks, in place, HOST buffer) before the LM decision, so all ranks take identical
 * decisions.  Same host-driven LM loop as mode 0.  The refPixelWasGood mask is only written for the rank's own
 * chunks (the depth map is not sharded: "replicas only"). */
#define LSDGPU_EVAL_NSUMS 40
typedef void (*lsdgpu_allreduce_fn)(void* user, float* sums, int n);
int lsdgpu_se3_track_sharded(lsdgpu_ctx* ctx, int kf_id, int frame_id, const double frameToRef_init_qt[7],
                             const lsdgpu_track_settings* s, int shard, int n_shards,
                             lsdgpu_allreduce_fn allreduce, void* user, lsdgpu_track_result* out);

/* ---- DepthMap: DepthEstimation/DepthMap.cpp ------------------------------------------------------ */
int lsdgpu_depth_reset(lsdgpu_ctx* ctx);                                  /* DepthMap::reset :102-108 */
int lsdgpu_depth_is_valid(lsdgpu_ctx* ctx);                               /* DepthMap::isValid, DepthMap.h:71 */
int lsdgpu_depth_invalidate(lsdgpu_ctx* ctx);                             /* DepthMap::invalidate :1215-1220 */
int lsdgpu_depth_init_from_gt(lsdgpu_ctx* ctx, int kf_id);                /* initializeFromGTDepth :965-1018 */
/* initializeRandomly :883-916 (host draws rand()) and setFromExistingKF :920-962 both reduce to
 * "load these hypotheses for keyframe kf_id"; reactivated != 0 also runs the regularizeDepthMap(false,24)
 * of :961 and sets activeKeyFrameIsReactivated.  do_set_depth mirrors the trailing setDepth of :915. */
int lsdgpu_depth_set_hypotheses(lsdgpu_ctx* ctx, int kf_id, const lsdgpu_hyp* aos, int reactivated, int do_set_depth);
/* DepthMap::updateKeyframe(referenceFrames) :1072-1213; ref_ids oldest first, all tracked on the active KF */
int lsdgpu_depth_update_keyframe(lsdgpu_ctx* ctx, const int* ref_ids, int n_refs);
/* The same with the reference-frame set-up of :1085-1101 spelled out.  DepthMap::updateKeyframe accepts frames that were tracked
 * on ANOTHER keyframe (the frames still queued in unmappedTrackedFrames when the keyframe changes, SlamSystem.cpp:559-575):
 *   refToKf = frame->pose->trackingParent == activeKeyFrame ? frame->pose->thisToParent_raw                           (:1096-1097)
 *           : activeKeyFrame->getScaledCamToWorld().inverse() * frame->getScaledCamToWorld()                          (:1098-1099)
 * and such frames do not apply their tracking mask (the `refFrame->getTrackingParent() == activeKeyFrame` gate of :245 / :322).
 * The absolute poses belong to the caller's pose graph (FramePoseStruct::getCamToWorld, KeyFrameGraph), so the caller passes the
 * product; tracked_on_kf != 0 uses the pose stored by the tracker and ignores refToKf_qts. */
typedef struct lsdgpu_ref_desc {
    int32_t frame_id;
    int32_t tracked_on_kf;          /* frame->getTrackingParent() == activeKeyFrame */
    double  refToKf_qts[8];         /* unit quaternion x,y,z,w, translation, scale; read when tracked_on_kf == 0 */
} lsdgpu_ref_desc;
int lsdgpu_depth_update_keyframe_refs(lsdgpu_ctx* ctx, const lsdgpu_ref_desc* refs, int n_refs);
/* DepthMap::createKeyFrame(new_keyframe) :1222-1327; writes the rescaled thisToParent_raw of the new KF */
int lsdgpu_depth_create_keyframe(lsdgpu_ctx* ctx, int new_kf_id, double new_thisToParent_qts[8]);
int lsdgpu_depth_finalize_keyframe(lsdgpu_ctx* ctx);                      /* finalizeKeyFrame :1363-1395 */
/* The `float sumIdepth` loop of createKeyFrame (:1286-1293) on host data: sum of x[i] over valid[i] != 0 (valid == NULL: all) in
 * index order with fp32 round-to-nearest after EVERY addition -- computed by the parallel kernels createKeyFrame itself uses
 * (csrc/seqsum.cuh), bit-identical to the sequential loop for any input.  A parity hook: it lets the tests feed ties, binade
 * crossings, negative and non-finite terms. */
int lsdgpu_seq_sum_f32(lsdgpu_ctx* ctx, const float* x, const unsigned char* valid, int n, float* sum, int* count);
int lsdgpu_depth_active_keyframe(lsdgpu_ctx* ctx);                        /* id or -1 */
/* currentDepthMap in the reference's 32-byte AoS layout (Frame::setDepth / takeReActivationData input) */
int lsdgpu_depth_download(lsdgpu_ctx* ctx, lsdgpu_hyp* aos_out);
int lsdgpu_depth_download_integral(lsdgpu_ctx* ctx, int32_t* out);        /* validityIntegralBuffer */
/* individual passes (per-kernel parity hooks; same order of operations as the drivers above) */
int lsdgpu_depth_observe(lsdgpu_ctx* ctx, const int* ref_ids, int n_refs);            /* observeDepth :147-178 */
int lsdgpu_depth_regularize_fill_holes(lsdgpu_ctx* ctx);                              /* :706-718 */
int lsdgpu_depth_regularize(lsdgpu_ctx* ctx, int removeOcclusions, int validityTH);   /* :853-880 */
int lsdgpu_depth_propagate(lsdgpu_ctx* ctx, int new_kf_id);                           /* :475-653 */

#ifdef __cplusplus
}
#endif
#endif
