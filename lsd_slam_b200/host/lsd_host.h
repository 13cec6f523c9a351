// lsd_host.h -- C++ host side of the B200 hot path: classes that keep the reference's names, call signatures and
// observable fields for the three seam methods, implemented on top of the C ABI (include/lsdgpu.h).
//
//   lsd_slam::SE3Tracker::trackFrame          Tracking/SE3Tracker.h:65-68
//   lsd_slam::DepthMap::updateKeyframe        DepthEstimation/DepthMap.h:58
//   lsd_slam::DepthMap::createKeyFrame        DepthEstimation/DepthMap.h:63
//
// The reference's headers need Eigen / Sophus / Boost / OpenCV, none of which exist in this image, so this
// header carries minimal stand-ins (lsd_slam::SE3, Sim3, Matrix3f) with the same semantics; inside
// lsd_slam_core the adapter in INTEGRATION.md maps them 1:1 onto Sophus::SE3d / Sophus::Sim3d / Eigen::Matrix3f.
// Host code only: no CUDA headers, no torch.  Everything device-side sits behind lsdgpu_* calls.
#pragma once

#include <deque>
#include <memory>
#include <ostream>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/lsdgpu.h"

namespace lsd_slam {

struct Matrix3f {
    float m[9];                                      // row-major
    float operator()(int r, int c) const { return m[r * 3 + c]; }
};

// Sophus::SE3d stand-in: unit quaternion (x,y,z,w) + translation
struct SE3 {
    double q[4] = { 0, 0, 0, 1 };
    double t[3] = { 0, 0, 0 };
    SE3 inverse() const;
    SE3 operator*(const SE3& o) const;
};
// Sophus::Sim3d stand-in
struct Sim3 {
    double q[4] = { 0, 0, 0, 1 };
    double t[3] = { 0, 0, 0 };
    double s = 1.0;
    Sim3 inverse() const;                            // thirdparty/Sophus/sophus/sim3.hpp:169-173
    Sim3 operator*(const Sim3& o) const;             // sim3.hpp:257-260
};
inline Sim3 sim3FromSE3(const SE3& se3, double scale)     // util/SophusUtil.h:53-58
{
    Sim3 r;
    for (int i = 0; i < 4; i++) r.q[i] = se3.q[i];
    for (int i = 0; i < 3; i++) r.t[i] = se3.t[i];
    r.s = scale;
    return r;
}
inline SE3 se3FromSim3(const Sim3& sim3)                  // util/SophusUtil.h:60-63
{
    SE3 r;
    for (int i = 0; i < 4; i++) r.q[i] = sim3.q[i];
    for (int i = 0; i < 3; i++) r.t[i] = sim3.t[i];
    return r;
}

class LsdGpuError : public std::runtime_error {
public:
    explicit LsdGpuError(const std::string& what) : std::runtime_error(what) {}
};

// One device context per SlamSystem (SlamSystem owns one SE3Tracker + one DepthMap, SlamSystem.h:126,131)
class DeviceContext {
public:
    DeviceContext(int device, int w, int h, const Matrix3f& K, int maxFrames = 16);
    ~DeviceContext();
    DeviceContext(const DeviceContext&) = delete;
    DeviceContext& operator=(const DeviceContext&) = delete;
    lsdgpu_ctx* raw() const { return ctx_; }
    void check(int rc, const char* where) const;
    int width() const { return w_; }
    int height() const { return h_; }

private:
    lsdgpu_ctx* ctx_ = nullptr;
    int w_, h_;
};

// FramePoseStruct, DataStructures/FramePoseStruct.h (the two members the path touches)
struct FramePoseStruct {
    Sim3 thisToParent_raw;
    FramePoseStruct* trackingParent = nullptr;
    int frameID = -1;
    // FramePoseStruct.cpp:84-105 without the pose-graph members (isOptimized / the cache belong to KeyFrameGraph, out of scope):
    // identity for the first frame, otherwise the parent's absolute pose times thisToParent_raw
    Sim3 getCamToWorld(int recursionDepth = 0) const;
};

// DataStructures/Frame.h -- device-resident frame; host keeps the bookkeeping the callers read
class Frame {
public:
    // `distorted` = true: `image` is the RAW camera image of the installed UndistorterPTAM's input size; undistortion is
    // fused into the pyramid construction on the device (replaces undistort() + this constructor, main_on_images.cpp:238-244)
    Frame(DeviceContext& dev, int id, int width, int height, const Matrix3f& K, double timestamp, const unsigned char* image,
          bool distorted = false);
    ~Frame();
    Frame(const Frame&) = delete;
    int id() const { return id_; }
    int width(int level = 0) const { return w_ >> level; }
    int height(int level = 0) const { return h_ >> level; }
    double timestamp() const { return timestamp_; }
    void setDepthFromGroundTruth(const float* depth, float cov_scale = 1.0f);      // Frame.cpp:245-293
    bool hasTrackingParent() const { return pose->trackingParent != nullptr; }
    Sim3 getScaledCamToWorld() const { return pose->getCamToWorld(); }              // Frame.h:276-280
    void clear_refPixelWasGood();                                                   // Frame.h:439
    float meanIdepth();                                                             // Frame.cpp:234 (lazy D2H)
    int numPoints();
    bool depthHasBeenUpdatedFlag() const;
    // buffers for callers that still need host copies (e.g. Output3DWrapper): explicit downloads
    void downloadIdepth(int level, std::vector<float>& idepth, std::vector<float>& idepthVar);
    void downloadRefPixelWasGood(std::vector<unsigned char>& mask);

    FramePoseStruct* pose;
    float initialTrackedResidual = 0;
    int numFramesTrackedOnThis = 0, numMappedOnThis = 0, numMappedOnThisTotal = 0;

    DeviceContext& dev() const { return dev_; }

private:
    DeviceContext& dev_;
    int id_, w_, h_;
    double timestamp_;
};

// Tracking/TrackingReference.h
class TrackingReference {
public:
    Frame* keyframe = nullptr;
    int frameID = -1;
    void importFrame(Frame* sourceKF);                                              // TrackingReference.cpp:71-87
    void invalidate() { keyframe = nullptr; }
};

// util/settings.h:355-402
struct DenseDepthTrackerSettings : lsdgpu_track_settings {
    DenseDepthTrackerSettings() { lsdgpu_default_track_settings(this); }
};

// Tracking/SE3Tracker.h
class SE3Tracker {
public:
    SE3Tracker(DeviceContext& dev, int w, int h, const Matrix3f& K);
    SE3Tracker(const SE3Tracker&) = delete;

    SE3 trackFrame(TrackingReference* reference, Frame* frame, const SE3& frameToReference_initialEstimate);

    DenseDepthTrackerSettings settings;
    float pointUsage = 0, lastGoodCount = 0, lastMeanRes = 0, lastBadCount = 0, lastResidual = 0;
    float affineEstimation_a = 1, affineEstimation_b = 0;
    bool diverged = false, trackingWasGood = false;
    int mode = 1;                 // 1: device-resident LM (one kernel per frame); 0: host-driven LM

private:
    DeviceContext& dev_;
    int width_, height_;
};

// Tracking/Sim3Tracker.h:59-160 (SURVEY 8f row 1)
struct Matrix7x7 {
    float m[49];                                     // row-major
    float operator()(int r, int c) const { return m[r * 7 + c]; }
    void setZero() { for (float& v : m) v = 0.f; }
};
class Sim3Tracker {
public:
    Sim3Tracker(DeviceContext& dev, int w, int h, const Matrix3f& K);
    Sim3Tracker(const Sim3Tracker&) = delete;

    Sim3 trackFrameSim3(TrackingReference* reference, Frame* frame, const Sim3& frameToReference_initialEstimate,
                        int startLevel, int finalLevel);
    // n independent (reference, frame) pairs in one launch; members below then describe the LAST problem,
    // results[] all of them (SlamSystem::tryTrackSim3 runs two per candidate, SlamSystem.cpp:1043-1127)
    void trackFrameSim3Batch(const std::vector<TrackingReference*>& references, const std::vector<Frame*>& frames,
                             const std::vector<Sim3>& frameToReference_initialEstimates, int startLevel, int finalLevel,
                             std::vector<Sim3>& frameToReference, std::vector<lsdgpu_sim3_result>& results);

    DenseDepthTrackerSettings settings;
    Matrix7x7 lastSim3Hessian;
    float pointUsage = 0;
    float lastResidual = 0, lastDepthResidual = 0, lastPhotometricResidual = 0;
    float affineEstimation_a = 1, affineEstimation_b = 0;
    bool diverged = false;

private:
    Sim3 take(const lsdgpu_sim3_result& r);
    DeviceContext& dev_;
    int width_, height_;
};

// util/Undistorter.h:96-160 (SURVEY 8f row 3).  The ATAN/PTAM calibration file has four lines:
//   fx fy cx cy dist   |   in_width in_height   |   "crop" / "full" / "none" / fx fy cx cy 0   |   out_width out_height
// An OpenCV-model file (8 numbers on the first line, Undistorter.cpp:70-79) is rejected: that model stays on the host.
class UndistorterPTAM {
public:
    explicit UndistorterPTAM(const char* configFileName);
    // undistort a raw 8-bit image (in_width x in_height) on the device of `dev`, whose size must be the output size
    void undistort(DeviceContext& dev, const unsigned char* image, unsigned char* result) const;
    // install the tables so that Frame(dev, id, w, h, K, ts, rawImage, /*distorted=*/true) feeds raw images to the device
    void install(DeviceContext& dev) const;
    const Matrix3f& getK() const { return K_; }
    int getOutputWidth() const { return out_width; }
    int getOutputHeight() const { return out_height; }
    int getInputWidth() const { return in_width; }
    int getInputHeight() const { return in_height; }
    bool isValid() const { return valid; }
    bool isPassThrough() const { return passThrough; }
    const std::vector<float>& remapTableX() const { return remapX; }
    const std::vector<float>& remapTableY() const { return remapY; }

private:
    Matrix3f K_;
    float inputCalibration[5], outputCalibration[5];
    int out_width = 0, out_height = 0, in_width = 0, in_height = 0;
    std::vector<float> remapX, remapY;
    bool valid = false, passThrough = false;
};

// DepthEstimation/DepthMap.h
class DepthMap {
public:
    DepthMap(DeviceContext& dev, int w, int h, const Matrix3f& K);
    DepthMap(const DepthMap&) = delete;

    void reset();
    void updateKeyframe(std::deque<std::shared_ptr<Frame>> referenceFrames);
    void createKeyFrame(Frame* new_keyframe);
    void finalizeKeyFrame();
    void invalidate();
    bool isValid() const { return activeKeyFrame != nullptr; }
    void initializeFromGTDepth(Frame* new_frame);
    void initializeRandomly(Frame* new_frame);
    void setFromExistingKF(Frame* kf, const float* idepth_reAct, const float* idepthVar_reAct, const unsigned char* validity_reAct);
    // currentDepthMap in the reference's AoS layout (w*h records)
    void download(std::vector<lsdgpu_hyp>& out);

    Frame* activeKeyFrame = nullptr;

private:
    DeviceContext& dev_;
    int width_, height_;
};

// lsd_slam_viewer's saved map (pc.ply, KeyFrameGraphDisplay::draw, KeyFrameGraphDisplay.cpp:63-93) of the given keyframes, computed
// on the device by lsdgpu_map_export_points from each keyframe's getScaledCamToWorld(): the binary PLY header of :75-82 followed by
// one (x, y, z, intensity) float record per point (without the stray trailing byte of the viewer's copy loop, :85).
// f == nullptr: the ROS viewer parameters (cfg/LSDSLAMViewerParams.cfg:20-22).  Returns the number of points.
long long writeMapPly(DeviceContext& dev, const std::vector<Frame*>& keyframes, std::ostream& out, int publishLevel = 0,
                      const lsdgpu_map_filter* f = nullptr);

}  // namespace lsd_slam
