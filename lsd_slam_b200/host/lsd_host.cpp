// lsd_host.cpp -- implementation of lsd_host.h over the C ABI.  See the header for the reference citations.
#include "lsd_host.h"

#include <cstdio>
#include <fstream>
#include <string>

#include <cmath>
#include <cstdlib>
#include <cstring>

namespace lsd_slam {

static void qmul(const double a[4], const double b[4], double o[4])
{
    double w = a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2];
    double x = a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1];
    double y = a[3] * b[1] + a[1] * b[3] + a[2] * b[0] - a[0] * b[2];
    double z = a[3] * b[2] + a[2] * b[3] + a[0] * b[1] - a[1] * b[0];
    o[0] = x; o[1] = y; o[2] = z; o[3] = w;
}
static void qrot(const double q[4], const double v[3], double o[3])
{
    double ux = q[1] * v[2] - q[2] * v[1], uy = q[2] * v[0] - q[0] * v[2], uz = q[0] * v[1] - q[1] * v[0];
    ux += ux; uy += uy; uz += uz;
    o[0] = v[0] + q[3] * ux + (q[1] * uz - q[2] * uy);
    o[1] = v[1] + q[3] * uy + (q[2] * ux - q[0] * uz);
    o[2] = v[2] + q[3] * uz + (q[0] * uy - q[1] * ux);
}
static void qnorm(double q[4])
{
    double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    for (int i = 0; i < 4; i++) q[i] /= n;
}
SE3 SE3::inverse() const
{   // thirdparty/Sophus/sophus/se3.hpp:167-172
    SE3 r;
    r.q[0] = -q[0]; r.q[1] = -q[1]; r.q[2] = -q[2]; r.q[3] = q[3];
    qnorm(r.q);
    double nt[3] = { -t[0], -t[1], -t[2] };
    qrot(r.q, nt, r.t);
    return r;
}
SE3 SE3::operator*(const SE3& o) const
{   // se3.hpp:239-259
    SE3 r;
    double rt[3];
    qrot(q, o.t, rt);
    qmul(q, o.q, r.q);
    qnorm(r.q);
    for (int i = 0; i < 3; i++) r.t[i] = t[i] + rt[i];
    return r;
}

Sim3 Sim3::inverse() const
{
    Sim3 r;
    r.q[0] = -q[0]; r.q[1] = -q[1]; r.q[2] = -q[2]; r.q[3] = q[3];
    qnorm(r.q);
    r.s = 1.0 / s;
    double nt[3] = { -t[0], -t[1], -t[2] }, rt[3];
    qrot(r.q, nt, rt);
    for (int i = 0; i < 3; i++) r.t[i] = r.s * rt[i];
    return r;
}
Sim3 Sim3::operator*(const Sim3& o) const
{
    Sim3 r;
    double rt[3];
    qrot(q, o.t, rt);
    qmul(q, o.q, r.q);
    qnorm(r.q);
    r.s = s * o.s;
    for (int i = 0; i < 3; i++) r.t[i] = t[i] + s * rt[i];
    return r;
}
Sim3 FramePoseStruct::getCamToWorld(int recursionDepth) const
{
    if (recursionDepth >= 5000) throw LsdGpuError("FramePoseStruct::getCamToWorld: assert(recursionDepth < 5000)");
    if (trackingParent == nullptr) return Sim3();
    return trackingParent->getCamToWorld(recursionDepth + 1) * thisToParent_raw;
}

DeviceContext::DeviceContext(int device, int w, int h, const Matrix3f& K, int maxFrames) : w_(w), h_(h)
{
    int rc = lsdgpu_create(device, w, h, K.m, maxFrames, &ctx_);
    if (rc != 0) {
        std::string msg = ctx_ ? lsdgpu_last_error(ctx_) : "lsdgpu_create failed (bad size: width and height must be multiples of 16)";
        if (ctx_) lsdgpu_destroy(ctx_);
        ctx_ = nullptr;
        throw LsdGpuError(msg);
    }
}
DeviceContext::~DeviceContext() { if (ctx_) lsdgpu_destroy(ctx_); }
void DeviceContext::check(int rc, const char* where) const
{
    if (rc != 0) throw LsdGpuError(std::string(where) + ": " + lsdgpu_last_error(ctx_));
}

Frame::Frame(DeviceContext& dev, int id, int width, int height, const Matrix3f&, double timestamp, const unsigned char* image, bool distorted)
    : dev_(dev), id_(id), w_(width), h_(height), timestamp_(timestamp)
{
    pose = new FramePoseStruct();
    pose->frameID = id;
    dev_.check(distorted ? lsdgpu_frame_upload_distorted_u8(dev_.raw(), id, image) : lsdgpu_frame_upload_u8(dev_.raw(), id, image), "Frame::Frame");
}
Frame::~Frame()
{
    lsdgpu_frame_release(dev_.raw(), id_);      // may fail for the active keyframe: DepthMap::invalidate() first
    delete pose;
}
void Frame::setDepthFromGroundTruth(const float* depth, float cov_scale)
{
    dev_.check(lsdgpu_frame_set_depth_gt(dev_.raw(), id_, depth, cov_scale), "Frame::setDepthFromGroundTruth");
}
void Frame::clear_refPixelWasGood() { dev_.check(lsdgpu_frame_clear_good_mask(dev_.raw(), id_), "Frame::clear_refPixelWasGood"); }
float Frame::meanIdepth()
{
    float m = 1; int n = 0, f = 0;
    dev_.check(lsdgpu_frame_get_depth_stats(dev_.raw(), id_, &m, &n, &f), "Frame::meanIdepth");
    return m;
}
int Frame::numPoints()
{
    float m = 1; int n = 0, f = 0;
    dev_.check(lsdgpu_frame_get_depth_stats(dev_.raw(), id_, &m, &n, &f), "Frame::numPoints");
    return n;
}
bool Frame::depthHasBeenUpdatedFlag() const
{
    int f = 0;
    dev_.check(lsdgpu_frame_get_depth_stats(dev_.raw(), id_, nullptr, nullptr, &f), "Frame::depthHasBeenUpdatedFlag");
    return f != 0;
}
void Frame::downloadIdepth(int level, std::vector<float>& idepth, std::vector<float>& idepthVar)
{
    size_t n = (size_t)width(level) * height(level);
    idepth.resize(n); idepthVar.resize(n);
    dev_.check(lsdgpu_frame_download(dev_.raw(), id_, LSDGPU_BUF_IDEPTH, level, idepth.data()), "Frame::idepth");
    dev_.check(lsdgpu_frame_download(dev_.raw(), id_, LSDGPU_BUF_IDEPTH_VAR, level, idepthVar.data()), "Frame::idepthVar");
}
void Frame::downloadRefPixelWasGood(std::vector<unsigned char>& mask)
{
    mask.resize((size_t)width(1) * height(1));
    dev_.check(lsdgpu_frame_download(dev_.raw(), id_, LSDGPU_BUF_GOODMASK, 1, mask.data()), "Frame::refPixelWasGood");
}

void TrackingReference::importFrame(Frame* sourceKF)
{
    keyframe = sourceKF;
    frameID = sourceKF->id();
    sourceKF->dev().check(lsdgpu_ref_import(sourceKF->dev().raw(), frameID), "TrackingReference::importFrame");
}

SE3Tracker::SE3Tracker(DeviceContext& dev, int w, int h, const Matrix3f&) : dev_(dev), width_(w), height_(h)
{
    if (w != dev.width() || h != dev.height()) throw LsdGpuError("SE3Tracker: size differs from the device context");
}

SE3 SE3Tracker::trackFrame(TrackingReference* reference, Frame* frame, const SE3& frameToReference_initialEstimate)
{
    double init[7];
    for (int i = 0; i < 4; i++) init[i] = frameToReference_initialEstimate.q[i];
    for (int i = 0; i < 3; i++) init[4 + i] = frameToReference_initialEstimate.t[i];
    lsdgpu_track_result r;
    dev_.check(lsdgpu_se3_track(dev_.raw(), reference->keyframe->id(), frame->id(), init, &settings, mode, &r), "SE3Tracker::trackFrame");
    pointUsage = r.pointUsage; lastGoodCount = r.lastGoodCount; lastBadCount = r.lastBadCount;
    lastMeanRes = r.lastMeanRes; lastResidual = r.lastResidual;
    affineEstimation_a = r.affineEstimation_a; affineEstimation_b = r.affineEstimation_b;
    diverged = r.diverged != 0; trackingWasGood = r.trackingWasGood != 0;
    SE3 out;
    if (diverged) return out;                                         // SE3(), SE3Tracker.cpp:324-329
    for (int i = 0; i < 4; i++) out.q[i] = r.frameToRef_qt[i];
    for (int i = 0; i < 3; i++) out.t[i] = r.frameToRef_qt[4 + i];
    if (trackingWasGood) reference->keyframe->numFramesTrackedOnThis++;   // :479-480
    frame->initialTrackedResidual = r.initialTrackedResidual;         // :482
    frame->pose->thisToParent_raw = sim3FromSE3(out, 1);              // :483
    frame->pose->trackingParent = reference->keyframe->pose;          // :484
    return out;
}

Sim3Tracker::Sim3Tracker(DeviceContext& dev, int w, int h, const Matrix3f&) : dev_(dev), width_(w), height_(h)
{
    if (w != dev.width() || h != dev.height()) throw LsdGpuError("Sim3Tracker: size differs from the device context");
    lastSim3Hessian.setZero();
}

static void sim3ToQts(const Sim3& a, double o[8])
{
    for (int i = 0; i < 4; i++) o[i] = a.q[i];
    for (int i = 0; i < 3; i++) o[4 + i] = a.t[i];
    o[7] = a.s;
}

Sim3 Sim3Tracker::take(const lsdgpu_sim3_result& r)
{
    // members a diverged / rejected tracking leaves untouched keep their previous values (Sim3Tracker.cpp:184-187, 212-217)
    pointUsage = r.pointUsage;
    affineEstimation_a = r.affineEstimation_a; affineEstimation_b = r.affineEstimation_b;
    diverged = r.diverged != 0;
    Sim3 out;                                                          // Sim3()
    bool hessianZero = true;
    for (float v : r.lastSim3Hessian) hessianZero = hessianZero && v == 0.f;
    if (diverged && hessianZero) return out;                           // :184-187, :231-235
    for (int i = 0; i < 49; i++) lastSim3Hessian.m[i] = r.lastSim3Hessian[i];     // :360 (also zeroed by :215)
    if (diverged || hessianZero) return out;                           // :363-367, :212-217
    lastResidual = r.lastResidual; lastDepthResidual = r.lastDepthResidual; lastPhotometricResidual = r.lastPhotometricResidual;
    for (int i = 0; i < 4; i++) out.q[i] = r.frameToRef_qts[i];
    for (int i = 0; i < 3; i++) out.t[i] = r.frameToRef_qts[4 + i];
    out.s = r.frameToRef_qts[7];
    return out;
}

Sim3 Sim3Tracker::trackFrameSim3(TrackingReference* reference, Frame* frame, const Sim3& frameToReference_initialEstimate,
                                 int startLevel, int finalLevel)
{
    double init[8];
    sim3ToQts(frameToReference_initialEstimate, init);
    lsdgpu_sim3_result r;
    dev_.check(lsdgpu_sim3_track(dev_.raw(), reference->keyframe->id(), frame->id(), init, startLevel, finalLevel, &settings, &r),
               "Sim3Tracker::trackFrameSim3");
    return take(r);
}

void Sim3Tracker::trackFrameSim3Batch(const std::vector<TrackingReference*>& references, const std::vector<Frame*>& frames,
                                      const std::vector<Sim3>& inits, int startLevel, int finalLevel,
                                      std::vector<Sim3>& frameToReference, std::vector<lsdgpu_sim3_result>& results)
{
    const size_t n = references.size();
    if (frames.size() != n || inits.size() != n) throw LsdGpuError("Sim3Tracker::trackFrameSim3Batch: list lengths differ");
    std::vector<int> refIds(n), frIds(n);
    std::vector<double> q(8 * n);
    for (size_t i = 0; i < n; i++) {
        refIds[i] = references[i]->keyframe->id(); frIds[i] = frames[i]->id();
        sim3ToQts(inits[i], &q[8 * i]);
    }
    results.resize(n);
    dev_.check(lsdgpu_sim3_track_batch(dev_.raw(), (int)n, refIds.data(), frIds.data(), q.data(), startLevel, finalLevel, &settings, results.data()),
               "Sim3Tracker::trackFrameSim3Batch");
    frameToReference.resize(n);
    for (size_t i = 0; i < n; i++) frameToReference[i] = take(results[i]);
}

UndistorterPTAM::UndistorterPTAM(const char* configFileName)
{   // parsing as Undistorter.cpp:100-166; everything after that is lsdgpu_undistorter_ptam_prepare (:171-317)
    for (int i = 0; i < 9; i++) K_.m[i] = 0.f;
    std::ifstream infile(configFileName);
    if (!infile.good()) return;
    std::string l1, l2, l3, l4;
    std::getline(infile, l1); std::getline(infile, l2); std::getline(infile, l3); std::getline(infile, l4);
    float probe[8];
    if (std::sscanf(l1.c_str(), "%f %f %f %f %f %f %f %f", &probe[0], &probe[1], &probe[2], &probe[3], &probe[4], &probe[5], &probe[6], &probe[7]) == 8)
        return;                                                        // OpenCV camera model (:70-79)
    valid = std::sscanf(l1.c_str(), "%f %f %f %f %f", &inputCalibration[0], &inputCalibration[1], &inputCalibration[2],
                        &inputCalibration[3], &inputCalibration[4]) == 5
            && std::sscanf(l2.c_str(), "%d %d", &in_width, &in_height) == 2;
    for (float& v : outputCalibration) v = 0.f;
    bool none = false;
    if (l3 == "crop") outputCalibration[0] = -1;
    else if (l3 == "full") outputCalibration[0] = -2;
    else if (l3 == "none") none = true;                                // "NO RECTIFICATION" (:138-141): explicit zeros
    else if (std::sscanf(l3.c_str(), "%f %f %f %f %f", &outputCalibration[0], &outputCalibration[1], &outputCalibration[2],
                         &outputCalibration[3], &outputCalibration[4]) != 5)
        valid = false;
    (void)none;
    if (std::sscanf(l4.c_str(), "%d %d", &out_width, &out_height) != 2) valid = false;
    if (!valid) return;
    remapX.resize((size_t)out_width * out_height);
    remapY.resize((size_t)out_width * out_height);
    const int st = lsdgpu_undistorter_ptam_prepare(inputCalibration, in_width, in_height, outputCalibration, out_width, out_height,
                                                   remapX.data(), remapY.data(), K_.m);
    if (st < 0) { valid = false; return; }
    passThrough = (st == 1);
}

void UndistorterPTAM::install(DeviceContext& dev) const
{
    if (!valid) throw LsdGpuError("UndistorterPTAM: invalid calibration");
    if (dev.width() != out_width || dev.height() != out_height) throw LsdGpuError("UndistorterPTAM: output size differs from the device context");
    dev.check(lsdgpu_set_undistorter(dev.raw(), in_width, in_height, passThrough ? nullptr : remapX.data(), passThrough ? nullptr : remapY.data()),
              "UndistorterPTAM::install");
}

void UndistorterPTAM::undistort(DeviceContext& dev, const unsigned char* image, unsigned char* result) const
{
    dev.check(lsdgpu_undistort_u8(dev.raw(), image, result), "UndistorterPTAM::undistort");
}

DepthMap::DepthMap(DeviceContext& dev, int w, int h, const Matrix3f&) : dev_(dev), width_(w), height_(h)
{
    if (w != dev.width() || h != dev.height()) throw LsdGpuError("DepthMap: size differs from the device context");
    reset();
}
void DepthMap::reset() { dev_.check(lsdgpu_depth_reset(dev_.raw()), "DepthMap::reset"); }
void DepthMap::invalidate()
{
    activeKeyFrame = nullptr;
    dev_.check(lsdgpu_depth_invalidate(dev_.raw()), "DepthMap::invalidate");
}
void DepthMap::initializeFromGTDepth(Frame* new_frame)
{
    dev_.check(lsdgpu_depth_init_from_gt(dev_.raw(), new_frame->id()), "DepthMap::initializeFromGTDepth");
    activeKeyFrame = new_frame;
}
void DepthMap::initializeRandomly(Frame* new_frame)
{   // DepthMap.cpp:883-916: the rand() draws stay on the host, the hypotheses are uploaded
    std::vector<float> maxGrad((size_t)width_ * height_);
    dev_.check(lsdgpu_frame_download(dev_.raw(), new_frame->id(), LSDGPU_BUF_MAXGRAD, 0, maxGrad.data()), "DepthMap::initializeRandomly");
    lsdgpu_globals g;
    dev_.check(lsdgpu_get_globals(dev_.raw(), &g), "DepthMap::initializeRandomly");
    const float minAbsGradCreate = g.minUseGrad;                    // MIN_ABS_GRAD_CREATE == minUseGrad (util/settings.h:157)
    // interior pixels as in the reference; the border keeps the constructor's state (isValid = false, blacklisted = 0),
    // which is what a freshly constructed / reset DepthMap holds there (DepthMapPixelHypothesis.h:63-64, DepthMap.cpp:102-109)
    std::vector<lsdgpu_hyp> hyp((size_t)width_ * height_);
    std::memset(hyp.data(), 0, hyp.size() * sizeof(lsdgpu_hyp));
    for (int y = 1; y < height_ - 1; y++)
        for (int x = 1; x < width_ - 1; x++) {
            lsdgpu_hyp& h = hyp[x + y * width_];
            if (maxGrad[x + y * width_] > minAbsGradCreate) {
                float idepth = 0.5f + 1.0f * ((rand() % 100001) / 100000.0f);
                h.isValid = 1; h.blacklisted = 0; h.nextStereoFrameMinID = 0; h.validity_counter = 20;
                h.idepth = idepth; h.idepth_smoothed = idepth;
                h.idepth_var = 0.5f * 0.5f * 0.5f; h.idepth_var_smoothed = 0.5f * 0.5f * 0.5f;   // VAR_RANDOM_INIT_INITIAL
            }
        }
    dev_.check(lsdgpu_depth_set_hypotheses(dev_.raw(), new_frame->id(), hyp.data(), 0, 1), "DepthMap::initializeRandomly");
    activeKeyFrame = new_frame;
}
void DepthMap::setFromExistingKF(Frame* kf, const float* idepth, const float* idepthVar, const unsigned char* validity)
{   // DepthMap.cpp:920-962
    std::vector<lsdgpu_hyp> hyp((size_t)width_ * height_);
    std::memset(hyp.data(), 0, hyp.size() * sizeof(lsdgpu_hyp));
    for (size_t i = 0; i < hyp.size(); i++) {
        lsdgpu_hyp& h = hyp[i];
        if (idepthVar[i] > 0) {
            h.isValid = 1; h.blacklisted = 0; h.nextStereoFrameMinID = 0; h.validity_counter = validity[i];
            h.idepth = idepth[i]; h.idepth_var = idepthVar[i]; h.idepth_smoothed = -1; h.idepth_var_smoothed = -1;
        } else {
            h.isValid = 0;
            h.blacklisted = (idepthVar[i] == -2) ? -2 : 0;
        }
    }
    kf->numMappedOnThis = 0; kf->numFramesTrackedOnThis = 0;
    dev_.check(lsdgpu_depth_set_hypotheses(dev_.raw(), kf->id(), hyp.data(), 1, 0), "DepthMap::setFromExistingKF");
    activeKeyFrame = kf;
}
void DepthMap::updateKeyframe(std::deque<std::shared_ptr<Frame>> referenceFrames)
{
    if (!isValid()) throw LsdGpuError("DepthMap::updateKeyframe: assert(isValid())");
    std::vector<lsdgpu_ref_desc> refs;
    for (auto& f : referenceFrames) {
        if (!f->hasTrackingParent()) throw LsdGpuError("DepthMap::updateKeyframe: assert(frame->hasTrackingParent())");   // :1085
        lsdgpu_ref_desc d;
        std::memset(&d, 0, sizeof(d));
        d.frame_id = f->id();
        d.tracked_on_kf = f->pose->trackingParent->frameID == activeKeyFrame->id();                    // :1096
        if (!d.tracked_on_kf) {
            // :1087-1099: "tracked on a different frame ... While this should work, it is not recommended."
            const Sim3 refToKf = activeKeyFrame->getScaledCamToWorld().inverse() * f->getScaledCamToWorld();
            for (int i = 0; i < 4; i++) d.refToKf_qts[i] = refToKf.q[i];
            for (int i = 0; i < 3; i++) d.refToKf_qts[4 + i] = refToKf.t[i];
            d.refToKf_qts[7] = refToKf.s;
        }
        refs.push_back(d);
    }
    // the device keeps its own copy of the counters the skip-ahead logic reads (DepthMap.cpp:454)
    dev_.check(lsdgpu_frame_set_counters(dev_.raw(), activeKeyFrame->id(), activeKeyFrame->numFramesTrackedOnThis, activeKeyFrame->numMappedOnThis),
               "DepthMap::updateKeyframe");
    dev_.check(lsdgpu_depth_update_keyframe_refs(dev_.raw(), refs.data(), (int)refs.size()), "DepthMap::updateKeyframe");
    activeKeyFrame->numMappedOnThis++;
    activeKeyFrame->numMappedOnThisTotal++;
}
void DepthMap::createKeyFrame(Frame* new_keyframe)
{
    if (!isValid()) throw LsdGpuError("DepthMap::createKeyFrame: assert(isValid())");
    if (!new_keyframe || !new_keyframe->hasTrackingParent()) throw LsdGpuError("DepthMap::createKeyFrame: new keyframe has no tracking parent");
    double qts[8];
    dev_.check(lsdgpu_depth_create_keyframe(dev_.raw(), new_keyframe->id(), qts), "DepthMap::createKeyFrame");
    Sim3 s;
    for (int i = 0; i < 4; i++) s.q[i] = qts[i];
    for (int i = 0; i < 3; i++) s.t[i] = qts[4 + i];
    s.s = qts[7];
    new_keyframe->pose->thisToParent_raw = s;                            // DepthMap.cpp:1305
    activeKeyFrame = new_keyframe;
}
void DepthMap::finalizeKeyFrame()
{
    if (!isValid()) throw LsdGpuError("DepthMap::finalizeKeyFrame: assert(isValid())");
    dev_.check(lsdgpu_depth_finalize_keyframe(dev_.raw()), "DepthMap::finalizeKeyFrame");
}
void DepthMap::download(std::vector<lsdgpu_hyp>& out)
{
    out.resize((size_t)width_ * height_);
    dev_.check(lsdgpu_depth_download(dev_.raw(), out.data()), "DepthMap::download");
}

long long writeMapPly(DeviceContext& dev, const std::vector<Frame*>& keyframes, std::ostream& out, int publishLevel,
                      const lsdgpu_map_filter* f)
{
    const lsdgpu_map_filter rosDefaults = { 1e-3f, 1e-1f, 7 };
    if (!f) f = &rosDefaults;
    const int n = (int)keyframes.size();
    std::vector<int> ids(n);
    std::vector<double> qts(8 * (size_t)n);
    for (int i = 0; i < n; i++) {
        ids[i] = keyframes[i]->id();
        const Sim3 c = keyframes[i]->getScaledCamToWorld();
        for (int j = 0; j < 4; j++) qts[8 * i + j] = c.q[j];
        for (int j = 0; j < 3; j++) qts[8 * i + 4 + j] = c.t[j];
        qts[8 * i + 7] = c.s;
    }
    long long total = 0;
    dev.check(lsdgpu_map_export_points(dev.raw(), n, ids.data(), qts.data(), publishLevel, f, nullptr, 0, nullptr, &total),
              "map export (count)");
    std::vector<lsdgpu_map_point> pts((size_t)total);
    dev.check(lsdgpu_map_export_points(dev.raw(), n, ids.data(), qts.data(), publishLevel, f, pts.data(), total, nullptr, &total),
              "map export");
    out << "ply\n" << "format binary_little_endian 1.0\n" << "element vertex " << total << "\n"
        << "property float x\n" << "property float y\n" << "property float z\n" << "property float intensity\n" << "end_header\n";
    out.write(reinterpret_cast<const char*>(pts.data()), (std::streamsize)(pts.size() * sizeof(lsdgpu_map_point)));
    return total;
}

}  // namespace lsd_slam
