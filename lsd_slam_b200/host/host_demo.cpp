// host_demo.cpp -- drives the C++ classes of lsd_host.h through the SlamSystem call order (SlamSystem.cpp:890-1040,
// 739-828) on frames read from a raw file written by tests/test_host_adapter.py:
//   int32 w, h, n ; float K[9] ; float depth0[w*h] ; n x uint8 image[w*h]
// Prints one line per tracked frame: "<id> qx qy qz qw tx ty tz good".
#include <cstdio>
#include <cstdlib>
#include <sstream>
#include <string>
#include <vector>

#include "lsd_host.h"

using namespace lsd_slam;

int main(int argc, char** argv)
{
    if (argc < 2) { std::fprintf(stderr, "usage: host_demo <frames.bin> [kf_every] | host_demo --undistorter <calib.cfg> <tables.bin>\n"); return 2; }
    if (std::string(argv[1]) == "--undistorter" && argc >= 4) {
        // host-only (no GPU needed): parse a PTAM/ATAN calibration file as util/Undistorter.cpp:100-166 does, print K and the
        // sizes, dump the remap tables for the parity test
        UndistorterPTAM u(argv[2]);
        std::printf("%d %d %d %d %d %d\n", u.isValid() ? 1 : 0, u.isPassThrough() ? 1 : 0, u.getInputWidth(), u.getInputHeight(),
                    u.getOutputWidth(), u.getOutputHeight());
        for (int i = 0; i < 9; i++) std::printf("%.9g ", u.getK().m[i]);
        std::printf("\n");
        if (u.isValid()) {
            FILE* o = std::fopen(argv[3], "wb");
            if (!o) return 2;
            std::fwrite(u.remapTableX().data(), 4, u.remapTableX().size(), o);
            std::fwrite(u.remapTableY().data(), 4, u.remapTableY().size(), o);
            std::fclose(o);
        }
        return 0;
    }
    const int kfEvery = argc > 2 ? std::atoi(argv[2]) : 0;
    // "late": after a keyframe change, a frame tracked on the OLD keyframe is mapped on the new one, as the frames still queued
    // in unmappedTrackedFrames are (SlamSystem.cpp:559-575 -> DepthMap.cpp:1085-1099).  The first frame of the old keyframe is
    // used: the last one is too close to the new keyframe for the epipolar-length gate (DepthMap.cpp:203).
    const bool lateMapping = argc > 3 && std::string(argv[3]) == "late";
    FILE* f = std::fopen(argv[1], "rb");
    if (!f) { std::perror("open"); return 2; }
    int w, h, n;
    Matrix3f K;
    if (std::fread(&w, 4, 1, f) != 1 || std::fread(&h, 4, 1, f) != 1 || std::fread(&n, 4, 1, f) != 1 || std::fread(K.m, 4, 9, f) != 9) return 2;
    std::vector<float> depth((size_t)w * h);
    if (std::fread(depth.data(), 4, depth.size(), f) != depth.size()) return 2;
    std::vector<unsigned char> img((size_t)w * h);
    try {
        DeviceContext dev(0, w, h, K, 8);
        SE3Tracker tracker(dev, w, h, K);
        tracker.settings.maxItsPerLvl[4] = 0;                              // SlamSystem.cpp:80-81
        DepthMap map(dev, w, h, K);
        TrackingReference ref;
        std::shared_ptr<Frame> kf, prev, early;              // early: first frame tracked on the current keyframe
        std::vector<std::shared_ptr<Frame>> oldKeyframes;                  // their FramePoseStructs stay in the pose chain
        SE3 last;
        for (int k = 0; k < n; k++) {
            if (std::fread(img.data(), 1, img.size(), f) != img.size()) return 2;
            auto fr = std::make_shared<Frame>(dev, k, w, h, K, 0.0, img.data());
            if (k == 0) {                                                  // SlamSystem::gtDepthInit, :831-854
                fr->setDepthFromGroundTruth(depth.data());
                map.initializeFromGTDepth(fr.get());
                kf = fr;
                continue;
            }
            if (ref.keyframe != kf.get() || kf->depthHasBeenUpdatedFlag()) ref.importFrame(kf.get());   // :907-912
            SE3 pose = tracker.trackFrame(&ref, fr.get(), last);           // :932
            std::printf("%d %.12g %.12g %.12g %.12g %.12g %.12g %.12g %d\n", k, pose.q[0], pose.q[1], pose.q[2], pose.q[3],
                        pose.t[0], pose.t[1], pose.t[2], tracker.trackingWasGood ? 1 : 0);
            if (kfEvery > 0 && k % kfEvery == 0) {
                map.finalizeKeyFrame();                                    // :400
                map.createKeyFrame(fr.get());                              // :473
                oldKeyframes.push_back(kf);
                kf = fr;
                if (lateMapping && early) {
                    std::deque<std::shared_ptr<Frame>> refs{ early };
                    map.updateKeyframe(refs);                              // refToKf from the chained absolute poses, :1099
                }
                prev.reset();
                early.reset();
                last = SE3();
            } else {
                std::deque<std::shared_ptr<Frame>> refs{ fr };
                map.updateKeyframe(refs);                                  // :571
                fr->clear_refPixelWasGood();                               // :573
                last = pose;
                prev = fr;
                if (!early) early = fr;
            }
        }
        {                                                                  // the saved map of every keyframe (pc.ply)
            std::vector<Frame*> kfs;
            for (auto& o : oldKeyframes) kfs.push_back(o.get());
            kfs.push_back(kf.get());
            std::ostringstream ply;
            const long long pts = writeMapPly(dev, kfs, ply);
            std::fprintf(stderr, "host_demo: map of %zu keyframes: %lld points, %zu PLY bytes\n", kfs.size(), pts, ply.str().size());
        }
        map.invalidate();
    } catch (const std::exception& e) {
        std::fprintf(stderr, "host_demo: %s\n", e.what());
        return 1;
    }
    return 0;
}
