// oracle/ref_viewer_driver.cpp -- TEST INFRASTRUCTURE (checker only; never linked or loaded by the product).
//
// One C entry point over the reference viewer's own KeyFrameDisplay (lsd_slam_viewer/src/KeyFrameDisplay.{h,cpp} and
// settings.cpp, compiled unmodified by oracle/map_oracle.py into oracle/_ref/liblsd_ref_viewer.so against the stand-in headers of
// oracle/ref_shim/: GL no-ops, QGLViewer / ros::package includes, the keyframeMsg class).  It does what the viewer does with one
// keyframe when the user saves the map:
//   KeyFrameGraphDisplay::addMsg -> KeyFrameDisplay::setFrom(msg)                  KeyFrameGraphDisplay.cpp:142-156
//   KeyFrameDisplay::drawPC -> refreshPC()  (takes the filter settings, my_*)       KeyFrameDisplay.cpp:106-222, 342-344
//   KeyFrameGraphDisplay::draw -> flushPC(&f)                                      KeyFrameGraphDisplay.cpp:63-70
// and returns the 16-byte records flushPC wrote.  The message is filled the way ROSOutput3DWrapper::publishKeyframe fills it
// (lsd_slam_core/src/IOWrapper/ROS/ROSOutput3DWrapper.cpp:69-110): camToWorld = getScaledCamToWorld().cast<float>() storage.
// No algorithm here.
#include <cstdint>
#include <cstring>
#include <fstream>
#include <memory>
#include <sstream>
#include <string>

#include "KeyFrameDisplay.h"
#include "settings.h"

extern "C" {

// records: w*h InputPointDense (the keyframeMsg.pointcloud bytes); fxfycxcy: the publish level's camera (Frame::fx(lvl) ...);
// camToWorld_qts: Sim3 as unit quaternion (x,y,z,w), translation, scale.  out: room for w*h records of 4 floats.
// Returns the number of records (flushPC's return value).
int lsdo_map_export(const void* records, int w, int h, const float fxfycxcy[4], const double camToWorld_qts[8],
                        float scaledTH, float absTH, int minNearSupportIn, float* out)
{
    Sophus::Sim3d camToWorld;
    double* d = camToWorld.data();                       // Sophus storage: quaternion with |q| = scale, then translation
    for (int i = 0; i < 4; i++) d[i] = camToWorld_qts[i] * camToWorld_qts[7];
    for (int i = 0; i < 3; i++) d[4 + i] = camToWorld_qts[4 + i];

    auto msg = std::make_shared<lsd_slam_viewer::keyframeMsg>();
    msg->id = 0;
    msg->isKeyframe = true;
    memcpy(msg->camToWorld.data(), camToWorld.cast<float>().data(), sizeof(float) * 7);
    msg->fx = fxfycxcy[0]; msg->fy = fxfycxcy[1]; msg->cx = fxfycxcy[2]; msg->cy = fxfycxcy[3];
    msg->width = w; msg->height = h;
    msg->pointcloud.resize((size_t)w * h * sizeof(InputPointDense));
    memcpy(msg->pointcloud.data(), records, msg->pointcloud.size());

    scaledDepthVarTH = scaledTH;
    absDepthVarTH = absTH;
    minNearSupport = minNearSupportIn;
    sparsifyFactor = 1;

    std::unique_ptr<KeyFrameDisplay> kf(new KeyFrameDisplay());
    kf->setFrom(msg);
    kf->refreshPC();
    std::ofstream f;                                      // flushPC writes through the stream's buffer: point it at memory
    std::stringbuf mem(std::ios::out | std::ios::binary);
    f.std::basic_ios<char>::rdbuf(&mem);
    const int num = kf->flushPC(&f);
    const std::string bytes = mem.str();
    if (bytes.size() != (size_t)num * 16) return -1;
    memcpy(out, bytes.data(), bytes.size());
    return num;
}

}
