// oracle/ref_shim/lsd_slam_viewer/keyframeMsg.h -- TEST INFRASTRUCTURE: the C++ message class genmsg writes for
// lsd_slam_viewer/msg/keyframeMsg.msg, with the fields of that file (fixed arrays as std::array, like boost::array in genmsg)
// and its ConstPtr typedef.  No ROS serialisation.
#ifndef LSD_REF_SHIM_KEYFRAMEMSG
#define LSD_REF_SHIM_KEYFRAMEMSG
#include <array>
#include <cstdint>
#include <memory>
#include <vector>
namespace lsd_slam_viewer {
struct keyframeMsg {
    int32_t id = 0;
    double time = 0;
    uint8_t isKeyframe = 0;
    std::array<float, 7> camToWorld{};          // serialisation of a Sophus Sim3f (quaternion with |q| = scale, translation)
    float fx = 0, fy = 0, cx = 0, cy = 0;
    uint32_t height = 0, width = 0;
    std::vector<uint8_t> pointcloud;            // InputPointDense records, width x height
};
typedef std::shared_ptr<keyframeMsg> keyframeMsgPtr;
typedef std::shared_ptr<const keyframeMsg> keyframeMsgConstPtr;
}
#endif
