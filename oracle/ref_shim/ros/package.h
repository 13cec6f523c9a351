// oracle/ref_shim/ros/package.h -- TEST INFRASTRUCTURE, not roslib.  KeyFrameDisplay.cpp includes it and calls nothing from it.
#ifndef LSD_REF_SHIM_ROS_PACKAGE
#define LSD_REF_SHIM_ROS_PACKAGE
#include <string>
namespace ros { namespace package {
inline std::string getPath(const std::string&) { return "."; }
} }
#endif
