// oracle/ref_shim/GL/glx.h -- TEST INFRASTRUCTURE: KeyFrameDisplay.cpp includes it and calls nothing from it.
#include "gl.h"
