// oracle/ref_shim/GL/glu.h -- TEST INFRASTRUCTURE: KeyFrameDisplay.cpp includes it and calls nothing from it.
#include "gl.h"
