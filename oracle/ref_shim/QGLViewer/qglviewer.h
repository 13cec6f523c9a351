// oracle/ref_shim/QGLViewer/qglviewer.h -- TEST INFRASTRUCTURE, not libQGLViewer.
// KeyFrameDisplay.h includes it for the GL types and, through Qt's qglobal.h, the global `uchar` typedef its structs use.
#ifndef LSD_REF_SHIM_QGLVIEWER
#define LSD_REF_SHIM_QGLVIEWER
#include "../GL/gl.h"
typedef unsigned char uchar;          /* qglobal.h */
#endif
