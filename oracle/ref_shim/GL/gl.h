// oracle/ref_shim/GL/gl.h -- TEST INFRASTRUCTURE, not OpenGL.
// lsd_slam_viewer/src/KeyFrameDisplay.cpp draws with OpenGL 1.x calls and uploads vertex buffers.  The reference-compiled viewer
// library (oracle/_ref/liblsd_ref_viewer.so) only runs setFrom / refreshPC / flushPC, whose numbers never pass through GL, so every
// GL call here is a no-op; glGenBuffers hands out a nonzero name so the reference's bookkeeping looks as it does with a context.
#ifndef LSD_REF_SHIM_GL
#define LSD_REF_SHIM_GL
typedef unsigned int GLenum;
typedef unsigned int GLuint;
typedef int GLint;
typedef int GLsizei;
typedef float GLfloat;
typedef long GLsizeiptr;
typedef unsigned char GLubyte;

#define GL_LINES 0x0001
#define GL_POINTS 0x0000
#define GL_FLOAT 0x1406
#define GL_UNSIGNED_BYTE 0x1401
#define GL_BLEND 0x0BE2
#define GL_SRC_ALPHA 0x0302
#define GL_ONE_MINUS_SRC_ALPHA 0x0303
#define GL_LIGHTING 0x0B50
#define GL_LIGHT0 0x4000
#define GL_LIGHT1 0x4001
#define GL_AMBIENT 0x1200
#define GL_AMBIENT_AND_DIFFUSE 0x1602
#define GL_VERTEX_ARRAY 0x8074
#define GL_COLOR_ARRAY 0x8076
#define GL_ARRAY_BUFFER 0x8892
#define GL_STATIC_DRAW 0x88E4

inline void glGenBuffers(GLsizei n, GLuint* b) { for (GLsizei i = 0; i < n; i++) b[i] = 1u + (GLuint)i; }
inline void glDeleteBuffers(GLsizei, const GLuint*) {}
inline void glBindBuffer(GLenum, GLuint) {}
inline void glBufferData(GLenum, GLsizeiptr, const void*, GLenum) {}
inline void glPushMatrix() {}
inline void glPopMatrix() {}
inline void glMultMatrixf(const GLfloat*) {}
inline void glColor3f(GLfloat, GLfloat, GLfloat) {}
inline void glLineWidth(GLfloat) {}
inline void glPointSize(GLfloat) {}
inline void glBegin(GLenum) {}
inline void glEnd() {}
inline void glVertex3f(GLfloat, GLfloat, GLfloat) {}
inline void glEnable(GLenum) {}
inline void glDisable(GLenum) {}
inline void glBlendFunc(GLenum, GLenum) {}
inline void glLightfv(GLenum, GLenum, const GLfloat*) {}
inline void glVertexPointer(GLint, GLenum, GLsizei, const void*) {}
inline void glColorPointer(GLint, GLenum, GLsizei, const void*) {}
inline void glEnableClientState(GLenum) {}
inline void glDisableClientState(GLenum) {}
inline void glDrawArrays(GLenum, GLint, GLsizei) {}
#endif
