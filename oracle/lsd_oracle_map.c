/*
 * lsd_oracle_map.c -- CPU ORACLE (test infrastructure, NOT product code) of the viewer's map export.
 *
 * A plain-C restatement of lsd_slam_viewer's KeyFrameDisplay::flushPC (lsd_slam_viewer/src/KeyFrameDisplay.cpp:269-340) on one
 * keyframeMsg, with the camera of setFrom (:70-78) and the filter settings refreshPC copies into my_* (:141-145; sparsifyFactor
 * == 1).  Built by oracle/map_oracle.py into oracle/liblsd_oracle_map.so (strict IEEE fp32, no FMA contraction, like
 * liblsd_oracle.so).  oracle/_ref/liblsd_ref_viewer.so exports the same name over the viewer's own KeyFrameDisplay
 * (oracle/ref_viewer_driver.cpp); tests/test_map_export_pin.py holds this restatement to it bit for bit.
 *
 * Third-party arithmetic restated (conventions of Eigen 3.2 as in oracle/lsd_oracle.h):
 *   - QuaternionBase::_transformVector (Eigen/src/Geometry/Quaternion.h, generic path)
 *   - coeffs().norm(): redux tree (x^2 + y^2) + (z^2 + w^2)
 */
#include <math.h>

/* records = the message's InputPointDense pointcloud (ROSOutput3DWrapper.h:34-39; lsdo_pack_pointcloud), w*h of them;
 * fxfycxcy = Frame::fx/fy/cx/cy(publishLvl); camToWorld_qts = getScaledCamToWorld() as unit quaternion (x,y,z,w), translation,
 * scale, cast to float as ROSOutput3DWrapper.cpp:85 does.  Writes one (x, y, z, intensity) record per kept pixel in the loop
 * order into out (room for w*h records); returns the number of records. */
int lsdo_map_export(const void* records, int w, int h, const float fxfycxcy[4], const double camToWorld_qts[8],
                    float scaledTH, float absTH, int minNearSupport, float* out)
{
    const struct { float idepth; float idepth_var; unsigned char color[4]; }* in = records;
    /* Sophus storage of the Sim3 (quaternion with |q| = scale, translation), each double coefficient cast to float */
    float q[4], t[3];
    for (int i = 0; i < 4; i++) q[i] = (float)(camToWorld_qts[i] * camToWorld_qts[7]);
    for (int i = 0; i < 3; i++) t[i] = (float)camToWorld_qts[4 + i];
    /* RxSO3::scale() = quaternion().norm() (rxso3.hpp:311-313) */
    const float scale = sqrtf((q[0]*q[0] + q[1]*q[1]) + (q[2]*q[2] + q[3]*q[3]));
    /* Sim3 * p = rxso3() * p + translation() (sim3.hpp:247-250); rxso3 * p divides the quaternion by its norm and applies
     * scale * _transformVector (rxso3.hpp:263-269) */
    const float nq[4] = { q[0] / scale, q[1] / scale, q[2] / scale, q[3] / scale };
    const float fx = fxfycxcy[0], fy = fxfycxcy[1], cx = fxfycxcy[2], cy = fxfycxcy[3];
    const float fxi = 1 / fx, fyi = 1 / fy, cxi = -cx / fx, cyi = -cy / fy;
    int num = 0;
    for (int y = 1; y < h - 1; y++)
        for (int x = 1; x < w - 1; x++) {
            const float idepth = in[x + y*w].idepth, var = in[x + y*w].idepth_var;
            if (idepth <= 0) continue;
            float depth = 1 / idepth;
            float depth4 = depth*depth; depth4 *= depth4;
            if (var * depth4 > scaledTH) continue;
            if (var * depth4 * scale * scale > absTH) continue;
            if (minNearSupport > 1) {
                int nearSupport = 0;
                for (int dx = -1; dx < 2; dx++)
                    for (int dy = -1; dy < 2; dy++) {
                        int idx = x + dx + (y + dy)*w;
                        if (in[idx].idepth > 0) {
                            float diff = in[idx].idepth - 1.0f / depth;
                            if (diff*diff < 2*var) nearSupport++;
                        }
                    }
                if (nearSupport < minNearSupport) continue;
            }
            const float p[3] = { (x*fxi + cxi) * depth, (y*fyi + cyi) * depth, 1.0f * depth };
            /* _transformVector: uv = q.vec x p; uv += uv; p + w*uv + q.vec x uv */
            float uv0 = nq[1]*p[2] - nq[2]*p[1], uv1 = nq[2]*p[0] - nq[0]*p[2], uv2 = nq[0]*p[1] - nq[1]*p[0];
            uv0 += uv0; uv1 += uv1; uv2 += uv2;
            const float c0 = nq[1]*uv2 - nq[2]*uv1, c1 = nq[2]*uv0 - nq[0]*uv2, c2 = nq[0]*uv1 - nq[1]*uv0;
            const float r[3] = { p[0] + nq[3]*uv0 + c0, p[1] + nq[3]*uv1 + c1, p[2] + nq[3]*uv2 + c2 };
            for (int i = 0; i < 3; i++) out[4*num + i] = scale * r[i] + t[i];
            /* MyVertex::color[0] = InputPointDense::color[2] (:318-320); written as color[0] / 255.0 in double (:331) */
            out[4*num + 3] = (float)(in[x + y*w].color[2] / 255.0);
            num++;
        }
    return num;
}
