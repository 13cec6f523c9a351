// mapexport.cuh -- the viewer's map export over resident keyframes: the point filter and world-frame transform of
// lsd_slam_viewer's KeyFrameDisplay::flushPC (lsd_slam_viewer/src/KeyFrameDisplay.cpp:269-340), which the viewer runs per
// keyframe on the keyframeMsg records of ROSOutput3DWrapper::publishKeyframe (lsd_slam_core/src/IOWrapper/ROS/
// ROSOutput3DWrapper.cpp:69-110) before KeyFrameGraphDisplay::draw writes pc.ply (KeyFrameGraphDisplay.cpp:60-93).
//
// Deterministic count -> scan -> write over keyframes x row bands:
//   k_map_points<false>  one CTA per (keyframe, band of rows): keep flags of the band, one count per CTA
//   k_map_scan           one CTA: exclusive scan of the CTA counts in (keyframe, band) order -> output offsets, per-keyframe counts
//   k_map_points<true>   recomputes the flags, block-scans them (row-major order inside the band) and writes the 16-byte records
// The band's idepth rows plus a one-row halo sit in shared memory for the 3x3 near-support test.  The planes are read straight from
// the frame slot (idepth, idepthVar, image of the publish level); the 12-byte keyframeMsg records are never materialised.
#pragma once
#include "internal.cuh"

#define MAP_THREADS 256
#define MAP_CHUNK 8                 // keyframes per staging buffer (two buffers: copy of chunk k overlaps the kernel of chunk k+1)

// per keyframe: planes of the publish level and the camToWorld Sim3 as the viewer holds it (Sophus::Sim3f storage)
struct MapKf {
    const float* idepth;
    const float* var;
    const float* img;
    float nq[4];                    // quaternion / |quaternion| (rxso3.hpp:263-269)
    float t[3];
    float scale;                    // RxSO3::scale() = quaternion().norm() (rxso3.hpp:311-313)
};

struct MapParams {
    int W, H;                       // publish level size
    int bandRows, nBands;           // interior rows 1..H-2 split into bands of bandRows
    float fxi, fyi, cxi, cyi;       // KeyFrameDisplay::setFrom, KeyFrameDisplay.cpp:75-78
    float scaledTH, absTH;
    int minNearSupport;
};

// keep decision of KeyFrameDisplay::flushPC for pixel (x, y), 1 <= x < W-1, 1 <= y < H-1 (KeyFrameDisplay.cpp:277-307), with
// the comparisons exactly as written: NaN / inf planes take the reference's paths.  sid = idepth rows y0-1 .. , row stride W.
__device__ __forceinline__ bool mapKeep(const float* __restrict__ sid, int ly, int x, float var, const MapParams& p, float scale,
                                        float& depth)
{
    const int W = p.W;
    const float idepth = sid[ly * W + x];
    if (idepth <= 0) return false;
    depth = 1 / idepth;
    float depth4 = depth * depth;
    depth4 *= depth4;
    if (var * depth4 > p.scaledTH) return false;
    if (var * depth4 * scale * scale > p.absTH) return false;
    if (p.minNearSupport > 1) {
        int nearSupport = 0;
        for (int dx = -1; dx < 2; dx++)
            for (int dy = -1; dy < 2; dy++) {
                const float n = sid[(ly + dy) * W + x + dx];
                if (n > 0) {
                    const float diff = n - 1.0f / depth;
                    if (diff * diff < 2 * var) nearSupport++;
                }
            }
        if (nearSupport < p.minNearSupport) return false;
    }
    return true;
}

// grid = (nBands, keyframes of this launch), kfBase = index of blockIdx.y == 0 in the call's keyframe list.
// WRITE == false: ctaCount[kf * nBands + band] = kept pixels of the band.
// WRITE == true : records of the band at out[ctaOff[kf * nBands + band] - outBase + i], i in row-major pixel order.
template <bool WRITE>
__global__ void __launch_bounds__(MAP_THREADS) k_map_points(const MapKf* __restrict__ kfs, int kfBase, MapParams p,
                                                            int* __restrict__ ctaCount, const long long* __restrict__ ctaOff,
                                                            long long outBase, float4* __restrict__ out)
{
    extern __shared__ float sid[];                      // (rows + 2) x W idepth
    __shared__ int warpTot[2][MAP_THREADS / 32];
    const int kfi = kfBase + blockIdx.y;
    const MapKf k = kfs[kfi];
    const int W = p.W;
    const int y0 = 1 + blockIdx.x * p.bandRows;
    const int y1 = min(y0 + p.bandRows, p.H - 1);       // rows y0 .. y1-1
    const int nLoad = (y1 - y0 + 2) * W;
    const float* src = k.idepth + (size_t)(y0 - 1) * W;
    for (int i = threadIdx.x; i < nLoad; i += MAP_THREADS) sid[i] = __ldg(src + i);
    __syncthreads();

    const int iw = W - 2;                               // interior columns 1 .. W-2
    const int nPix = (y1 - y0) * iw;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long pos = WRITE ? ctaOff[(size_t)kfi * p.nBands + blockIdx.x] - outBase : 0;
    int count = 0, buf = 0;
    for (int base = 0; base < nPix; base += MAP_THREADS) {
        const int i = base + threadIdx.x;
        bool keep = false;
        float depth = 0.f;
        int x = 0, y = 0;
        if (i < nPix) {
            const int r = i / iw;
            y = y0 + r;
            x = 1 + (i - r * iw);
            keep = mapKeep(sid, r + 1, x, __ldg(k.var + (size_t)y * W + x), p, k.scale, depth);
        }
        if (!WRITE) {
            count += __syncthreads_count(keep);
            continue;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) warpTot[buf][warp] = __popc(bal);
        __syncthreads();
        int before = 0, tot = 0;
        for (int w = 0; w < MAP_THREADS / 32; w++) {
            const int c = warpTot[buf][w];
            before += (w < warp) ? c : 0;
            tot += c;
        }
        if (keep) {
            // Sophus::Vector3f((x*fxi + cxi), (y*fyi + cyi), 1) * depth, then camToWorld * p = scale * q._transformVector(p) + t
            const float v[3] = { (x * p.fxi + p.cxi) * depth, (y * p.fyi + p.cyi) * depth, 1.0f * depth };
            float rv[3];
            lsd::quatRotate(k.nq, v, rv);
            const unsigned char c = (unsigned char)__ldg(k.img + (size_t)y * W + x);   // keyframeMsg colour (ROSOutput3DWrapper.cpp:103-106)
            float4 rec;
            rec.x = k.scale * rv[0] + k.t[0];
            rec.y = k.scale * rv[1] + k.t[1];
            rec.z = k.scale * rv[2] + k.t[2];
            rec.w = (float)(c / 255.0);                  // KeyFrameDisplay.cpp:331, a double division
            out[pos + before + __popc(bal & ((1u << lane) - 1u))] = rec;
        }
        pos += tot;
        buf ^= 1;                                        // the next tile writes the other half: one barrier per tile suffices
    }
    if (!WRITE && threadIdx.x == 0) ctaCount[(size_t)kfi * p.nBands + blockIdx.x] = count;
}

// one CTA: ctaOff = exclusive scan of ctaCount[0 .. n) in index order; kfCount[k] = points of keyframe k; *total
__global__ void __launch_bounds__(1024) k_map_scan(const int* __restrict__ ctaCount, int n, int nBands, long long* __restrict__ ctaOff,
                                                   int* __restrict__ kfCount, long long* __restrict__ total)
{
    __shared__ long long wsum[32];
    __shared__ long long carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        const int i = base + threadIdx.x;
        long long v = (i < n) ? ctaCount[i] : 0, incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            const long long u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += u;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        long long wbefore = 0, tileTot = 0;
        for (int w = 0; w < 32; w++) {
            wbefore += (w < warp) ? wsum[w] : 0;
            tileTot += wsum[w];
        }
        if (i < n) ctaOff[i] = carry + wbefore + incl - v;
        __syncthreads();
        if (threadIdx.x == 0) carry += tileTot;
        __syncthreads();
    }
    const int nKf = n / nBands;
    for (int k = threadIdx.x; k < nKf; k += 1024) {
        const long long end = (k + 1 < nKf) ? ctaOff[(size_t)(k + 1) * nBands] : carry;
        kfCount[k] = (int)(end - ctaOff[(size_t)k * nBands]);
    }
    if (threadIdx.x == 0) *total = carry;
}
