// Rectification (K1), 3x3 median (K5), speckle filter (K6), reprojection + ROI means (K8) on sm_100a.
#include "mvsv_internal.h"

#include <cstdint>
#include <cfloat>
#include <cmath>

namespace {

// ------------------------------------------------------------------------------------------------
// K1: cv::remap(INTER_LINEAR, CV_32FC1 maps, BORDER_CONSTANT 0) + crop  (reference
// src/Stereosystem.cpp:252-256; semantics SURVEY.md A.1).  Maps are converted once to fixed point.
// ------------------------------------------------------------------------------------------------
__global__ void k_convert_maps(const float* __restrict__ mx, const float* __restrict__ my, size_t strideElems,
                               int rx, int ry, int rw, int rh, int2* __restrict__ out)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= rw || y >= rh) return;
    size_t mi = (size_t)(y + ry) * strideElems + (size_t)(x + rx);
    out[(size_t)y * rw + x] = make_int2(__float2int_rn(mx[mi] * 32.0f), __float2int_rn(my[mi] * 32.0f));
}

// cv::initUndistortRectifyMap(K, D, R, P, size, CV_32FC1) evaluated straight into the fixed-point map
// (reference src/Stereosystem.cpp:214-217).  Double precision with explicitly rounded multiplies and adds
// (no fused multiply-add), the float rounding of the CV_32FC1 map, then the same x32 conversion as above.
__global__ void k_rectify_maps(RectifyCoef q, int rx, int ry, int rw, int rh, int2* __restrict__ out)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= rw || y >= rh) return;
    const double j = (double)(x + rx), i = (double)(y + ry);
    auto lin = [&](const double* r) { return __dadd_rn(__dadd_rn(__dmul_rn(j, r[0]), __dmul_rn(i, r[1])), r[2]); };
    const double w = lin(q.iR + 6);
    const double px = __ddiv_rn(lin(q.iR), w), py = __ddiv_rn(lin(q.iR + 3), w);
    const double x2 = __dmul_rn(px, px), y2 = __dmul_rn(py, py), r2 = __dadd_rn(x2, y2);
    const double _2xy = __dmul_rn(__dmul_rn(2.0, px), py);
    const double kr = __dadd_rn(1.0, __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(q.k3, r2), q.k2), r2), q.k1), r2));
    const double xd = __dadd_rn(__dadd_rn(__dmul_rn(px, kr), __dmul_rn(q.p1, _2xy)),
                                __dmul_rn(q.p2, __dadd_rn(r2, __dmul_rn(2.0, x2))));
    const double yd = __dadd_rn(__dadd_rn(__dmul_rn(py, kr), __dmul_rn(q.p1, __dadd_rn(r2, __dmul_rn(2.0, y2)))),
                                __dmul_rn(q.p2, _2xy));
    const float u = (float)__dadd_rn(__dmul_rn(q.fx, xd), q.cx), v = (float)__dadd_rn(__dmul_rn(q.fy, yd), q.cy);
    out[(size_t)y * rw + x] = make_int2(__float2int_rn(u * 32.0f), __float2int_rn(v * 32.0f));
}

__device__ __forceinline__ int sat16(int v) { return max(-32768, min(32767, v)); }

// One thread = four neighbouring output pixels of up to RM_FRAMES frames: the map entries and the bilinear weights are
// the same for every frame of the batch, so they are fetched and expanded once and only the four taps per pixel are
// gathered per frame; the four results leave as one 32-bit store.  RM_FRAMES: mvsv_internal.h

// frames f0 .. f1-1 of the batch (single rig), or, ORDERED, the frames order[f0 .. f1-1] that are below B (one rig)
template <bool ORDERED>
__device__ __forceinline__ void
remap_frames(const uint8_t* __restrict__ src, size_t spitch, int fw, int fh, const int2* __restrict__ map,
             uint8_t* __restrict__ dst, size_t dpitch, int W, int H, int B, int x4, int y, int f0, int f1,
             const int* __restrict__ order)
{
    int off[4][4];              // byte offsets of the four taps inside a frame, -1 = outside (BORDER_CONSTANT 0)
    int wgt[4][4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int x = min(x4 + k, W - 1);
        const int2 m = map[(size_t)y * W + x];
        const int sx = sat16(m.x >> 5), sy = sat16(m.y >> 5), fx = m.x & 31, fy = m.y & 31;
        const bool x0 = sx >= 0 && sx < fw, x1 = sx + 1 >= 0 && sx + 1 < fw;
        const bool y0 = sy >= 0 && sy < fh, y1 = sy + 1 >= 0 && sy + 1 < fh;
        off[k][0] = (y0 && x0) ? sy * (int)spitch + sx : -1;
        off[k][1] = (y0 && x1) ? sy * (int)spitch + sx + 1 : -1;
        off[k][2] = (y1 && x0) ? (sy + 1) * (int)spitch + sx : -1;
        off[k][3] = (y1 && x1) ? (sy + 1) * (int)spitch + sx + 1 : -1;
        wgt[k][0] = (32 - fx) * (32 - fy) * 32; wgt[k][1] = fx * (32 - fy) * 32;
        wgt[k][2] = (32 - fx) * fy * 32; wgt[k][3] = fx * fy * 32;
    }
    for (int i = f0; i < f1; ++i) {
        const int f = ORDERED ? order[i] : i;
        if (ORDERED && f >= B) break;                       // a chunk's frames ascend: the rest are past the batch too
        const uint8_t* s = src + (size_t)f * fh * spitch;
        unsigned out = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int acc = 16384;
#pragma unroll
            for (int t = 0; t < 4; ++t) acc += (off[k][t] >= 0 ? (int)s[off[k][t]] : 0) * wgt[k][t];
            out |= (unsigned)max(0, min(255, acc >> 15)) << (8 * k);
        }
        uint8_t* d = dst + ((size_t)f * H + y) * dpitch + x4;
        if (x4 + 3 < W) {
            *reinterpret_cast<unsigned*>(d) = out;          // dpitch and x4 are multiples of 4
        } else {
            for (int k = 0; x4 + k < W; ++k) d[k] = (uint8_t)(out >> (8 * k));
        }
    }
}

__global__ void __launch_bounds__(128)
k_remap(const uint8_t* __restrict__ src, size_t spitch, int fw, int fh, const int2* __restrict__ map,
        uint8_t* __restrict__ dst, size_t dpitch, int W, int H, int B)
{
    const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4, y = blockIdx.y;
    if (x4 >= W) return;
    const int f0 = blockIdx.z * RM_FRAMES, f1 = min(f0 + RM_FRAMES, B);
    remap_frames<false>(src, spitch, fw, fh, map, dst, dpitch, W, H, B, x4, y, f0, f1, nullptr);
}

// Frames of several rigs: blockIdx.z walks the chunks of mvsv_set_frame_rigs, each up to RM_FRAMES frames of one rig,
// which read and write at their own batch index through their rig's map.
__global__ void __launch_bounds__(128)
k_remap_rigs(const uint8_t* __restrict__ src, size_t spitch, int fw, int fh, const RigTables* __restrict__ rigs, int cam,
             const int4* __restrict__ chunks, const int* __restrict__ order, uint8_t* __restrict__ dst, size_t dpitch,
             int W, int H, int B)
{
    const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4, y = blockIdx.y;
    if (x4 >= W) return;
    const int4 ch = chunks[blockIdx.z];                     // rig, first, count
    if (order[ch.y] >= B) return;
    remap_frames<true>(src, spitch, fw, fh, rigs->map[cam][ch.x], dst, dpitch, W, H, B, x4, y, ch.y, ch.y + ch.z, order);
}

// cv::resize(src, dst, Size(0,0), f, f) for CV_8UC1, default INTER_LINEAR (reference src/Stereosystem.cpp:294-295):
// 11-bit fixed-point separable bilinear; horizontal taps clamp the coordinate and zero the fraction at the image
// edge, vertical taps clamp only the row index.  OpenCV switches to its 2x2 area average when the scale is exactly
// 1/2 (full blocks (a+b+c+d+2)>>2, clipped blocks at an odd edge: float mean rounded to nearest even).
__global__ void k_resize_linear(const uint8_t* __restrict__ src, size_t spitch, int sw, int sh, uint8_t* __restrict__ dst,
                                size_t dpitch, int dw, int dh, double scale)
{
    int dx = blockIdx.x * blockDim.x + threadIdx.x, dy = blockIdx.y, f = blockIdx.z;
    if (dx >= dw) return;
    float fx = (float)__dadd_rn(__dmul_rn((double)dx + 0.5, scale), -0.5);
    int sx = (int)floorf(fx);
    fx -= (float)sx;
    if (sx < 0) { sx = 0; fx = 0.f; }
    if (sx >= sw - 1) { sx = sw - 1; fx = 0.f; }
    float fy = (float)__dadd_rn(__dmul_rn((double)dy + 0.5, scale), -0.5);
    const int sy = (int)floorf(fy);
    fy -= (float)sy;
    const int a0 = __float2int_rn((1.f - fx) * 2048.f), a1 = __float2int_rn(fx * 2048.f);
    const int b0 = __float2int_rn((1.f - fy) * 2048.f), b1 = __float2int_rn(fy * 2048.f);
    const uint8_t* img = src + (size_t)f * sh * spitch;
    const uint8_t* r0 = img + (size_t)min(max(sy, 0), sh - 1) * spitch;
    const uint8_t* r1 = img + (size_t)min(max(sy + 1, 0), sh - 1) * spitch;
    const int x1 = min(sx + 1, sw - 1);
    const int s0 = r0[sx] * a0 + r0[x1] * a1, s1 = r1[sx] * a0 + r1[x1] * a1;
    const int v = (((b0 * (s0 >> 4)) >> 16) + ((b1 * (s1 >> 4)) >> 16) + 2) >> 2;
    dst[((size_t)f * dh + dy) * dpitch + dx] = (uint8_t)max(0, min(255, v));
}

__global__ void k_resize_half(const uint8_t* __restrict__ src, size_t spitch, int sw, int sh, uint8_t* __restrict__ dst,
                              size_t dpitch, int dw, int dh)
{
    int dx = blockIdx.x * blockDim.x + threadIdx.x, dy = blockIdx.y, f = blockIdx.z;
    if (dx >= dw) return;
    const uint8_t* img = src + (size_t)f * sh * spitch;
    const int x0 = 2 * dx, y0 = 2 * dy;
    int v;
    if (x0 + 2 <= sw && y0 + 2 <= sh) {
        const uint8_t *r0 = img + (size_t)y0 * spitch, *r1 = r0 + spitch;
        v = (r0[x0] + r0[x0 + 1] + r1[x0] + r1[x0 + 1] + 2) >> 2;
    } else {
        int sum = 0, cnt = 0;
        for (int y = y0; y < min(y0 + 2, sh); ++y)
            for (int x = x0; x < min(x0 + 2, sw); ++x) { sum += img[(size_t)y * spitch + x]; ++cnt; }
        v = cnt ? __float2int_rn(__fdiv_rn((float)sum, (float)cnt)) : 0;
    }
    dst[((size_t)f * dh + dy) * dpitch + dx] = (uint8_t)v;
}

// ------------------------------------------------------------------------------------------------
// K5: medianBlur(CV_16S, 3), replicate border (inside StereoSGBM::compute)
// ------------------------------------------------------------------------------------------------
// Row-marching: a lane keeps its column's three rows in registers (one 2-byte load per pixel), sorts them, and takes
// the neighbouring columns' sorted triples by shuffle; median9 = med3(max of the minima, med of the medians, min of
// the maxima).  Lanes 0 and 31 only feed neighbours (30 outputs per warp); clamped coordinates give the replicate
// border.
constexpr int MED_ROWS = 16, MED_COLS = 30, MED_WARPS = 4;
__device__ __forceinline__ int med3i(int a, int b, int c) { return max(min(a, b), min(max(a, b), c)); }

__global__ void __launch_bounds__(MED_WARPS * 32)
k_median3(const int16_t* __restrict__ in, int16_t* __restrict__ out, int W, int H)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x = (blockIdx.x * MED_WARPS + warp) * MED_COLS + lane - 1;
    const int y0 = blockIdx.y * MED_ROWS, y1 = min(y0 + MED_ROWS, H);
    const int16_t* img = in + (size_t)blockIdx.z * W * H;
    int16_t* dst = out + (size_t)blockIdx.z * W * H;
    const int xc = min(max(x, 0), W - 1);
    const bool writer = x >= 0 && x < W && lane >= 1 && lane <= MED_COLS;
    int p0 = img[(size_t)max(y0 - 1, 0) * W + xc], p1 = img[(size_t)y0 * W + xc];
    for (int y = y0; y < y1; ++y) {
        const int p2 = img[(size_t)min(y + 1, H - 1) * W + xc];
        const int lo = min(p0, min(p1, p2)), hi = max(p0, max(p1, p2)), mid = med3i(p0, p1, p2);
        const int loL = __shfl_up_sync(0xffffffffu, lo, 1), loR = __shfl_down_sync(0xffffffffu, lo, 1);
        const int miL = __shfl_up_sync(0xffffffffu, mid, 1), miR = __shfl_down_sync(0xffffffffu, mid, 1);
        const int hiL = __shfl_up_sync(0xffffffffu, hi, 1), hiR = __shfl_down_sync(0xffffffffu, hi, 1);
        const int m = med3i(max(lo, max(loL, loR)), med3i(mid, miL, miR), min(hi, min(hiL, hiR)));
        if (writer) dst[(size_t)y * W + x] = (int16_t)m;
        p0 = p1; p1 = p2;
    }
}

// Four columns per lane (W % 4 == 0: one 8-byte load and store per row), packed signed 16x2 arithmetic, values as pairs by
// position as in the SGBM prefilter: the sorted triples of the columns (x0-1, x0) and (x0+1, x0+2), (x0+3, x0+4) are
// one permute away from the lane's own pairs and its neighbours'.  Lanes 1..30 of a warp produce output.
constexpr int MED4_COLS = 120;
__device__ __forceinline__ unsigned med3s2(unsigned a, unsigned b, unsigned c)
{
    return __vmaxs2(__vmins2(a, b), __vmins2(__vmaxs2(a, b), c));
}

__global__ void __launch_bounds__(MED_WARPS * 32)
k_median3_w4(const int16_t* __restrict__ in, int16_t* __restrict__ out, int W, int H, int ncx, int nbands)
{
    const int lane = threadIdx.x & 31;
    const int gw = blockIdx.x * MED_WARPS + (threadIdx.x >> 5);
    const int band = gw / ncx, cx = gw - band * ncx;
    if (band >= nbands) return;                                         // whole warps only
    const int x0 = cx * MED4_COLS + 4 * (lane - 1);
    const int y0 = band * MED_ROWS, y1 = min(y0 + MED_ROWS, H);
    const int xl = min(max(x0, 0), W - 4);                              // lanes outside the row only feed edge lanes, which replicate
    const int16_t* img = in + (size_t)blockIdx.y * W * H + xl;
    int16_t* dst = out + (size_t)blockIdx.y * W * H + xl;
    const bool writer = lane >= 1 && lane <= 30 && x0 < W;
    const bool first = x0 == 0, last = x0 + 4 == W;
    auto ld = [&](int y) { return *reinterpret_cast<const uint2*>(img + (size_t)min(max(y, 0), H - 1) * W); };
    uint2 p0 = ld(y0 - 1), p1 = ld(y0);
    for (int y = y0; y < y1; ++y) {
        const uint2 p2 = ld(y + 1);
        // sorted column triples of the lane's pairs (x0, x0+1) and (x0+2, x0+3)
        const unsigned lo0 = __vimin3_s16x2(p0.x, p1.x, p2.x), hi0 = __vimax3_s16x2(p0.x, p1.x, p2.x), mi0 = med3s2(p0.x, p1.x, p2.x);
        const unsigned lo1 = __vimin3_s16x2(p0.y, p1.y, p2.y), hi1 = __vimax3_s16x2(p0.y, p1.y, p2.y), mi1 = med3s2(p0.y, p1.y, p2.y);
        unsigned res[2];
        // neighbours' pairs: (x0-1, x0) from the previous lane's second pair, (x0+3, x0+4) towards the next lane's first
        auto side = [&](unsigned q0, unsigned q1, unsigned& L0, unsigned& R0, unsigned& R1) {
            const unsigned qm = __shfl_up_sync(0xffffffffu, q1, 1), qp = __shfl_down_sync(0xffffffffu, q0, 1);
            L0 = first ? __byte_perm(q0, 0, 0x1010) : __byte_perm(qm, q0, 0x5432);      // replicate border
            R0 = __byte_perm(q0, q1, 0x5432);                                          // (x0+1, x0+2): also the left of pair 1
            R1 = last ? __byte_perm(q1, 0, 0x3232) : __byte_perm(q1, qp, 0x5432);
        };
        unsigned loL, loM, loR, miL, miM, miR, hiL, hiM, hiR;
        side(lo0, lo1, loL, loM, loR);
        side(mi0, mi1, miL, miM, miR);
        side(hi0, hi1, hiL, hiM, hiR);
        // median9 = med3(max of the minima, med of the medians, min of the maxima)
        res[0] = med3s2(__vimax3_s16x2(lo0, loL, loM), med3s2(mi0, miL, miM), __vimin3_s16x2(hi0, hiL, hiM));
        res[1] = med3s2(__vimax3_s16x2(lo1, loM, loR), med3s2(mi1, miM, miR), __vimin3_s16x2(hi1, hiM, hiR));
        if (writer) *reinterpret_cast<uint2*>(dst + (size_t)y * W) = make_uint2(res[0], res[1]);
        p0 = p1; p1 = p2;
    }
}

// ------------------------------------------------------------------------------------------------
// K6: filterSpeckles as exact connected components (SURVEY.md A.3): run-based label-equivalence CCL.
//   1. rows:    every pixel gets the index of the first pixel of its horizontal run (warp ballot scan)
//   2. vmerge:  lock-free union (atomicMin) of vertically connected runs, skipping links the left
//               neighbour already established
//   3. flatten: run starts := root; the last pixel of each run adds the run length to the root's size
//   4. apply:   components with size <= maxSize are set to newVal
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool conn(int a, int b, int newVal, int maxDiff)
{
    return a != newVal && b != newVal && abs(a - b) <= maxDiff;
}

__global__ void k_ccl_rows(const int16_t* __restrict__ img, int* __restrict__ label, int W, int nrows, int newVal,
                           int maxDiff)
{
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= nrows) return;
    const size_t base = (size_t)warp * W;
    int carry = 0;
    for (int cb = 0; cb < W; cb += 32) {
        const int x = cb + lane;
        int v = newVal, vl = newVal;
        if (x < W) {
            v = img[base + x];
            if (x > 0) vl = img[base + x - 1];
        }
        const bool valid = (x < W) && v != newVal;
        const bool start = valid && !conn(v, vl, newVal, maxDiff);
        const unsigned sb = __ballot_sync(0xffffffffu, start);
        const unsigned le = sb & (0xffffffffu >> (31 - lane));
        const int xs = le ? cb + (31 - __clz(le)) : carry;
        if (x < W) label[base + x] = valid ? (int)(base + xs) : -1;
        if (sb) carry = cb + (31 - __clz(sb));
    }
}

__device__ __forceinline__ int ccl_find(const int* L, int i)
{
    int p = L[i];
    while (p != i) { i = p; p = L[i]; }
    return i;
}

__device__ __forceinline__ void ccl_unite(int* L, int a, int b)
{
    while (true) {
        a = ccl_find(L, a);
        b = ccl_find(L, b);
        if (a == b) return;
        if (a < b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(&L[a], b);
        if (old == a) return;
        a = old;
    }
}

// vmerge / flatten: a thread owns one column of a CCL_ROWS-row strip (a CTA per pixel row would be bound by the CTA
// launch rate: the per-pixel work is a handful of loads)
constexpr int CCL_ROWS = 16;

__global__ void __launch_bounds__(128)
k_ccl_vmerge(const int16_t* __restrict__ img, int* __restrict__ label, int W, int H, int newVal, int maxDiff)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= W) return;
    const int ya = max((int)blockIdx.y * CCL_ROWS, 1), yb = min(((int)blockIdx.y + 1) * CCL_ROWS, H);
    if (ya >= yb) return;
    const size_t frameBase = (size_t)blockIdx.z * H * W;
    size_t i = frameBase + (size_t)ya * W + x;
    int vu = img[i - W], vul = x > 0 ? img[i - W - 1] : newVal;
    constexpr int CH = 4;                                     // rows whose pixel loads are issued together
    for (int y0 = ya; y0 < yb; y0 += CH) {
        int v[CH], vl[CH];
#pragma unroll
        for (int k = 0; k < CH; ++k) {
            const size_t j = frameBase + (size_t)min(y0 + k, yb - 1) * W + x;
            v[k] = img[j]; vl[k] = x > 0 ? img[j - 1] : newVal;
        }
#pragma unroll
        for (int k = 0; k < CH; ++k) {
            if (y0 + k >= yb) break;
            if (conn(v[k], vu, newVal, maxDiff)) {
                // the left neighbours already link the two rows: skip the redundant union
                const bool linked = conn(v[k], vl[k], newVal, maxDiff) && conn(vu, vul, newVal, maxDiff) &&
                                    conn(vl[k], vul, newVal, maxDiff);
                if (!linked) ccl_unite(label, label[i], label[i - W]);
            }
            vu = v[k]; vul = vl[k];
            i += W;
        }
    }
}

// One pass after all unions: run starts (the union-find tree nodes) are pointed straight at their root, so that the
// apply pass finds any pixel's root in at most two hops, and the last pixel of each run adds the run length to the
// root's size.  Compressing links while other threads still walk them is benign: a link only ever moves to an
// ancestor (monotone decreasing indices).
__global__ void __launch_bounds__(128)
k_ccl_flatten(const int16_t* __restrict__ img, int* __restrict__ label, int* __restrict__ sizes, int W, int H, int newVal,
              int maxDiff)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= W) return;
    const int ya = (int)blockIdx.y * CCL_ROWS, yb = min(ya + CCL_ROWS, H);
    const size_t frameBase = (size_t)blockIdx.z * H * W;
    // four rows at a time: all loads of the chunk are issued before any of its (possibly aliasing) label stores, so
    // they overlap instead of paying one memory latency per row
    constexpr int CH = 4;
    for (int y0 = ya; y0 < yb; y0 += CH) {
        int l[CH], v[CH], vl[CH], vr[CH];
#pragma unroll
        for (int k = 0; k < CH; ++k) {
            const int y = min(y0 + k, yb - 1);
            const size_t i = frameBase + (size_t)y * W + x;
            l[k] = label[i]; v[k] = img[i];
            vl[k] = x > 0 ? img[i - 1] : newVal; vr[k] = x < W - 1 ? img[i + 1] : newVal;
        }
#pragma unroll
        for (int k = 0; k < CH; ++k) {
            if (y0 + k >= yb || l[k] < 0) continue;
            const size_t rowBase = frameBase + (size_t)(y0 + k) * W;
            const size_t i = rowBase + x;
            const bool runStart = !conn(v[k], vl[k], newVal, maxDiff);
            const bool runEnd = !conn(v[k], vr[k], newVal, maxDiff);
            if (!runStart && !runEnd) continue;
            // label of a run start = tree link; label of the other pixels = their run start
            const int start = runStart ? (int)i : l[k];
            const int root = ccl_find(label, start);
            if (runStart && l[k] != root) label[i] = root;
            if (runEnd) atomicAdd(&sizes[root], x - (start - (int)rowBase) + 1);
        }
    }
}

// Eight consecutive pixels per thread (128-bit accesses); pixels of one run share their label, so the root / size
// lookup is done once per run segment.
__global__ void __launch_bounds__(256)
k_ccl_apply(const int16_t* __restrict__ img, int16_t* __restrict__ out, const int* __restrict__ label,
            const int* __restrict__ sizes, size_t n, int newVal, int maxSize)
{
    const size_t i0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
    if (i0 >= n) return;
    int l[8];
    __align__(16) int16_t v[8];
    const int cnt = (int)min((size_t)8, n - i0);
    if (cnt == 8) {
        const int4 la = *reinterpret_cast<const int4*>(label + i0), lb = *reinterpret_cast<const int4*>(label + i0 + 4);
        l[0] = la.x; l[1] = la.y; l[2] = la.z; l[3] = la.w; l[4] = lb.x; l[5] = lb.y; l[6] = lb.z; l[7] = lb.w;
        *reinterpret_cast<uint4*>(v) = *reinterpret_cast<const uint4*>(img + i0);
    } else {
        for (int k = 0; k < cnt; ++k) { l[k] = label[i0 + k]; v[k] = img[i0 + k]; }
    }
    int prev = -2;
    bool kill = false;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (k >= cnt) break;
        if (l[k] < 0) { v[k] = (int16_t)newVal; continue; }
        if (l[k] != prev) {
            prev = l[k];
            kill = sizes[ccl_find(label, prev)] <= maxSize;          // <= 2 hops after k_ccl_flatten
        }
        if (kill) v[k] = (int16_t)newVal;
    }
    if (cnt == 8) *reinterpret_cast<uint4*>(out + i0) = *reinterpret_cast<const uint4*>(v);
    else for (int k = 0; k < cnt; ++k) out[i0 + k] = v[k];
}

// ------------------------------------------------------------------------------------------------
// K8: reprojection (Utility::calcCoordinate over dmap2pcl's loop, reference src/utility.cpp:176-200,
// 242-262) and per-ROI mean disparity (Utility::calcMeanDisparity, src/utility.cpp:265-285).
// ------------------------------------------------------------------------------------------------
struct QMat { double q[16]; };     // the CV_32F matrix, widened on the host (cv::Mat_<float> products accumulate in double)

// Utility::calcCoordinate of one pixel (x, y) of frame f with disparity value > 0; q(f, i) is element i of the frame's
// Q.  dx, dy: the pixel's coordinates, exact in double (the reference's float coordinates are integers < 2^24).
template <class QOf>
__device__ __forceinline__ void reproject(QOf q, int f, double dx, double dy, float value, float& X, float& Y, float& Z)
{
    const double dd = (double)(value / 16.f);
    float cc[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        // ((((0 + q0 x) + q1 y) + q2 d) + q3 1): every product of two floats is exact in double, one rounding per add
        double acc = q(f, r * 4) * dx;
        acc = __fma_rn(q(f, r * 4 + 1), dy, acc);
        acc = __fma_rn(q(f, r * 4 + 2), dd, acc);
        acc += q(f, r * 4 + 3);
        cc[r] = (float)acc;
    }
    X = cc[0] / cc[3]; Y = cc[1] / cc[3]; Z = cc[2] / cc[3];
    if (isinf(Z / 1000.f)) Z = 0.f;
}

// One thread = four consecutive pixels of the batch's linear pixel index: one 8-byte load, three 16-byte stores.
// q(f, i) is element i of the Q of frame f (the four pixels may cross a frame boundary).
template <class QOf>
__device__ __forceinline__ void xyz_pixels(const int16_t* __restrict__ disp, float* __restrict__ xyz, int W, int H, size_t npx, QOf q)
{
    const size_t i0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i0 >= npx) return;
    short v4[4] = {0, 0, 0, 0};
    if (i0 + 3 < npx) {
        const uint2 raw = *reinterpret_cast<const uint2*>(disp + i0);
        v4[0] = (short)(raw.x & 0xffffu); v4[1] = (short)(raw.x >> 16); v4[2] = (short)(raw.y & 0xffffu); v4[3] = (short)(raw.y >> 16);
    } else {
        for (int k = 0; i0 + k < npx; ++k) v4[k] = disp[i0 + k];
    }
    const size_t row = i0 / W;
    int x = (int)(i0 - row * W), y = (int)(row % H);
    int f = (int)(row / H);
    double dx = (double)x, dy = (double)y;                  // exact: the reference's float coordinates are integers < 2^24
    float o[12];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float value = (float)v4[k];
        float X = 0.f, Y = 0.f, Z = 0.f;
        if (value > 0.f) reproject(q, f, dx, dy, value, X, Y, Z);
        o[3 * k] = X; o[3 * k + 1] = Y; o[3 * k + 2] = Z;
        dx += 1.0;
        if (++x == W) { x = 0; dx = 0.0; if (++y == H) { y = 0; ++f; } dy = (double)y; }
    }
    float* dst = xyz + i0 * 3;
    if (i0 + 3 < npx) {
        float4* d4 = reinterpret_cast<float4*>(dst);           // i0 is a multiple of 4: 48-byte aligned groups
        d4[0] = make_float4(o[0], o[1], o[2], o[3]); d4[1] = make_float4(o[4], o[5], o[6], o[7]); d4[2] = make_float4(o[8], o[9], o[10], o[11]);
    } else {
        for (int k = 0; i0 + k < npx; ++k) { dst[3 * k] = o[3 * k]; dst[3 * k + 1] = o[3 * k + 1]; dst[3 * k + 2] = o[3 * k + 2]; }
    }
}

__global__ void __launch_bounds__(256) k_xyz(const int16_t* __restrict__ disp, float* __restrict__ xyz, int W, int H, size_t npx, QMat Q)
{
    xyz_pixels(disp, xyz, W, H, npx, [&](int, int i) { return Q.q[i]; });
}

// Frames of several rigs: each pixel reprojects with the Q of its frame's rig, with the same arithmetic as k_xyz.
__global__ void __launch_bounds__(256)
k_xyz_rigs(const int16_t* __restrict__ disp, float* __restrict__ xyz, int W, int H, size_t npx, const RigTables* __restrict__ rigs,
           const int* __restrict__ rig_of_frame)
{
    xyz_pixels(disp, xyz, W, H, npx, [&](int f, int i) { return rigs->Q[rig_of_frame[f]][i]; });
}

// Point list (dmap2pcl's selection, reference src/utility.cpp:242-262): the pixels with disparity > 0 in (frame, row,
// column) order, reprojected as k_xyz does.  Ordered stream compaction in three kernels, none of which waits for
// another CTA: count the valid pixels of every tile, scan the counts in one CTA, then re-read each tile and write its
// points at the tile's base.  A tile is PT_TILE pixels of one frame (PT_THREADS threads x 8 consecutive pixels), so
// a frame's offset is the base of its first tile.  8 pixels per thread keep the emit kernel's staging at 32 KB: shared
// memory admits seven CTAs per SM, the registers six of k_points_emit (40 per thread) and four of k_points_emit_rigs
// (57), which is still 1024 threads per SM for a kernel bound by its 2-byte loads and 12-byte stores.
constexpr int PT_THREADS = 256, PT_PIX = 8, PT_TILE = PT_THREADS * PT_PIX;

// This thread's PT_PIX pixels of the tile starting at p0 of a frame of HW pixels: values in v (0 past the frame), bit k
// of the result set when v[k] > 0.  One 16-byte load where frames start 16-byte aligned (HW % 8 == 0).
__device__ __forceinline__ unsigned points_load(const int16_t* __restrict__ frame, int HW, int p0, short (&v)[PT_PIX])
{
    if (HW % 8 == 0 && p0 + PT_PIX <= HW) {
        const uint4 r = ld128(frame + p0);
        const unsigned w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) { v[2 * k] = (short)(w[k] & 0xffffu); v[2 * k + 1] = (short)(w[k] >> 16); }
    } else {
#pragma unroll
        for (int k = 0; k < PT_PIX; ++k) v[k] = p0 + k < HW ? frame[p0 + k] : (short)0;
    }
    unsigned m = 0;
#pragma unroll
    for (int k = 0; k < PT_PIX; ++k) m |= (v[k] > 0 ? 1u : 0u) << k;
    return m;
}

// one CTA per tile: its number of valid pixels
__global__ void __launch_bounds__(PT_THREADS)
k_points_count(const int16_t* __restrict__ disp, int HW, int tpf, long long* __restrict__ tiles)
{
    __shared__ int s_warp[PT_THREADS / 32];
    const int f = blockIdx.x / tpf, t = blockIdx.x - f * tpf;
    short v[PT_PIX];
    const int n = __popc(points_load(disp + (size_t)f * HW, HW, t * PT_TILE + threadIdx.x * PT_PIX, v));
    const int sum = __reduce_add_sync(0xffffffffu, n);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        int total = 0;
#pragma unroll
        for (int w = 0; w < PT_THREADS / 32; ++w) total += s_warp[w];
        tiles[blockIdx.x] = total;
    }
}

// One CTA: the counts of the ntiles tiles become their exclusive bases in place; offsets[f] = base of frame f's first
// tile, offsets[B] = the total.  A thread scans a contiguous segment (26 tiles at 148 frames of 752 x 479).
constexpr int PT_SCAN_THREADS = 1024;

__global__ void __launch_bounds__(PT_SCAN_THREADS)
k_points_scan(long long* __restrict__ tiles, int ntiles, int tpf, long long* __restrict__ offsets, int B)
{
    __shared__ long long s_warp[PT_SCAN_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int seg = (ntiles + PT_SCAN_THREADS - 1) / PT_SCAN_THREADS;
    const int i0 = min((int)threadIdx.x * seg, ntiles), i1 = min(i0 + seg, ntiles);
    long long sum = 0;
    for (int i = i0; i < i1; ++i) sum += tiles[i];
    long long incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    long long run = incl - sum;
    for (int w = 0; w < warp; ++w) run += s_warp[w];
    if (threadIdx.x == PT_SCAN_THREADS - 1) offsets[B] = run + sum;
    for (int i = i0; i < i1; ++i) {
        const long long n = tiles[i];
        tiles[i] = run;
        if (i % tpf == 0) offsets[i / tpf] = run;
        run += n;
    }
}

// One CTA per tile: the valid pixels are ranked within the tile (per-thread prefix, then warp and CTA scans), listed
// in shared memory in pixel order, reprojected one per thread with the arithmetic of k_xyz, and the tile's span of
// floats leaves as coalesced 4-byte stores (the span starts at 12 * base bytes: only 4-byte aligned).
template <class QOf>
__device__ __forceinline__ void points_emit(const int16_t* __restrict__ disp, int W, int HW, int tpf,
                                            const long long* __restrict__ tiles, float* __restrict__ points, QOf q)
{
    __shared__ unsigned s_pix[PT_TILE];          // value << 16 | pixel index within the tile, in pixel order
    __shared__ float s_xyz[PT_TILE * 3];
    __shared__ int s_warp[PT_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = blockIdx.x / tpf, t = blockIdx.x - f * tpf;
    const int local0 = threadIdx.x * PT_PIX;
    short v[PT_PIX];
    unsigned m = points_load(disp + (size_t)f * HW, HW, t * PT_TILE + local0, v);
    const int n = __popc(m);
    int incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int rank = incl - n, total = 0;
#pragma unroll
    for (int w = 0; w < PT_THREADS / 32; ++w) {
        const int s = s_warp[w];
        rank += w < warp ? s : 0;
        total += s;
    }
#pragma unroll
    for (int k = 0; k < PT_PIX; ++k)
        if ((m >> k) & 1u) s_pix[rank++] = (unsigned)(unsigned short)v[k] << 16 | (unsigned)(local0 + k);
    __syncthreads();
    for (int i = threadIdx.x; i < total; i += PT_THREADS) {
        const unsigned e = s_pix[i];
        const int p = t * PT_TILE + (int)(e & 0xffffu), y = p / W, x = p - y * W;
        float X, Y, Z;
        reproject(q, f, (double)x, (double)y, (float)(short)(e >> 16), X, Y, Z);
        s_xyz[3 * i] = X; s_xyz[3 * i + 1] = Y; s_xyz[3 * i + 2] = Z;
    }
    __syncthreads();
    float* dst = points + 3 * (size_t)tiles[blockIdx.x];
    for (int j = threadIdx.x; j < 3 * total; j += PT_THREADS) dst[j] = s_xyz[j];
}

__global__ void __launch_bounds__(PT_THREADS)
k_points_emit(const int16_t* __restrict__ disp, int W, int HW, int tpf, const long long* __restrict__ tiles,
              float* __restrict__ points, QMat Q)
{
    points_emit(disp, W, HW, tpf, tiles, points, [&](int, int i) { return Q.q[i]; });
}

// Frames of several rigs: each frame's points reproject with the Q of its rig, as in k_xyz_rigs.
__global__ void __launch_bounds__(PT_THREADS)
k_points_emit_rigs(const int16_t* __restrict__ disp, int W, int HW, int tpf, const long long* __restrict__ tiles,
                   float* __restrict__ points, const RigTables* __restrict__ rigs, const int* __restrict__ rig_of_frame)
{
    points_emit(disp, W, HW, tpf, tiles, points, [&](int f, int i) { return rigs->Q[rig_of_frame[f]][i]; });
}

// Eight lanes per ROI (and frame), four ROIs per warp: the reference's Samplepoint windows are 5 x 5 pixels (a whole warp
// per window left 27 lanes idle and paid one warp per 25 pixels: 0.35 ms for 5 096 ROIs x 148 frames); lanes walk the
// ROI row by row, no division per element; a CTA holds 4 * MEANS_WARPS ROIs.
constexpr int MEANS_WARPS = 8;

__global__ void __launch_bounds__(MEANS_WARPS * 32)
k_means(const int16_t* __restrict__ disp, const int* __restrict__ rois, float* __restrict__ means, int W, int H, int nrois)
{
    const int sub = threadIdx.x >> 3, l8 = threadIdx.x & 7;
    const int r = blockIdx.x * (MEANS_WARPS * 4) + sub, f = blockIdx.y;
    const int rc = min(r, nrois - 1);                                   // lanes past the last ROI repeat it and do not store
    const int4 roi = *reinterpret_cast<const int4*>(rois + rc * 4);     // x, y, w, h
    const int16_t* img = disp + (size_t)f * W * H + (size_t)roi.y * W + roi.x;
    int total = 0, n = 0;
    for (int yy = 0; yy < roi.w; ++yy, img += W)
        for (int xx = l8; xx < roi.z; xx += 8) {
            const int v = img[xx];
            if (v > 1) { total += v; ++n; }
        }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
        total += __shfl_xor_sync(0xffffffffu, total, o, 8);
        n += __shfl_xor_sync(0xffffffffu, n, o, 8);
    }
    if (l8 == 0 && r < nrois) means[(size_t)f * nrois + r] = (total == 0 || n == 0) ? 0.f : (float)(total / n);
}

__global__ void k_minmax_init(int* mm, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) mm[i] = (i & 1) ? -32768 : 32767;
}
__global__ void k_minmax(const int16_t* __restrict__ disp, int* __restrict__ mm, int npx)
{
    const int16_t* img = disp + (size_t)blockIdx.y * npx;
    int lo = 32767, hi = -32768;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += gridDim.x * blockDim.x) {
        const int v = img[i];
        if (v > 0) { lo = min(lo, v); hi = max(hi, v); }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if ((threadIdx.x & 31) == 0 && hi > 0) {
        atomicMin(&mm[2 * blockIdx.y], lo);
        atomicMax(&mm[2 * blockIdx.y + 1], hi);
    }
}

}  // namespace

cudaError_t launch_minmax(Engine* c, int B)
{
    { KernelTimer kt(c, KID_MINMAX); k_minmax_init<<<(2 * B + 127) / 128, 128, 0, c->stream>>>(c->minmax, 2 * B); }
    dim3 grd(32, B);
    KernelTimer kt(c, KID_MINMAX);
    k_minmax<<<grd, 256, 0, c->stream>>>(io(c).disp, c->minmax, c->W * c->H);
    return cudaGetLastError();
}

cudaError_t launch_convert_maps(Engine* c, int rig, int cam, const float* dmapx, const float* dmapy, size_t strideElems)
{
    dim3 blk(128), grd((c->roi_w + 127) / 128, c->roi_h);
    KernelTimer kt(c, KID_REMAP);
    k_convert_maps<<<grd, blk, 0, c->stream>>>(dmapx, dmapy, strideElems, c->roi_xy[rig][0], c->roi_xy[rig][1], c->roi_w, c->roi_h,
                                               c->map_xy[rig][cam]);
    return cudaGetLastError();
}

cudaError_t launch_rectify_maps(Engine* c, int rig, int cam, const RectifyCoef& q)
{
    dim3 blk(128), grd((c->roi_w + 127) / 128, c->roi_h);
    KernelTimer kt(c, KID_REMAP);
    k_rectify_maps<<<grd, blk, 0, c->stream>>>(q, c->roi_xy[rig][0], c->roi_xy[rig][1], c->roi_w, c->roi_h, c->map_xy[rig][cam]);
    return cudaGetLastError();
}

cudaError_t launch_remap(Engine* c, int cam, int B)
{
    const int rw = c->roi_w, rh = c->roi_h;
    const bool resized = c->resize_factor > 0.0;
    dim3 blk(128), grd((rw + 511) / 512, rh, (B + RM_FRAMES - 1) / RM_FRAMES);
    KernelTimer kt(c, KID_REMAP);
    k_remap<<<grd, blk, 0, c->stream>>>(io(c).raw[cam], c->raw_pitch, c->fw, c->fh, c->map_xy[0][cam],
                                        resized ? c->crop[cam] : io(c).rect[cam], resized ? c->crop_pitch : c->pitch, rw, rh, B);
    return cudaGetLastError();
}

cudaError_t launch_remap_rigs(Engine* c, int cam, int B)
{
    const int rw = c->roi_w, rh = c->roi_h;
    const bool resized = c->resize_factor > 0.0;
    const RigFrames& t = c->rig_frames;
    dim3 blk(128), grd((rw + 511) / 512, rh, t.nchunks);
    KernelTimer kt(c, KID_REMAP);
    k_remap_rigs<<<grd, blk, 0, c->stream>>>(io(c).raw[cam], c->raw_pitch, c->fw, c->fh, c->rig_tables, cam, t.chunk, t.order,
                                             resized ? c->crop[cam] : io(c).rect[cam], resized ? c->crop_pitch : c->pitch, rw, rh, B);
    return cudaGetLastError();
}

cudaError_t launch_resize(Engine* c, int cam, int B)
{
    const int rw = c->roi_w, rh = c->roi_h;
    const double scale = 1.0 / c->resize_factor;
    const long iscale = lrint(scale);
    dim3 blk(128), grd((c->W + 127) / 128, c->H, B);
    KernelTimer kt(c, KID_REMAP);
    if (fabs(scale - (double)iscale) < DBL_EPSILON && iscale == 2)
        k_resize_half<<<grd, blk, 0, c->stream>>>(c->crop[cam], c->crop_pitch, rw, rh, io(c).rect[cam], c->pitch, c->W, c->H);
    else
        k_resize_linear<<<grd, blk, 0, c->stream>>>(c->crop[cam], c->crop_pitch, rw, rh, io(c).rect[cam], c->pitch, c->W, c->H, scale);
    return cudaGetLastError();
}

cudaError_t launch_median(Engine* c, const int16_t* in, int16_t* out, int B)
{
    KernelTimer kt(c, KID_MEDIAN);
    const bool scalar = c->debug_flags & 4u;        // debug bit 2: k_median3 also where k_median3_w4 qualifies
    if (!scalar && c->W % 4 == 0 && c->W >= 4 && (reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) % 8 == 0) {
        const int ncx = (c->W + MED4_COLS - 1) / MED4_COLS, nbands = (c->H + MED_ROWS - 1) / MED_ROWS;
        dim3 grd((ncx * nbands + MED_WARPS - 1) / MED_WARPS, B);
        k_median3_w4<<<grd, MED_WARPS * 32, 0, c->stream>>>(in, out, c->W, c->H, ncx, nbands);
        return cudaGetLastError();
    }
    dim3 blk(MED_WARPS * 32), grd((c->W + MED_WARPS * MED_COLS - 1) / (MED_WARPS * MED_COLS), (c->H + MED_ROWS - 1) / MED_ROWS, B);
    k_median3<<<grd, blk, 0, c->stream>>>(in, out, c->W, c->H);
    return cudaGetLastError();
}

cudaError_t launch_speckle(Engine* c, const int16_t* img, int16_t* out, int B, int newVal, int maxSize, int maxDiff)
{
    const int W = c->W, H = c->H;
    const size_t n = (size_t)B * W * H;
    MVSV_TRY(cudaMemsetAsync(c->sizes, 0, n * sizeof(int), c->stream));
    const int nrows = B * H;
    { KernelTimer kt(c, KID_CCL_ROWS); k_ccl_rows<<<(nrows * 32 + 127) / 128, 128, 0, c->stream>>>(img, c->labels, W, nrows, newVal, maxDiff); }
    dim3 blk(128), grd((W + 127) / 128, (H + CCL_ROWS - 1) / CCL_ROWS, B);
    if (H > 1) {
        KernelTimer kt(c, KID_CCL_VMERGE);
        k_ccl_vmerge<<<grd, blk, 0, c->stream>>>(img, c->labels, W, H, newVal, maxDiff);
    }
    { KernelTimer kt(c, KID_CCL_FLATTEN); k_ccl_flatten<<<grd, blk, 0, c->stream>>>(img, c->labels, c->sizes, W, H, newVal, maxDiff); }
    { KernelTimer kt(c, KID_CCL_APPLY); k_ccl_apply<<<(unsigned)((n + 2047) / 2048), 256, 0, c->stream>>>(img, out, c->labels, c->sizes, n, newVal, maxSize); }
    return cudaGetLastError();
}

cudaError_t launch_xyz(Engine* c, int B)
{
    QMat Q;
    for (int i = 0; i < 16; ++i) Q.q[i] = (double)c->Q[0][i];
    const size_t npx = (size_t)B * c->H * c->W;
    KernelTimer kt(c, KID_XYZ);
    k_xyz<<<(unsigned)((npx / 4 + 256) / 256), 256, 0, c->stream>>>(io(c).disp, io(c).xyz, c->W, c->H, npx, Q);
    return cudaGetLastError();
}

cudaError_t launch_xyz_rigs(Engine* c, int B)
{
    const size_t npx = (size_t)B * c->H * c->W;
    KernelTimer kt(c, KID_XYZ);
    k_xyz_rigs<<<(unsigned)((npx / 4 + 256) / 256), 256, 0, c->stream>>>(io(c).disp, io(c).xyz, c->W, c->H, npx, c->rig_tables,
                                                                         c->rig_frames.rig);
    return cudaGetLastError();
}

size_t points_tiles(int W, int H, int B) { return (size_t)B * (((size_t)W * H + PT_TILE - 1) / PT_TILE); }

cudaError_t launch_points(Engine* c, int B, bool rigs)
{
    const int HW = c->W * c->H, tpf = (int)points_tiles(c->W, c->H, 1), ntiles = (int)points_tiles(c->W, c->H, B);
    const int16_t* disp = io(c).disp;
    { KernelTimer kt(c, KID_POINTS); k_points_count<<<ntiles, PT_THREADS, 0, c->stream>>>(disp, HW, tpf, c->pt_tiles); }
    { KernelTimer kt(c, KID_POINTS); k_points_scan<<<1, PT_SCAN_THREADS, 0, c->stream>>>(c->pt_tiles, ntiles, tpf, io(c).offsets, B); }
    KernelTimer kt(c, KID_POINTS);
    if (rigs) {
        k_points_emit_rigs<<<ntiles, PT_THREADS, 0, c->stream>>>(disp, c->W, HW, tpf, c->pt_tiles, io(c).points, c->rig_tables,
                                                                 c->rig_frames.rig);
    } else {
        QMat Q;
        for (int i = 0; i < 16; ++i) Q.q[i] = (double)c->Q[0][i];
        k_points_emit<<<ntiles, PT_THREADS, 0, c->stream>>>(disp, c->W, HW, tpf, c->pt_tiles, io(c).points, Q);
    }
    return cudaGetLastError();
}

cudaError_t launch_means(Engine* c, int B)
{
    if (c->nrois <= 0) return cudaSuccess;
    dim3 grd((c->nrois + MEANS_WARPS * 4 - 1) / (MEANS_WARPS * 4), B);
    KernelTimer kt(c, KID_MEANS);
    k_means<<<grd, MEANS_WARPS * 32, 0, c->stream>>>(io(c).disp, c->rois, io(c).means, c->W, c->H, c->nrois);
    return cudaGetLastError();
}
