// StereoSGBM on sm_100a -- replaces cv::StereoSGBM::compute behind Disparity::sgbm
// (reference src/disparity.cpp:6-10).  Stage semantics: SURVEY.md Appendix A.2 (pinned against cv2 4.13).
// This file: prefilter, cost kernel, the two row scans (+ WTA) and the launch sequence; the fused previous-row sweep
// lives in sweep.cu.
//
// Data layout in HBM (volumes: disparity innermost, pixel stride Dp = numDisp rounded up to 8 / 16 / 32 for
// D <= 64 / 128 / 256):
//   recL[B][H][W] 8-byte records, plR[6][B][H][RP] u16 : prefilter channels a/lo/hi of the clipped x-Sobel and the raw image
//   VS[B][H][W1][Dp] u16            : vertical box sums of the Birchfield-Tomasi pixel cost
//   C [B][H][W1][Dp] u16            : block cost (horizontal box sum of VS)
//   S [B][H][W1][Dp] u16 or u8      : sum of path costs L_r -- as one byte per cell (the paths' excess over npaths * C)
//                                     while npaths * P2 <= 255 ("S8", see sweep.cu / DESIGN.md section 3)
// Lane mapping of the kernels in this file: a pixel's disparities are spread over G adjacent lanes (G = next power of
// two >= Dp / 8), 8 disparities (four packed u16x2 registers) per lane; lanes beyond Dp hold padding and never touch
// memory; the min over d is a width-G shuffle butterfly; all arithmetic is packed 16x2 (VIADD / VIMNMX.U16x2 /
// VIMNMX3 / VIADDMNMX on the integer ALU pipe of sm_100a).
#include "mvsv_internal.h"

#include <algorithm>
#include <cstdlib>
#include <functional>

namespace {

constexpr unsigned FULL = 0xffffffffu;
// compute threads of the cost kernel: 512 when a pixel needs >= 8 lanes (D > 32), so that the staging of the right-image
// entries (PX - 1 + Dp per row, eight shifted copies each) is amortised over more columns, else 256.  Measured at cfg 2
// (D = 64): 256 threads 3.16 ms, 512 threads 2.82 ms, 768 threads 3.59 ms; at D = 128 768 threads lose (2.62 -> 3.26 ms)
constexpr int vs_compute_threads(int G) { return G >= 8 ? 512 : 256; }

// ------------------------------------------------------------------------------------------------
// K2a: prefilter (A.2: sob/raw channels with ftzero borders, lo/hi half-sample bounds).
//   right image -> six u16 planes (a_s, lo_s, -hi_s, a_r, lo_r, -hi_r), stored REVERSED in x at index
//                  j = JOFF + W-1-x of a zero-padded row of RP elements, so that "disparity ascending" is
//                  "address ascending" and every CTA's first entry is 16-byte aligned;
//   left image  -> one 8-byte record per pixel (a_s, lo_s, hi_s, a_r, lo_r, hi_r, 0, 0).
// ------------------------------------------------------------------------------------------------
// A lane owns four adjacent columns (one 32-bit load per row; lanes 1..30 of a warp produce output, the outer two only
// feed their neighbours) and marches down PF_ROWS rows.  With s(x) = r0[x] + 2 r1[x] + r2[x] the Sobel response is
// s(x+1) - s(x-1); values are kept as packed 16-bit pairs BY POSITION -- (x-1, x), (x+1, x+2), (x+3, x+4) relative to
// the lane's first column -- one set per channel: the pairs of the neighbouring positions are then exactly the
// registers a pixel pair's left / right neighbours live in, and only the centre pairs need a permute.  Every position
// x <= 0 or x >= W-1 holds ftzero in both channels (the reference's border rule): the half-sample bounds of the first
// and last column then come out right without a special case ((ftzero + ftzero) >> 1 = ftzero).
constexpr int PF_ROWS = 16, PF_COLS = 120, PF_WARPS = 4;

__device__ __forceinline__ unsigned pf_lo2(unsigned w) { return __byte_perm(w, 0, 0x4140); }     // bytes 0, 1 as a u16 pair
__device__ __forceinline__ unsigned pf_hi2(unsigned w) { return __byte_perm(w, 0, 0x4342); }     // bytes 2, 3

// centre pairs, lower and upper half-sample bounds of four pixels of one channel from its three position pairs
__device__ __forceinline__ void pf_bounds(unsigned Pm, unsigned P1, unsigned P3, unsigned (&A)[2], unsigned (&LO)[2], unsigned (&HI)[2])
{
    A[0] = __byte_perm(Pm, P1, 0x5432); A[1] = __byte_perm(P1, P3, 0x5432);
    // (a + neighbour) >> 1 per half: the sums stay below 2^9, so a plain add and a masked shift are exact
    const unsigned ml0 = ((A[0] + Pm) >> 1) & 0x7fff7fffu, mr0 = ((A[0] + P1) >> 1) & 0x7fff7fffu;
    const unsigned ml1 = ((A[1] + P1) >> 1) & 0x7fff7fffu, mr1 = ((A[1] + P3) >> 1) & 0x7fff7fffu;
    LO[0] = __vimin3_u16x2(A[0], ml0, mr0); HI[0] = __vimax3_u16x2(A[0], ml0, mr0);
    LO[1] = __vimin3_u16x2(A[1], ml1, mr1); HI[1] = __vimax3_u16x2(A[1], ml1, mr1);
}

__global__ void __launch_bounds__(PF_WARPS * 32)
k_sgbm_prefilter(const uint8_t* __restrict__ img0, const uint8_t* __restrict__ img1, size_t pitch,
                 int W, int H, int ftzero, uint2* __restrict__ recL, uint16_t* __restrict__ plR,
                 size_t planeStrideR, int RP, int JOFF, int ncx, int nbands)
{
    const int lane = threadIdx.x & 31;
    const int gw = blockIdx.x * PF_WARPS + (threadIdx.x >> 5);          // warp -> (column chunk, row band)
    const int band = gw / ncx, cx = gw - band * ncx;
    if (band >= nbands) return;                                         // whole warps only
    const int x0 = cx * PF_COLS + 4 * (lane - 1);                       // this lane's first column (a multiple of 4)
    const int y0 = band * PF_ROWS, y1 = min(y0 + PF_ROWS, H);
    const int f = blockIdx.y >> 1, im = blockIdx.y & 1;
    // columns outside the row load some valid word instead: every position they feed is a border position
    const int xl = min(max(x0, 0), (int)pitch - 4);
    const uint8_t* img = (im ? img1 : img0) + (size_t)f * H * pitch + xl;
    auto ldw = [&](int y) { return *reinterpret_cast<const unsigned*>(img + (size_t)min(max(y, 0), H - 1) * pitch); };
    auto keep = [&](int xa) -> unsigned {       // halves of the pair (xa, xa + 1) that are not border positions
        return ((xa > 0 && xa < W - 1) ? 0xffffu : 0u) | ((xa + 1 > 0 && xa + 1 < W - 1) ? 0xffff0000u : 0u);
    };
    const unsigned km = keep(x0 - 1), k1 = keep(x0 + 1), k3 = keep(x0 + 3);
    const unsigned ftzp = (unsigned)ftzero * 0x10001u;
    const unsigned fm = ftzp & ~km, f1 = ftzp & ~k1, f3 = ftzp & ~k3;
    constexpr unsigned BIAS = 0x08000800u;                              // 2048 per half: the differences stay positive
    const unsigned clo = (unsigned)(2048 - ftzero) * 0x10001u, chi = (unsigned)(2048 + ftzero) * 0x10001u;
    const bool outLane = lane >= 1 && lane <= 30 && x0 < W;
    const bool full = outLane && x0 + 3 < W;                            // all four columns inside the image
    const bool vecL = (W & 1) == 0;                                     // four records = two aligned 16-byte stores
    const int alignR = (JOFF + W) & 3;                                  // 0: 8-byte stores into the planes, 2: 4-byte, odd: 2-byte
    const size_t rowsF = (size_t)f * H;

    unsigned wb = ldw(y0), wc = ldw(y0 + 1);
    unsigned a01, a23, b01 = pf_lo2(wb), b23 = pf_hi2(wb);
    { const unsigned wa = ldw(y0 - 1); a01 = pf_lo2(wa); a23 = pf_hi2(wa); }
    for (int y = y0; y < y1; ++y) {
        const unsigned wn = ldw(y + 2);                                 // two rows ahead: consumed at the end of the iteration
        const unsigned c01 = pf_lo2(wc), c23 = pf_hi2(wc);
        const unsigned S01 = a01 + 2 * b01 + c01, S23 = a23 + 2 * b23 + c23;    // s(x0), s(x0+1) | s(x0+2), s(x0+3)
        const unsigned Sm = __shfl_up_sync(FULL, S23, 1), Sp = __shfl_down_sync(FULL, S01, 1);
        // clipped Sobel + ftzero at the positions (x0-1, x0), (x0+1, x0+2), (x0+3, x0+4)
        unsigned sm = __vminu2(__vmaxu2(S01 + BIAS - Sm, clo), chi) - clo;
        unsigned s1 = __vminu2(__vmaxu2(S23 + BIAS - S01, clo), chi) - clo;
        unsigned s3 = __vminu2(__vmaxu2(Sp + BIAS - S23, clo), chi) - clo;
        // raw channel at the same positions
        const unsigned wl = __shfl_up_sync(FULL, wb, 1), wr = __shfl_down_sync(FULL, wb, 1);
        const unsigned F = __funnelshift_l(wl, wb, 8), Gw = __funnelshift_r(wb, wr, 24);
        unsigned rm = pf_lo2(F), r1 = pf_hi2(F), r3 = pf_lo2(Gw);
        sm = (sm & km) | fm; s1 = (s1 & k1) | f1; s3 = (s3 & k3) | f3;
        rm = (rm & km) | fm; r1 = (r1 & k1) | f1; r3 = (r3 & k3) | f3;
        unsigned As[2], Ls[2], Hs[2], Ar[2], Lr[2], Hr[2];
        pf_bounds(sm, s1, s3, As, Ls, Hs);
        pf_bounds(rm, r1, r3, Ar, Lr, Hr);
        if (outLane) {
            if (im == 0) {
                // record of a pixel: bytes a_s lo_s hi_s a_r | lo_r hi_r 0 0
                uint2 rec[4];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const unsigned T1 = __byte_perm(As[h], Ls[h], 0x6240), T2 = __byte_perm(Hs[h], Ar[h], 0x6240);
                    const unsigned T3 = __byte_perm(Lr[h], Hr[h], 0x6240);
                    rec[2 * h] = make_uint2(__byte_perm(T1, T2, 0x5410), T3 & 0xffffu);
                    rec[2 * h + 1] = make_uint2(__byte_perm(T1, T2, 0x7632), T3 >> 16);
                }
                uint2* dst = recL + (rowsF + y) * W + x0;
                if (full && vecL) {
                    reinterpret_cast<uint4*>(dst)[0] = make_uint4(rec[0].x, rec[0].y, rec[1].x, rec[1].y);
                    reinterpret_cast<uint4*>(dst)[1] = make_uint4(rec[2].x, rec[2].y, rec[3].x, rec[3].y);
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (x0 + k < W) dst[k] = rec[k];
                }
            } else {
                // planes a_s, lo_s, -hi_s, a_r, lo_r, -hi_r, reversed in x: columns x0+3 .. x0 at indices j0-3 .. j0
                const unsigned V[6][2] = {{As[0], As[1]}, {Ls[0], Ls[1]}, {__vneg2(Hs[0]), __vneg2(Hs[1])},
                                          {Ar[0], Ar[1]}, {Lr[0], Lr[1]}, {__vneg2(Hr[0]), __vneg2(Hr[1])}};
                uint16_t* o = plR + (rowsF + y) * RP + (JOFF + W - 1 - x0);
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    uint16_t* op = o + (size_t)k * planeStrideR;
                    const unsigned lo = __byte_perm(V[k][1], 0, 0x1032), hi = __byte_perm(V[k][0], 0, 0x1032);    // (x0+3, x0+2), (x0+1, x0)
                    if (full && alignR == 0) {
                        *reinterpret_cast<uint2*>(op - 3) = make_uint2(lo, hi);
                    } else if (full && alignR == 2) {
                        *reinterpret_cast<unsigned*>(op - 3) = lo; *reinterpret_cast<unsigned*>(op - 1) = hi;
                    } else {
                        if (x0 < W) op[0] = (uint16_t)(V[k][0] & 0xffffu);
                        if (x0 + 1 < W) op[-1] = (uint16_t)(V[k][0] >> 16);
                        if (x0 + 2 < W) op[-2] = (uint16_t)(V[k][1] & 0xffffu);
                        if (x0 + 3 < W) op[-3] = (uint16_t)(V[k][1] >> 16);
                    }
                }
            }
        }
        a01 = b01; a23 = b23; b01 = c01; b23 = c23; wb = wc; wc = wn;
    }
}

// ------------------------------------------------------------------------------------------------
// K2b: Birchfield-Tomasi pixel cost + vertical box sum.  One CTA = PX = 256/G adjacent columns of one frame,
// marching down the rows in lock-step.  Lane (p, q) evaluates column xa+p at disparities 8q..8q+7: the left
// pixel is a broadcast scalar, the right pixels are eight consecutive entries of the reversed planes.  Their
// start is only 2-byte aligned, so each row's entries are staged in shared memory as EIGHT element-shifted copies
// (built from aligned 128-bit global loads with funnel shifts); every lane then fetches a channel's eight values
// with one aligned LDS.128 from the copy matching its alignment.  Staging is double buffered (global loads for
// row t+2 in flight, copies of row t+1 written while row t is consumed): one __syncthreads per row.
// ------------------------------------------------------------------------------------------------
struct VsArgs {
    const uint2* recL; const uint16_t* plR; size_t planeStrideR;
    uint16_t* VS;
    int W, H, W1, D, Dp, minD, minX1, SH2, NV, LEN, RP, JOFF;
    int bandRows;               // output rows per blockIdx.z (== H: one band); a band restarts the vertical sum
};

__device__ __forceinline__ unsigned bt_pair(unsigned v, unsigned v0, unsigned nv1, unsigned uu, unsigned nuu,
                                            unsigned uu1, unsigned uu0, unsigned kk)
{
    unsigned c0 = __vimax_s16x2_relu(__vadd2(uu, nv1), __vadd2(v0, nuu));   // max(0, u-v1, v0-u)
    unsigned c1 = __vmaxs2(v, uu1) - __vmins2(v, uu0) - kk;                  // max(0, v-u1, u0-v), no cross-half borrow
    return __vmins2(c0, c1);
}

// cp.async (LDGSTS) helpers: asynchronous global -> shared copies, completion tracked per thread in groups
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
constexpr int VS_RD = 4;       // raw-ring depth of the cost kernel's producer (rows in flight + 1)

// geometry fixed by G: entries a CTA can touch, 8-entry vectors per channel, producer warps.  WIDE (G = 32, D > 128
// only): 768 compute threads = 24 columns per CTA instead of 16, when the row ring still fits shared memory -- the
// 271 staged entries per row are then shared by more columns (cfg 4: 8.14 -> 7.3 ms per 14 frames).
template <int G, bool WIDE> struct VsGeom {
    static constexpr int CT = (WIDE && G == 32) ? 768 : vs_compute_threads(G);
    static constexpr int PX = CT / G;
    static constexpr int NE = PX - 1 + 8 * G;
    static constexpr int NV = (NE + 2 + 7) / 8;                // one spare entry pair for the odd copies
    static constexpr int ITEMS = 6 * NV;                       // (channel, vector) staging items per row
    static constexpr int NPW = (ITEMS + 95) / 96;              // producer warps: <= 3 items per producer lane
    static constexpr int NPT = 32 * NPW;                       // producer threads
    static constexpr int IPL = (ITEMS + NPT - 1) / NPT;        // items per producer lane
    static constexpr int RPL = (PX + NPT - 1) / NPT;           // left records per producer lane
    static constexpr int THREADS = CT + NPT;
};

__device__ __forceinline__ void named_bar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

template <int G, bool R8, bool BANDS, bool WIDE>
__global__ void __launch_bounds__(VsGeom<G, WIDE>::THREADS) k_sgbm_vsum(VsArgs a)
{
    using GE = VsGeom<G, WIDE>;
    constexpr int PX = GE::PX;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // layout: sR[2 buf][6][8][LEN] u16 | sL[2 buf][PX][12] u32 | ring[bs][CT] (uint2 if the pixel cost
    // fits a byte -- 2*ftzero+63 <= 255 -- else uint4)
    uint16_t* sR = reinterpret_cast<uint16_t*>(smem_raw);
    unsigned* sL = reinterpret_cast<unsigned*>(sR + (size_t)2 * 6 * 8 * a.LEN);
    unsigned char* ring = reinterpret_cast<unsigned char*>(sL + 2 * PX * 12);

    const int tid = threadIdx.x;
    const int f = blockIdx.y;
    const int xa = blockIdx.x * PX;
    const int bs = 2 * a.SH2 + 1;
    // Row band [ya, yb) of this CTA (small batches are split into bands to fill the GPU; a band pays blockSize-1
    // warm-up rows): step t adds pixel row clamp(t - SH2) and, once bs rows are in, emits output row t - (bs-1)
    const int ya = BANDS ? blockIdx.z * a.bandRows : 0, yb = BANDS ? min(ya + a.bandRows, a.H) : a.H;
    const int tb = ya, steps = yb + 2 * a.SH2;
    const size_t rowsR = (size_t)f * a.H;
    // named barriers: 1 + buf = "stage buf is full", 3 + buf = "stage buf is free again"
    constexpr int NTH = GE::THREADS;

    constexpr int CT = GE::CT;
    if (tid >= CT) {
        // ===================== producer warps: stage row t while the compute warps consume row t-1 ===============
        // Global loads run VS_RD-1 rows ahead through cp.async into a private raw ring (every lane reads back only
        // what it copied), so the producer's critical path is LDS -> funnel shifts -> STS.
        const int pt = tid - CT;
        const int xr_max = xa + PX - 1 + a.minX1 - a.minD;       // entry e <-> right column xr_max - e
        const int j0 = a.JOFF + a.W - 1 - xr_max;                // reversed-plane index of entry 0 (multiple of 8)
        uint4* rawPQ = reinterpret_cast<uint4*>(ring + (size_t)bs * CT * (R8 ? 8 : 16));   // [VS_RD][IPL][2][NPT]
        uint2* rawL = reinterpret_cast<uint2*>(rawPQ + VS_RD * GE::IPL * 2 * GE::NPT);             // [VS_RD][RPL][NPT]
        size_t srcOff[GE::IPL]; int dstOff[GE::IPL]; bool itemOn[GE::IPL];
#pragma unroll
        for (int k = 0; k < GE::IPL; ++k) {
            const int item = pt + k * GE::NPT;
            itemOn[k] = item < GE::ITEMS;
            const int arr = itemOn[k] ? item / GE::NV : 0, m = itemOn[k] ? item % GE::NV : 0;
            srcOff[k] = (size_t)arr * a.planeStrideR + rowsR * a.RP + j0 + 8 * m;
            dstOff[k] = arr * 8 * a.LEN + 8 * m;
        }
        auto issue_loads = [&](int t) {
            if (t < steps) {
                const int y = min(max(t - a.SH2, 0), a.H - 1);
                const int rs = t % VS_RD;
#pragma unroll
                for (int k = 0; k < GE::IPL; ++k) {
                    if (itemOn[k]) {
                        const uint16_t* src = a.plR + srcOff[k] + (size_t)y * a.RP;
                        uint4* d = rawPQ + ((rs * GE::IPL + k) * 2) * GE::NPT + pt;
                        cp_async16(d, src - 8);
                        cp_async16(d + GE::NPT, src);
                    }
                }
#pragma unroll
                for (int k = 0; k < GE::RPL; ++k) {
                    const int px = pt + k * GE::NPT;
                    if (px < PX && xa + px < a.W1)
                        cp_async8(rawL + (rs * GE::RPL + k) * GE::NPT + pt, a.recL + (rowsR + y) * a.W + xa + px + a.minX1);
                }
            }
            cp_async_commit();
        };
        auto store_stage = [&](int buf, int t) {
            const int rs = t % VS_RD;
#pragma unroll
            for (int k = 0; k < GE::IPL; ++k) {
                if (itemOn[k]) {
                    uint16_t* dst = sR + (size_t)buf * 6 * 8 * a.LEN + dstOff[k];
                    const uint4* d = rawPQ + ((rs * GE::IPL + k) * 2) * GE::NPT + pt;
                    const uint4 p4 = d[0], q4 = d[GE::NPT];
                    const unsigned f0 = __funnelshift_r(p4.x, p4.y, 16), f1 = __funnelshift_r(p4.y, p4.z, 16);
                    const unsigned f2 = __funnelshift_r(p4.z, p4.w, 16), f3 = __funnelshift_r(p4.w, q4.x, 16);
                    const unsigned f4 = __funnelshift_r(q4.x, q4.y, 16), f5 = __funnelshift_r(q4.y, q4.z, 16);
                    const unsigned f6 = __funnelshift_r(q4.z, q4.w, 16);
                    // copy s holds entry e at position e+s: positions [8m, 8m+8) of copy s = entries [8m-s, 8m-s+8)
                    st128(dst + 0 * a.LEN, q4);
                    st128(dst + 1 * a.LEN, make_uint4(f3, f4, f5, f6));
                    st128(dst + 2 * a.LEN, make_uint4(p4.w, q4.x, q4.y, q4.z));
                    st128(dst + 3 * a.LEN, make_uint4(f2, f3, f4, f5));
                    st128(dst + 4 * a.LEN, make_uint4(p4.z, p4.w, q4.x, q4.y));
                    st128(dst + 5 * a.LEN, make_uint4(f1, f2, f3, f4));
                    st128(dst + 6 * a.LEN, make_uint4(p4.y, p4.z, p4.w, q4.x));
                    st128(dst + 7 * a.LEN, make_uint4(f0, f1, f2, f3));
                }
            }
#pragma unroll
            for (int k = 0; k < GE::RPL; ++k) {
                const int px = pt + k * GE::NPT;
                if (px < PX) {
                    // words: 0 uu_s 1 nuu_s 2 uu1_s 3 uu0_s 4 kk_s 5 uu_r 6 nuu_r 7 uu1_r 8 uu0_r 9 kk_r
                    const uint2 lr = (xa + px < a.W1) ? rawL[(rs * GE::RPL + k) * GE::NPT + pt] : make_uint2(0, 0);
                    const int us = lr.x & 0xff, los = (lr.x >> 8) & 0xff, his = (lr.x >> 16) & 0xff, ur = lr.x >> 24;
                    const int lor = lr.y & 0xff, hir = (lr.y >> 8) & 0xff;
                    unsigned* d = sL + (buf * PX + px) * 12;
                    st128(d, make_uint4(pk16(us), pk16(-us), pk16(his), pk16(los)));
                    st128(d + 4, make_uint4(pk16(his - los), pk16(ur), pk16(-ur), pk16(hir)));
                    st128(d + 8, make_uint4(pk16(lor), pk16(hir - lor), 0u, 0u));
                }
            }
        };
#pragma unroll
        for (int t0 = 0; t0 < VS_RD - 1; ++t0) issue_loads(tb + t0);
        for (int t = tb; t < steps; ++t) {
            const int buf = t & 1;
            issue_loads(t + VS_RD - 1);                        // into the raw slot consumed at step t-1
            cp_async_wait<VS_RD - 1>();                        // row t has landed
            if (t - tb >= 2) named_bar_sync(3 + buf, NTH);     // compute warps are done with row t-2 (same buffer)
            store_stage(buf, t);
            named_bar_arrive(1 + buf, NTH);
        }
        cp_async_wait<0>();
        return;
    }

    // ===================== compute warps ==========================================================================
    const int p = tid / G, q = tid % G;
    const int xi = xa + p;
    const bool live = (xi < a.W1) && (q * 8 < a.D);
    const int e0 = (PX - 1 - p) + 8 * q;
    const int sh = (-e0) & 7;
    const int rbase = sh * a.LEN + e0 + sh;                   // + (buf*6 + arr)*8*LEN
    uint4 acc = make_uint4(0, 0, 0, 0);
    int slot = 0;
    for (int t = tb; t < steps; ++t) {
        const int buf = t & 1;
        named_bar_sync(1 + buf, NTH);
        if (live) {
            const uint16_t* rb = sR + (size_t)buf * 6 * 8 * a.LEN + rbase;
            const uint4 A0 = ld128(rb + 0 * 8 * a.LEN), A1 = ld128(rb + 1 * 8 * a.LEN), A2 = ld128(rb + 2 * 8 * a.LEN);
            const uint4 A3 = ld128(rb + 3 * 8 * a.LEN), A4 = ld128(rb + 4 * 8 * a.LEN), A5 = ld128(rb + 5 * 8 * a.LEN);
            const unsigned* lw = sL + (buf * PX + p) * 12;
            const uint4 w0 = ld128(lw), w1 = ld128(lw + 4), w2 = ld128(lw + 8);
            uint4 pix;
#define MVSV_PIX(c)                                                                                   \
    {                                                                                                 \
        unsigned cs = bt_pair(A0.c, A1.c, A2.c, w0.x, w0.y, w0.z, w0.w, w1.x);                        \
        unsigned cr = bt_pair(A3.c, A4.c, A5.c, w1.y, w1.z, w1.w, w2.x, w2.y);                        \
        pix.c = cs + ((cr >> 2) & 0x3fff3fffu);                                                       \
    }
            MVSV_PIX(x) MVSV_PIX(y) MVSV_PIX(z) MVSV_PIX(w)
#undef MVSV_PIX
            uint4 old = make_uint4(0, 0, 0, 0);
            if (R8) {
                uint2* rs = reinterpret_cast<uint2*>(ring) + (size_t)slot * CT + tid;
                if (t - tb >= bs) {
                    const uint2 o = *rs;
                    old = make_uint4(__byte_perm(o.x, 0, 0x4140), __byte_perm(o.x, 0, 0x4342), __byte_perm(o.y, 0, 0x4140),
                                     __byte_perm(o.y, 0, 0x4342));
                }
                *rs = make_uint2(__byte_perm(pix.x, pix.y, 0x6420), __byte_perm(pix.z, pix.w, 0x6420));
            } else {
                uint4* rs = reinterpret_cast<uint4*>(ring) + (size_t)slot * CT + tid;
                if (t - tb >= bs) old = *rs;
                *rs = pix;
            }
            acc.x += pix.x - old.x; acc.y += pix.y - old.y; acc.z += pix.z - old.z; acc.w += pix.w - old.w;
            if (t - tb >= bs - 1) {
                const int yo = t - (bs - 1);
                st128(a.VS + (((size_t)f * a.H + yo) * a.W1 + xi) * a.Dp + q * 8, acc);
            }
        }
        // barrier instructions need a converged warp (`live` differs between lanes in edge CTAs / padded lanes)
        __syncwarp();
        if (t + 2 < steps) named_bar_arrive(3 + buf, NTH);       // stage buffer consumed: hand it back
        if (++slot == bs) slot = 0;
    }
}

// ------------------------------------------------------------------------------------------------
// K3: one step of the path recurrence (A.2 `step`) on 8 disparities per lane.
//   L[k] = C[k] + min(Lp[k], Lp[k-1]+P1, Lp[k+1]+P1, m+P2) - m ;  mm = packed min_k L[k]
// Off-domain predecessor == state (L = 0, mm = 0), which yields L = C.
// PAD: numDisp is not 8*G, lanes with q*8 >= D hold the constant 0x7fff (the out-of-range neighbour value).
// ------------------------------------------------------------------------------------------------
// minimum of a 32-bit value over the G lanes of a pixel: REDUX where a pixel is the whole warp or half of it (two
// warp-wide reductions with the other half masked out), shuffle butterfly below that
template <int G>
__device__ __forceinline__ unsigned group_min_u32(unsigned v)
{
    if constexpr (G == 32) {
        return __reduce_min_sync(FULL, v);
    } else if constexpr (G == 16) {
        const bool upper = (threadIdx.x & 16) != 0;
        const unsigned r0 = __reduce_min_sync(FULL, upper ? 0xffffffffu : v), r1 = __reduce_min_sync(FULL, upper ? v : 0xffffffffu);
        return upper ? r1 : r0;
    } else {
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(FULL, v, o, G));
        return v;
    }
}

template <int G, bool PAD>
__device__ __forceinline__ void sgm_step(unsigned (&L)[4], unsigned& mm, const uint4& C, unsigned P1P1, unsigned P2P2,
                                         int q, bool padLane)
{
    // min(min(Lp[k-1], Lp[k+1]) + P1, Lp[k], m + P2) == min3(Lp[k-1] + P1, Lp[k+1] + P1, min(Lp[k], m + P2)):
    // P1 is added once per register with a plain 32-bit add (no carry between the halves: L + P1 < 65536), which
    // issues at full rate, and one VIMNMX3 replaces a VIMNMX + VIADDMNMX pair on the half-rate DPX pipe.
    const unsigned P0 = L[0] + P1P1, P3 = L[3] + P1P1;
    unsigned up = 0xffffffffu, dn = 0xffffffffu;        // out-of-range neighbour: larger than any L + P1
    if (G > 1) {
        const unsigned u = __shfl_up_sync(FULL, P3, 1, G);
        const unsigned d = __shfl_down_sync(FULL, P0, 1, G);
        if (q != 0) up = u;
        if (q != G - 1) dn = d;
    }
    const unsigned Q1 = L[1] + P1P1, Q2 = L[2] + P1P1;
    const unsigned X0 = __byte_perm(up, P0, 0x5432);
    const unsigned X1 = __byte_perm(P0, Q1, 0x5432);
    const unsigned X2 = __byte_perm(Q1, Q2, 0x5432);
    const unsigned X3 = __byte_perm(Q2, P3, 0x5432);
    const unsigned X4 = __byte_perm(P3, dn, 0x5432);
    const unsigned mP2 = mm + P2P2;
    unsigned n0 = __vimin3_u16x2(X0, X1, __vminu2(L[0], mP2)) + C.x - mm;
    unsigned n1 = __vimin3_u16x2(X1, X2, __vminu2(L[1], mP2)) + C.y - mm;
    unsigned n2 = __vimin3_u16x2(X2, X3, __vminu2(L[2], mP2)) + C.z - mm;
    unsigned n3 = __vimin3_u16x2(X3, X4, __vminu2(L[3], mP2)) + C.w - mm;
    if (PAD && padLane) { n0 = n1 = n2 = n3 = MVSV_PK_MAX; }
    unsigned m = __vminu2(__vimin3_u16x2(n0, n1, n2), n3);
    if (G >= 16) {
        // a pixel is the whole warp or half of it: REDUX instead of a five- / four-step shuffle butterfly
        mm = group_min_u32<G>(min(m & 0xffffu, m >> 16)) * 0x10001u;
    } else {
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) m = __vminu2(m, __shfl_xor_sync(FULL, m, o, G));
        mm = __vminu2(m, __byte_perm(m, 0, 0x1032));
    }
    L[0] = n0; L[1] = n1; L[2] = n2; L[3] = n3;
}

template <bool PAD>
__device__ __forceinline__ void reset_state(unsigned (&L)[4], unsigned& mm, bool padLane)
{
    const unsigned v = (PAD && padLane) ? MVSV_PK_MAX : 0u;
    L[0] = L[1] = L[2] = L[3] = v;
    mm = 0u;
}

__device__ __forceinline__ void sat_acc(uint4& S, const unsigned (&L)[4])
{
    S.x = __viaddmin_u16x2(S.x, L[0], MVSV_PK_MAX); S.y = __viaddmin_u16x2(S.y, L[1], MVSV_PK_MAX);
    S.z = __viaddmin_u16x2(S.z, L[2], MVSV_PK_MAX); S.w = __viaddmin_u16x2(S.w, L[3], MVSV_PK_MAX);
}

struct AggArgs {
    const uint16_t* VS; uint16_t* C; uint16_t* S;
    int H, W, W1, D, Dp, SW2, B;
    unsigned P1P1, P2P2;
    // WTA
    int16_t* disp; int* d2;
    int minD, minX1, maxX1, INV, uniq, d12;
    int storeS;
    // S8: the S volume holds, per cell, the byte (sum of the paths so far) - (paths so far) * C (see sweep.cu)
    uint16_t* Sdbg;             // where the final S goes when the test hook asks for it in S8 mode (the dead VS volume)
    unsigned nprevPk, kclampPk; // S8: number of paths, and ceil(32767 / that), both packed x2
};

// The row scans stream their operands through a per-lane shared-memory ring filled by cp.async (LDGSTS): the
// loads of the next PFD steps are in flight without holding registers.  Each lane only ever reads back the 16
// bytes it copied itself, so cp.async.wait_group is the only synchronisation needed.
constexpr int H1_PFD = 8;
constexpr int HPF = 2;         // k_sgbm_h2_wta is issue-bound: it keeps a cheap 2-step register prefetch instead


// K3a: horizontal box sum (VS -> C) fused with the left-to-right path r=(-1,0).  Writes C and S = L
// (S8: the bytes L - C, one per disparity).
template <int G, bool PAD, bool S8>
__global__ void __launch_bounds__(128) k_sgbm_h1(AggArgs a)
{
    // a pixel's stride in the volumes is a.Dp <= 8*G: lanes beyond it hold padding only and never touch memory
    const int DP = a.Dp;
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nrows = (long long)a.B * a.H;
    long long row = gtid / G;
    const int q = (int)(gtid % G);
    const bool mem = q * 8 < DP;
    const bool active = row < nrows && mem;
    if (row >= nrows) row = nrows - 1;
    const bool padLane = q * 8 >= a.D;
    const int W1 = a.W1, SW2 = a.SW2;
    const size_t rowBase = (size_t)row * W1 * DP + (mem ? q * 8 : 0);
    const uint16_t* __restrict__ vs = a.VS + rowBase;
    uint16_t* __restrict__ cp = a.C + rowBase;
    uint16_t* __restrict__ sp = a.S + rowBase;
    uint8_t* __restrict__ sp8 = reinterpret_cast<uint8_t*>(a.S) + rowBase;      // S8: one byte per cell, same indexing

    // Stream element t = VS[clamp(t - SW2)], t >= 0.  The window of step xi is t in [xi, xi + bs): it gains
    // t = xi + bs and loses t = xi.  Ring slot of t is t mod R with R = bs + PFD, so the element fetched at step
    // xi (t = xi + bs + PFD) lands in the slot of the element that has just left.
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint4* ring = reinterpret_cast<uint4*>(smem_raw) + threadIdx.x;
    const int bs = 2 * SW2 + 1, R = bs + H1_PFD;
    auto src = [&](int t) { return vs + min(max(t - SW2, 0), W1 - 1) * DP; };
    for (int t = 0; t < bs; ++t) cp_async16(ring + t * 128, src(t));
    cp_async_commit();
#pragma unroll
    for (int k = 0; k < H1_PFD; ++k) { cp_async16(ring + (bs + k) * 128, src(bs + k)); cp_async_commit(); }
    // (lanes beyond the pixel stride read the first lane's data: valid addresses, values unused)
    cp_async_wait<H1_PFD>();
    uint4 hs = make_uint4(0, 0, 0, 0);
    for (int t = 0; t < bs; ++t) {
        const uint4 v = ring[t * 128];
        hs.x += v.x; hs.y += v.y; hs.z += v.z; hs.w += v.w;
    }
    unsigned L[4], mm;
    reset_state<PAD>(L, mm, padLane);
    int sOut = 0, sIn = bs;                         // slots of t = xi and t = xi + bs
    for (int xi = 0; xi < W1; ++xi) {
        cp_async_wait<H1_PFD - 1>();                // the group issued H1_PFD steps ago (t = xi + bs) has landed
        const uint4 od = ring[sOut * 128];
        const uint4 nx = ring[sIn * 128];
        cp_async16(ring + sOut * 128, src(xi + bs + H1_PFD));
        cp_async_commit();
        if (++sOut == R) sOut = 0;
        if (++sIn == R) sIn = 0;
        sgm_step<G, PAD>(L, mm, hs, a.P1P1, a.P2P2, q, padLane);
        if (active) {
            st128(cp + xi * DP, hs);
            if (S8) {
                // L - C is in [0, P2] for every disparity (no borrow between the halves): keep the low bytes
                const unsigned e0 = L[0] - hs.x, e1 = L[1] - hs.y, e2 = L[2] - hs.z, e3 = L[3] - hs.w;
                *reinterpret_cast<uint2*>(sp8 + xi * DP) = make_uint2(__byte_perm(e0, e1, 0x6420), __byte_perm(e2, e3, 0x6420));
            } else {
                st128(sp + xi * DP, make_uint4(L[0], L[1], L[2], L[3]));
            }
        }
        hs.x += nx.x - od.x; hs.y += nx.y - od.y; hs.z += nx.z - od.z; hs.w += nx.w - od.w;
    }
    cp_async_wait<0>();
}

// K3b: vertical / diagonal paths, one direction per launch (generic fallback when the fused sweep below does
// not fit in shared memory).  One lane group follows one path line through the frame: the vertical line of
// column g, or the diagonal that starts at column g and wraps around the cost domain (a wrap is exactly an
// off-domain predecessor, so the state is reset there).  No inter-thread communication.
//   dxs: x offset of the predecessor (-1, 0, +1);  bottomUp: predecessor row is y+1 instead of y-1.
template <int G, bool PAD>
__global__ void __launch_bounds__(128) k_sgbm_vdir(AggArgs a, int dxs, int bottomUp)
{
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long ncols = (long long)a.B * a.W1;
    long long col = gtid / G;
    const int q = (int)(gtid % G);
    const bool active = col < ncols;
    if (!active) col = ncols - 1;
    const int f = (int)(col / a.W1);
    int x = (int)(col % a.W1);
    const bool padLane = q * 8 >= a.D;
    const int DP = a.Dp;
    const bool mem = q * 8 < DP;
    const size_t frameBase = (size_t)f * a.H * a.W1 * DP + (mem ? q * 8 : 0);

    unsigned L[4], mm;
    reset_state<PAD>(L, mm, padLane);
    for (int yi = 0; yi < a.H; ++yi) {
        const int y = bottomUp ? a.H - 1 - yi : yi;
        const size_t off = frameBase + ((size_t)y * a.W1 + x) * DP;
        const uint4 Cc = ld128(a.C + off);
        uint4 Sc = ld128(a.S + off);
        if ((dxs < 0 && x == 0) || (dxs > 0 && x == a.W1 - 1)) reset_state<PAD>(L, mm, padLane);
        sgm_step<G, PAD>(L, mm, Cc, a.P1P1, a.P2P2, q, padLane);
        sat_acc(Sc, L);
        if (active && mem) st128(a.S + off, Sc);
        x -= dxs;
        if (x >= a.W1) x = 0;
        if (x < 0) x = a.W1 - 1;
    }
}

// K3c + K4: right-to-left path r=(+1,0) fused with winner-take-all, uniqueness, sub-pixel interpolation,
// the disp2 scatter (sequential in x per row, exactly the reference order) and the left-right check.
template <int G>
__device__ __forceinline__ bool group_any(bool v)
{
    const unsigned b = __ballot_sync(FULL, v);
    const unsigned gmask = (G == 32) ? FULL : (((1u << G) - 1u) << (((threadIdx.x & 31) / G) * G));
    return (b & gmask) != 0u;
}

// trunc(n / d) for |n| < 2^22, 0 < d < 2^20: float reciprocal estimate plus an exact two-sided correction
__device__ __forceinline__ int div_trunc_small(int n, int d)
{
    const int an = abs(n);
    int qq = __float2int_rz(__fdividef((float)an, (float)d));
    const int rem = an - qq * d;
    qq += (rem >= d) - (rem < 0);
    return n < 0 ? -qq : qq;
}

template <int G, bool PAD, bool S8>
__global__ void __launch_bounds__(128) k_sgbm_h2_wta(AggArgs a)
{
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nrows = (long long)a.B * a.H;
    long long row = gtid / G;
    const int q = (int)(gtid % G);
    const bool active = row < nrows;
    if (!active) row = nrows - 1;
    const bool padLane = q * 8 >= a.D;
    const int Dp = a.Dp;                            // pixel stride of the volumes (<= 8*G; lanes beyond it hold padding)
    const bool mem = q * 8 < Dp;
    const int W1 = a.W1;
    const size_t rowBase = (size_t)row * W1 * Dp + (mem ? q * 8 : 0);
    const uint16_t* __restrict__ cp = a.C + rowBase;
    uint16_t* __restrict__ sp = a.S + rowBase;
    const uint8_t* __restrict__ sp8 = reinterpret_cast<const uint8_t*>(a.S) + rowBase;
    uint16_t* __restrict__ sdbg = (S8 ? a.Sdbg : a.S) + rowBase;       // test hook: where the final S is stored
    int16_t* __restrict__ drow = a.disp + (size_t)row * a.W;
    int* __restrict__ d2row = a.d2 + (size_t)row * a.W;
    // disp2 entry of right-image column j: (minS << 16) | (W1-1-xi) of the best left pixel xi that maps to j.  The
    // reference scans x downwards and replaces an entry only by a strictly smaller cost, i.e. it keeps the lowest
    // cost and among equals the largest x: exactly the minimum of this key, so the scatter is an order-free
    // atomicMin and the matched disparity is recovered as xi + minX1 - j.
    constexpr unsigned D2_EMPTY = 0xffffffffu;
    if (active)
        for (int x = q; x < a.W; x += G) { drow[x] = (int16_t)a.INV; d2row[x] = (int)D2_EMPTY; }
    __syncwarp();

    unsigned L[4], mm;
    reset_state<PAD>(L, mm, padLane);
    const int umul = 100 - a.uniq;
    const unsigned kb = (unsigned)q * 8u;
    // The winner's neighbours S[best -/+ 1] are read from a shared-memory copy of the pixel's sums (any lane can address
    // any disparity there: no register picks, no index shuffles); two copies used in turn, one warp barrier per step.
    __shared__ __align__(16) uint16_t sS[2][128 * 8];
    uint16_t* smine = &sS[0][0] + threadIdx.x * 8;
    const uint16_t* spix = &sS[0][0] + (threadIdx.x / G) * G * 8;
    int alt = 0;
    // The per-pixel epilogue (parabola, division, scatter, store) is identical on all G lanes of a pixel, so it is
    // deferred: lane q keeps the winner of every G-th step and the G lanes finish G pixels at once.
    unsigned svKey = 0, svM = 0, svP = 0;
    int svX = -1, sc = 0;
    auto flush = [&]() {
        if (svX >= 0) {
            const int minS = (int)(svKey >> 16), best = (int)(svKey & 0xffffu);
            const int sm1 = (int)svM, sp1 = (int)svP;
            int v = 16 * best;
            if (best > 0 && best < a.D - 1) {
                const int den = max(sm1 + sp1 - 2 * minS, 1);
                v += div_trunc_small((sm1 - sp1) * 16 + den, 2 * den);
            }
            if (active) {
                atomicMin(reinterpret_cast<unsigned*>(d2row) + (svX + a.minX1 - best - a.minD),
                          ((unsigned)minS << 16) | (unsigned)(W1 - 1 - svX));
                drow[svX + a.minX1] = (int16_t)(v + 16 * a.minD);
            }
        }
        svX = -1;
    };
    auto step = [&](const uint4& Cq, const uint4& Sq, int xi) {
        sgm_step<G, PAD>(L, mm, Cq, a.P1P1, a.P2P2, q, padLane);
        unsigned Sf[4];
        if (S8) {
            // Sum of all paths = (n + 1) * C + byte + (L - C), n paths before this one.  With c' = min(C, ceil(32767 / (n+1)))
            // the product (n + 1) * c' plus the small excess fits 16 bits and reaches 32767 exactly when the true sum does:
            // one clamp, one multiply-add and one saturation per register instead of rebuilding S and adding L.
            const unsigned b0 = __byte_perm(Sq.x, 0, 0x4140), b1 = __byte_perm(Sq.x, 0, 0x4342);
            const unsigned b2 = __byte_perm(Sq.y, 0, 0x4140), b3 = __byte_perm(Sq.y, 0, 0x4342);
            const unsigned n1 = a.nprevPk & 0xffffu;          // n + 1
            Sf[0] = __vminu2(__vminu2(Cq.x, a.kclampPk) * n1 + (b0 + L[0] - Cq.x), MVSV_PK_MAX);
            Sf[1] = __vminu2(__vminu2(Cq.y, a.kclampPk) * n1 + (b1 + L[1] - Cq.y), MVSV_PK_MAX);
            Sf[2] = __vminu2(__vminu2(Cq.z, a.kclampPk) * n1 + (b2 + L[2] - Cq.z), MVSV_PK_MAX);
            Sf[3] = __vminu2(__vminu2(Cq.w, a.kclampPk) * n1 + (b3 + L[3] - Cq.w), MVSV_PK_MAX);
        } else {
            Sf[0] = __viaddmin_u16x2(Sq.x, L[0], MVSV_PK_MAX);
            Sf[1] = __viaddmin_u16x2(Sq.y, L[1], MVSV_PK_MAX);
            Sf[2] = __viaddmin_u16x2(Sq.z, L[2], MVSV_PK_MAX);
            Sf[3] = __viaddmin_u16x2(Sq.w, L[3], MVSV_PK_MAX);
        }
        if (PAD && padLane) Sf[0] = Sf[1] = Sf[2] = Sf[3] = MVSV_PK_MAX;
        st128(smine + alt, make_uint4(Sf[0], Sf[1], Sf[2], Sf[3]));
        if (a.storeS && active && mem) st128(sdbg + xi * Dp, make_uint4(Sf[0], Sf[1], Sf[2], Sf[3]));
        // ---- first argmin via (S << 16 | k) keys
        unsigned key = min(min((Sf[0] << 16) | kb, (Sf[0] & 0xffff0000u) | (kb + 1)),
                           min((Sf[1] << 16) | (kb + 2), (Sf[1] & 0xffff0000u) | (kb + 3)));
        key = min(key, min(min((Sf[2] << 16) | (kb + 4), (Sf[2] & 0xffff0000u) | (kb + 5)),
                           min((Sf[3] << 16) | (kb + 6), (Sf[3] & 0xffff0000u) | (kb + 7))));
        key = group_min_u32<G>(key);
        const int minS = (int)(key >> 16);
        const int best = (int)(key & 0xffffu);
        bool reject = (minS >= MVSV_MAX_COST);      // every S[d] saturated: best = -1, output stays INVALID
        // ---- neighbours of the winner for the parabola
        const int im = max(best - 1, 0), ip = min(best + 1, a.D - 1);
        __syncwarp();
        const unsigned vm = spix[alt + im], vp = spix[alt + ip];
        alt ^= 128 * 8;
        if (a.uniq > 0) {
            // Rejected when some disparity further than 1 from the winner has S * (100 - uniq) < minS * 100.  The test is
            // monotone in S (100 - uniq > 0), so the lane only needs the smallest of its sums outside best-1..best+1:
            // the (at most three) exempt positions are overwritten with 0xffff -- no real sum exceeds 0x7fff -- by a
            // packed compare of the lane's disparity indices against best-1, then one packed min tree and one multiply.
            // (A packed count of the sums below floor((minS * 100 - 1) / (100 - uniq)) was measured slower: the division
            // per step costs more than eight multiply-compares.)
            bool bad = false;
            if (umul > 0) {
                if (!(PAD && padLane)) {
                    const unsigned b1 = ((unsigned)(best - 1) & 0xffffu) * 0x10001u;    // best - 1 mod 2^16 in both halves (best may be 0)
                    unsigned mn = 0xffffffffu;
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const unsigned kk2 = (kb + 2u * r) * 0x10001u + 0x00010000u;    // (kb + 2r, kb + 2r + 1)
                        const unsigned ex = __vcmpleu2(__vsub2(kk2, b1), 0x00020002u);  // 0xffff where |k - best| <= 1
                        mn = __vminu2(mn, Sf[r] | ex);
                    }
                    const int s = (int)min(mn & 0xffffu, mn >> 16);
                    bad = s <= 0x7fff && s * umul < minS * 100;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int kk = (int)kb + j;
                    const int s = (int)((j & 1) ? (Sf[j >> 1] >> 16) : (Sf[j >> 1] & 0xffffu));
                    bad |= (!PAD || kk < a.D) && (s * umul < minS * 100) && (abs(kk - best) > 1);
                }
            }
            reject |= group_any<G>(bad);
        }
        if (sc == q) { svKey = key; svM = vm; svP = vp; svX = reject ? -1 : xi; }
        if (++sc == G) { flush(); sc = 0; }
    };
    // operands of two steps are held one pair of steps ahead, in two register sets used alternately
    uint4 CA[HPF], SA[HPF], CB[HPF], SB[HPF];
    auto fetch = [&](uint4 (&Cd)[HPF], uint4 (&Sd)[HPF], int xfirst) {
#pragma unroll
        for (int k = 0; k < HPF; ++k) {
            const int xn = max(xfirst - k, 0);
            Cd[k] = ld128(cp + xn * Dp);
            if (S8) {
                const uint2 e = *reinterpret_cast<const uint2*>(sp8 + xn * Dp);
                Sd[k] = make_uint4(e.x, e.y, 0u, 0u);
            } else {
                Sd[k] = ld128(sp + xn * Dp);
            }
        }
    };
    auto run = [&](const uint4 (&Cs)[HPF], const uint4 (&Ss)[HPF], int xfirst) {
#pragma unroll
        for (int k = 0; k < HPF; ++k)
            if (xfirst - k >= 0) step(Cs[k], Ss[k], xfirst - k);
    };
    fetch(CA, SA, W1 - 1);
    for (int x0 = W1 - 1; x0 >= 0; x0 -= 2 * HPF) {
        fetch(CB, SB, x0 - HPF);
        run(CA, SA, x0);
        fetch(CA, SA, x0 - 2 * HPF);
        run(CB, SB, x0 - HPF);
    }
    flush();
    __syncwarp();
    if (active) {
        for (int x = a.minX1 + q; x < a.maxX1; x += G) {
            const int d1 = drow[x];
            if (d1 == a.INV) continue;
            const int _d = d1 >> 4, d_ = (d1 + 15) >> 4;
            const int _x = x - _d, x_ = x - d_;
            if (_x < 0 || _x >= a.W || x_ < 0 || x_ >= a.W) continue;
            // the entries were produced by atomics (performed in L2): read them past L1
            const unsigned ea = (unsigned)__ldcg(d2row + _x), eb = (unsigned)__ldcg(d2row + x_);
            // an untouched entry reads as the reference's initial value INVALID_DISP_SCALED = (minD-1)*16, which
            // passes the `>= minD` test below once minD >= 2 (kept: it is what cv::StereoSGBM computes)
            const int da = ea == D2_EMPTY ? a.INV : (W1 - 1 - (int)(ea & 0xffffu)) + a.minX1 - _x;
            const int db = eb == D2_EMPTY ? a.INV : (W1 - 1 - (int)(eb & 0xffffu)) + a.minX1 - x_;
            if (da >= a.minD && abs(da - _d) > a.d12 && db >= a.minD && abs(db - d_) > a.d12) drow[x] = (int16_t)a.INV;
        }
    }
}

__global__ void k_fill_i16(int16_t* p, size_t n, int16_t v)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// dynamic shared memory of the cost kernel (see its layout comment)
template <int G, bool WIDE>
size_t vsum_smem_bytes(int bs, bool r8)
{
    using GE = VsGeom<G, WIDE>;
    const int LEN = 8 * GE::NV + 8;
    return (size_t)2 * 6 * 8 * LEN * 2 + (size_t)2 * GE::PX * 12 * 4 + (size_t)bs * GE::CT * (r8 ? 8 : 16) +
           (size_t)VS_RD * GE::IPL * 2 * GE::NPT * 16 + (size_t)VS_RD * GE::RPL * GE::NPT * 8;
}

template <int G, bool PAD>
cudaError_t launch_sgbm_g(Engine* c, int B)
{
    const SgbmNorm& n = c->sg;
    cudaStream_t st = c->stream;
    const size_t planeStrideR = (size_t)c->maxB * c->H * c->vsRP;
    {
        const int ncx = (c->W + PF_COLS - 1) / PF_COLS, nbands = (c->H + PF_ROWS - 1) / PF_ROWS;
        dim3 blk(PF_WARPS * 32), grd((ncx * nbands + PF_WARPS - 1) / PF_WARPS, 2 * B);
        KernelTimer kt(c, KID_SGBM_PREFILTER);
        k_sgbm_prefilter<<<grd, blk, 0, st>>>(io(c).rect[0], io(c).rect[1], c->pitch, c->W, c->H, n.ftzero, c->recL, c->plR,
                                              planeStrideR, c->vsRP, c->vsJOFF, ncx, nbands);
    }
    std::function<cudaError_t(int, int)> launch_vsum;
    int vsum_gx = 1;                                  // column strips (CTAs) of the cost kernel per frame
    auto make_vsum = [&](auto wideTag) {
        constexpr bool WIDE = decltype(wideTag)::value;
        using GE = VsGeom<G, WIDE>;
        constexpr int PX = GE::PX;
        VsArgs a;
        a.recL = c->recL; a.plR = c->plR; a.planeStrideR = planeStrideR;
        a.VS = c->VS; a.W = c->W; a.H = c->H; a.W1 = n.W1; a.D = n.D; a.Dp = n.Dp; a.minD = n.minD; a.minX1 = n.minX1;
        a.SH2 = n.SH2; a.NV = c->vsNV; a.LEN = 8 * c->vsNV + 8; a.RP = c->vsRP; a.JOFF = c->vsJOFF;
        const bool r8 = 2 * n.ftzero + 63 <= 255;
        const size_t smem = vsum_smem_bytes<G, WIDE>(2 * n.SH2 + 1, r8);
        // small batches: split the rows into bands until the grid covers the SMs (each band repeats bs-1 rows)
        const int gx = (n.W1 + PX - 1) / PX, bs = 2 * n.SH2 + 1;
        vsum_gx = gx;
        int bands = 1;
        while (bands < 8 && (long long)gx * B * (bands * 2) <= c->num_sms && c->H / (bands * 2) >= 4 * bs) bands *= 2;
        a.bandRows = (c->H + bands - 1) / bands;
        const auto kern = bands > 1 ? (r8 ? k_sgbm_vsum<G, true, true, WIDE> : k_sgbm_vsum<G, false, true, WIDE>)
                                    : (r8 ? k_sgbm_vsum<G, true, false, WIDE> : k_sgbm_vsum<G, false, false, WIDE>);
        launch_vsum = [=](int f0, int nb) {
            MVSV_TRY(smem_limit((const void*)kern, 200 * 1024));
            VsArgs v = a;
            v.recL += (size_t)f0 * c->H * c->W; v.plR += (size_t)f0 * c->H * c->vsRP; v.VS += (size_t)f0 * c->H * n.W1 * n.Dp;
            dim3 grd(gx, nb, (c->H + v.bandRows - 1) / v.bandRows);
            KernelTimer kt(c, KID_SGBM_VSUM);
            kern<<<grd, GE::THREADS, smem, st>>>(v);
            return cudaSuccess;
        };
    };
    if constexpr (G == 32) {
        if (n.vsWide) make_vsum(std::true_type());
        else make_vsum(std::false_type());
    } else {
        make_vsum(std::false_type());
    }
    AggArgs a;
    a.VS = c->VS; a.C = c->C; a.S = c->S; a.H = c->H; a.W = c->W; a.W1 = n.W1; a.D = n.D; a.Dp = n.Dp; a.SW2 = n.SW2;
    a.B = B; a.P1P1 = ((unsigned)n.P1 & 0xffffu) * 0x10001u; a.P2P2 = ((unsigned)n.P2 & 0xffffu) * 0x10001u;
    a.disp = c->disp_raw; a.d2 = c->d2; a.minD = n.minD; a.minX1 = n.minX1; a.maxX1 = n.maxX1; a.INV = n.INV;
    a.uniq = n.uniq; a.d12 = n.d12;
    a.storeS = (c->debug_flags & 1) ? 1 : 0;
    const int TPB = 128;
    const long long rowThreads = (long long)B * c->H * G, colThreads = (long long)B * n.W1 * G;
    const unsigned rowBlocks = (unsigned)((rowThreads + TPB - 1) / TPB), colBlocks = (unsigned)((colThreads + TPB - 1) / TPB);
    // the three previous-row paths: fused strip sweep (csrc/sweep.cu); independent passes only when it cannot run
    SweepPlan plan;
    {
        const int forced = (int)((c->debug_flags >> 8) & 0xff);
        if (forced != 0xff) sweep_plan(c, B, forced, &plan);
    }
    // S8: every path cost is C + e with 0 <= e <= P2, so while npaths * P2 <= 255 the S volume only carries the byte
    // sum of the e's (half the traffic of S in all three aggregation kernels); needs the sweep's lane layout
    const bool s8 = plan.NS > 0 && sweep_s8_ok(c, plan) && !(c->debug_flags & 2);
    c->last_s8 = s8;
    a.Sdbg = c->VS;
    {
        const unsigned nall = (unsigned)n.npaths, kcl = (32767u + nall - 1) / nall;     // all paths, see k_sgbm_h2_wta
        a.nprevPk = nall * 0x10001u; a.kclampPk = kcl * 0x10001u;
    }
    // Cost kernel (shared-memory / ALU bound) and first row scan (HBM bound) of different chunks of frames side by side:
    // chunk i's scan runs on the second stream while the cost kernel of chunk i + 1 runs on the engine's; joined before
    // the sweep.  About seven chunks per batch, each at least ~0.9 waves of cost-kernel CTAs (measured, ms per step --
    // cfg 2, frames per chunk 13 / 15 / 19 / 26 / all: 12.26 / 12.13 / 11.73 / 11.93 / 12.29; cfg 4, 2 / 3 / 4 / 5 / all:
    // 35.9 / 36.3 / 36.0 / 37.0 / 37.2; cfg 5, 1 / 2 / 3 / all: 78.3 / 74.3 / 76.0 / 76.2; a higher stream priority for the
    // scan: slower).
    const auto h1 = s8 ? k_sgbm_h1<G, PAD, true> : k_sgbm_h1<G, PAD, false>;
    MVSV_TRY(smem_limit((const void*)h1, 200 * 1024));
    auto launch_h1 = [&](int f0, int nb, cudaStream_t on) {
        AggArgs h = a;
        const size_t off = (size_t)f0 * c->H * n.W1 * n.Dp;
        h.VS += off; h.C += off; h.S += s8 ? off / 2 : off; h.B = nb;
        const unsigned blocks = (unsigned)(((long long)nb * c->H * G + TPB - 1) / TPB);
        KernelTimer kt(c, KID_SGBM_H1, on);
        const size_t sm = (size_t)(2 * n.SW2 + 1 + H1_PFD) * TPB * 16;
        h1<<<blocks, TPB, sm, on>>>(h);
    };
    int fpc = std::max((B + 6) / 7, (int)(0.9 * c->num_sms / vsum_gx + 0.999));   // frames per chunk
    if ((c->debug_flags >> 16) & 0xffu) fpc = (int)((c->debug_flags >> 16) & 0xffu);     // test hook: frames per chunk
    // per-kernel timing (mvsv_profile_enable) runs the kernels one after the other: a duration only means something alone
    // (MVSV_SERIAL=1 does the same for a whole process: under ncu every kernel runs alone anyway, and the chunked cost
    // kernel then shows its partial waves without the scan that fills them)
    static const bool serialEnv = [] { const char* e = getenv("MVSV_SERIAL"); return e && atoi(e) != 0; }();
    const int nchunks = (c->prof || serialEnv) ? 1 : std::min((B + fpc - 1) / fpc, (int)Engine::kMaxChunks);
    if (nchunks <= 1) {
        MVSV_TRY(launch_vsum(0, B));
        launch_h1(0, B, st);
    } else {
        for (int i = 0; i < nchunks; ++i) {
            const int f0 = i * fpc, f1 = (i + 1 == nchunks) ? B : f0 + fpc;
            MVSV_TRY(launch_vsum(f0, f1 - f0));
            MVSV_TRY(cudaEventRecord(c->ev_chunk[i], st));
            MVSV_TRY(cudaStreamWaitEvent(c->aux_stream, c->ev_chunk[i], 0));
            launch_h1(f0, f1 - f0, c->aux_stream);
        }
        MVSV_TRY(cudaEventRecord(c->ev_join, c->aux_stream));
        MVSV_TRY(cudaStreamWaitEvent(st, c->ev_join, 0));
    }
    auto vdirs = [&](int bottomUp) {
        if (plan.NS > 0) return launch_sweep(c, B, plan, bottomUp, s8);
        { KernelTimer kt(c, KID_SGBM_VDIR); k_sgbm_vdir<G, PAD><<<colBlocks, TPB, 0, st>>>(a, -1, bottomUp); }
        { KernelTimer kt(c, KID_SGBM_VDIR); k_sgbm_vdir<G, PAD><<<colBlocks, TPB, 0, st>>>(a, 0, bottomUp); }
        { KernelTimer kt(c, KID_SGBM_VDIR); k_sgbm_vdir<G, PAD><<<colBlocks, TPB, 0, st>>>(a, +1, bottomUp); }
        return cudaSuccess;
    };
    MVSV_TRY(vdirs(0));
    if (n.mode == 1) MVSV_TRY(vdirs(1));
    {
        KernelTimer kt(c, KID_SGBM_H2_WTA);
        if (s8) k_sgbm_h2_wta<G, PAD, true><<<rowBlocks, TPB, 0, st>>>(a);
        else k_sgbm_h2_wta<G, PAD, false><<<rowBlocks, TPB, 0, st>>>(a);
    }
    return cudaGetLastError();
}

}  // namespace

// Strips per frame the fused previous-row sweep uses for a full batch (reported by mvsv_get_info);
// 0 = it cannot run (volume stride differs from the sweep's lane layout, or forced off): independent passes.
int sgbm_choose_td_cluster(Engine* c)
{
    const int forced = (int)((c->debug_flags >> 8) & 0xff);
    if (forced == 0xff) return 0;
    SweepPlan p;
    sweep_plan(c, c->maxB, forced, &p);
    return p.NS;
}

// Geometry of the reversed right-image planes for the cost kernel (see k_sgbm_prefilter / k_sgbm_vsum).
// 768 compute threads for the cost kernel at D > 128 when its shared memory still fits (k_sgbm_vsum, VsGeom)
bool sgbm_vsum_wide(const SgbmNorm& n)
{
    if (n.G != 32) return false;
    return vsum_smem_bytes<32, true>(2 * n.SH2 + 1, 2 * n.ftzero + 63 <= 255) <= (size_t)200 * 1024;
}

void sgbm_plane_geometry(const SgbmNorm& n, int W, int* NV, int* RP, int* JOFF)
{
    const int PX = (n.vsWide ? 768 : vs_compute_threads(n.G)) / n.G;
    const int NE = PX - 1 + 8 * n.G;                 // entries a CTA can touch (== VsGeom<G>::NE)
    const int nv = (NE + 2 + 7) / 8;                 // == VsGeom<G>::NV
    const int K = W - PX - n.minX1 + n.minD;         // j0 = JOFF + K - xa must be a multiple of 8 (xa is)
    const int joff = PX + 8 + (((8 - ((PX + 8 + K) % 8)) % 8 + 8) % 8);
    *NV = nv; *JOFF = joff; *RP = (joff + W + nv * 8 + 16 + 7) / 8 * 8;
}

cudaError_t launch_sgbm(Engine* c, int B)
{
    const SgbmNorm& n = c->sg;
    const size_t npx = (size_t)B * c->H * c->W;
    if (n.W1 <= 0) {
        KernelTimer kt(c, KID_FILL);
        k_fill_i16<<<(unsigned)((npx + 255) / 256), 256, 0, c->stream>>>(c->disp_raw, npx, (int16_t)n.INV);
    } else {
        const bool pad = n.D != 8 * n.G;             // some lanes of a pixel's lane group hold no disparity
        cudaError_t e;
        switch (n.G) {
            case 1: e = pad ? launch_sgbm_g<1, true>(c, B) : launch_sgbm_g<1, false>(c, B); break;
            case 2: e = pad ? launch_sgbm_g<2, true>(c, B) : launch_sgbm_g<2, false>(c, B); break;
            case 4: e = pad ? launch_sgbm_g<4, true>(c, B) : launch_sgbm_g<4, false>(c, B); break;
            case 8: e = pad ? launch_sgbm_g<8, true>(c, B) : launch_sgbm_g<8, false>(c, B); break;
            case 16: e = pad ? launch_sgbm_g<16, true>(c, B) : launch_sgbm_g<16, false>(c, B); break;
            default: e = pad ? launch_sgbm_g<32, true>(c, B) : launch_sgbm_g<32, false>(c, B); break;
        }
        MVSV_TRY(e);
    }
    if (n.speckleWin > 0) {
        MVSV_TRY(launch_median(c, c->disp_raw, c->disp_med, B));
        return launch_speckle(c, c->disp_med, io(c).disp, B, n.INV, n.speckleWin, 16 * n.speckleRange);
    }
    return launch_median(c, c->disp_raw, io(c).disp, B);
}
