// Disparity::tm (reference src/disparity.cpp:25-58): per pixel, cv::matchTemplate(TM_CCORR_NORMED) of the k x k left
// block against the right image's row strip to its right, cv::minMaxLoc, x of the first maximum as a byte.
//
// One CTA per image row.  The k-row strips of both images sit in shared memory.  For an offset x every column c has
// the vertical product sum P_x(c) = sum_v L(c, v) * R(c + x, v); the correlation numerator of block j is the sum of k
// neighbouring P_x, the right block's energy B(j + x) a box sum of squared column sums computed once per row.
// The score N / sqrt(A * B) is ranked as N^2 / B with exact 128-bit integer cross-multiplication (A is constant per
// pixel), so the result does not depend on summation order.
#include "mvsv_internal.h"

namespace {

constexpr int TM_THREADS = 256;
constexpr int TM_XB = 4;          // offsets evaluated per barrier pair
constexpr int TM_MAXC = 16;       // columns per thread: W <= 4096

__device__ __forceinline__ bool tm_better(unsigned long long n, unsigned long long b, unsigned long long nb, unsigned long long bb)
{
    // n^2 * bb > nb^2 * b, all factors < 2^64 after squaring (n <= 255^2 * k^2, k <= 31)
    const unsigned long long n2 = n * n, nb2 = nb * nb;
    const unsigned long long lh = __umul64hi(n2, bb), ll = n2 * bb, rh = __umul64hi(nb2, b), rl = nb2 * b;
    return lh > rh || (lh == rh && ll > rl);
}

__global__ void __launch_bounds__(TM_THREADS)
k_tm(const uint8_t* __restrict__ left, const uint8_t* __restrict__ right, size_t pitch, int W, int H, int k,
     uint8_t* __restrict__ out, size_t opitch)
{
    extern __shared__ __align__(16) unsigned char tm_smem[];
    const int i = blockIdx.x, f = blockIdx.y, tid = threadIdx.x;
    uint8_t* Ls = tm_smem;                                   // [k][W]
    uint8_t* Rs = Ls + (size_t)k * W;                        // [k][W]
    unsigned* Bx = reinterpret_cast<unsigned*>(tm_smem + (((size_t)2 * k * W + 15) & ~(size_t)15));   // [W] box energy of right
    unsigned* P = Bx + W;                                    // [TM_XB][W]
    const uint8_t* lrow = left + ((size_t)f * H + i) * pitch;
    const uint8_t* rrow = right + ((size_t)f * H + i) * pitch;
    for (int t = tid; t < k * W; t += TM_THREADS) {
        const int v = t / W, c = t - v * W;
        Ls[t] = lrow[(size_t)v * pitch + c];
        Rs[t] = rrow[(size_t)v * pitch + c];
    }
    __syncthreads();
    // squared column sums of the right strip, then their k-wide box sums
    for (int c = tid; c < W; c += TM_THREADS) {
        unsigned s = 0;
        for (int v = 0; v < k; ++v) { const unsigned r = Rs[v * W + c]; s += r * r; }
        P[c] = s;
    }
    __syncthreads();
    for (int c = tid; c < W; c += TM_THREADS) {
        unsigned s = 0;
        for (int u = 0; u < k && c + u < W; ++u) s += P[c + u];
        Bx[c] = s;
    }
    __syncthreads();

    const int NJ = W - k;                                    // blocks j in [0, NJ)
    unsigned long long nb[TM_MAXC], bb[TM_MAXC];
    int bx[TM_MAXC];
#pragma unroll
    for (int q = 0; q < TM_MAXC; ++q) { nb[q] = 0; bb[q] = 1; bx[q] = 0; }

    for (int x0 = 0; x0 < NJ; x0 += TM_XB) {
        // column products for offsets x0 .. x0+XB-1; right column c + x must stay inside the strip (<= W-2)
        for (int c = tid; c < W; c += TM_THREADS) {
#pragma unroll
            for (int t = 0; t < TM_XB; ++t) {
                const int rc = c + x0 + t;
                unsigned s = 0;
                if (rc < W - 1)
                    for (int v = 0; v < k; ++v) s += (unsigned)Ls[v * W + c] * (unsigned)Rs[v * W + rc];
                P[t * W + c] = s;
            }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < TM_MAXC; ++q) {
            const int j = tid + q * TM_THREADS;
            if (j < NJ) {
#pragma unroll
                for (int t = 0; t < TM_XB; ++t) {
                    const int x = x0 + t;
                    if (x < NJ - j) {
                        unsigned long long n = 0;
                        for (int u = 0; u < k; ++u) n += P[t * W + j + u];
                        const unsigned long long b = Bx[j + x];
                        if (tm_better(n, b, nb[q], bb[q])) { nb[q] = n; bb[q] = b; bx[q] = x; }
                    }
                }
            }
        }
        __syncthreads();
    }
    uint8_t* orow = out + ((size_t)f * H + i) * opitch;
#pragma unroll
    for (int q = 0; q < TM_MAXC; ++q) {
        const int j = tid + q * TM_THREADS;
        if (j < NJ) orow[j] = (uint8_t)bx[q];
    }
}

}  // namespace

size_t tm_smem_bytes(int W, int k)
{
    return (((size_t)2 * k * W + 15) & ~(size_t)15) + (size_t)(1 + TM_XB) * W * sizeof(unsigned);
}

int tm_max_width() { return TM_THREADS * TM_MAXC; }

// out: [B][H][opitch] bytes, zero-filled by the caller
cudaError_t launch_tm(Engine* c, int B, int k, uint8_t* out, size_t opitch)
{
    const size_t smem = tm_smem_bytes(c->W, k);
    MVSV_TRY(smem_limit((const void*)k_tm, (int)smem));
    dim3 grd(c->H - k, B);
    KernelTimer kt(c, KID_TM);
    k_tm<<<grd, TM_THREADS, smem, c->stream>>>(io(c).rect[0], io(c).rect[1], c->pitch, c->W, c->H, k, out, opitch);
    return cudaGetLastError();
}
