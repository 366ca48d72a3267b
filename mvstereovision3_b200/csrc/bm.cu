// StereoBM (PREFILTER_XSOBEL, minDisparity 0) on sm_100a -- replaces cv::StereoBM::compute behind
// Disparity::bm (reference src/disparity.cpp:18-22, parameters configs/bm.yml).  Semantics: SURVEY.md A.4.
//
//   pre[img][B][H][pitch] u8        : x-Sobel prefiltered images                                   (k_bm_prefilter)
//   tex[B][H][W] int                : window sums of |L - cap| (texture)                           (k_bm_tex_w / k_bm_tex)
//   col[B][H][width1][D] u16 or u8  : column sums  sum_dy |L[y+dy][x'+lofs] - R[y+dy][x'+k]|       (k_bm_colsum)
//                                     one byte per cell while blockSize * 2 * cap <= 255 (configs/bm.yml: 84)
// The horizontal window sum of `col`, winner-take-all, texture / uniqueness tests and the sub-pixel step are fused in
// one row-marching kernel (k_bm_wta) that reads every column of the volume from HBM once (window ring in shared
// memory).  DESIGN.md section 4 "StereoBM" has the measurements behind each choice.
#include "mvsv_internal.h"

#include <algorithm>

namespace {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Prefilter (x-Sobel, clipped to [-cap, cap], + cap).  The reference walks the rows in pairs; written out, every row is
// out[y] = clip(d[y-1] + 2 d[y] + d[y+1]) with d[r] = p[r][x+1] - p[r][x-1], rows reflected at the top and the bottom
// (-1 -> 1, H -> H-2), the first and last column and -- when H is odd -- the last row being the constant `cap`.
// A lane owns four adjacent columns (one 32-bit load and store per row) of a band of BM_PF_ROWS rows; the neighbouring
// bytes come from the adjacent lanes' words by shuffle.  The differences are kept as packed 16-bit pairs with a bias
// of 256 (no negative halves: plain 32-bit adds / subtracts are exact), so a row costs ~7 instructions per pixel.
constexpr int BM_PF_ROWS = 32;

__global__ void __launch_bounds__(128)
k_bm_prefilter(const uint8_t* __restrict__ img0, const uint8_t* __restrict__ img1, size_t pitch, int W, int H, int cap,
               uint8_t* __restrict__ o0, uint8_t* __restrict__ o1)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int xw = blockIdx.x * 128 + lane * 4;               // first of this lane's four columns
    const int ya = (blockIdx.y * 4 + warp) * BM_PF_ROWS, yb = min(ya + BM_PF_ROWS, H);
    if (ya >= H) return;                                      // whole warps only
    const int f = blockIdx.z >> 1, im = blockIdx.z & 1;
    const bool inrow = xw < (int)pitch;                       // pitch is a multiple of 16 bytes: the whole word is inside
    const int xl = inrow ? xw : (int)pitch - 4;
    const uint8_t* img = (im ? img1 : img0) + (size_t)f * H * pitch + xl;
    uint8_t* out = (im ? o1 : o0) + (size_t)f * H * pitch + xl;
    const bool nbL = lane == 0 && xw >= 4, nbR = lane == 31 && xw + 4 < (int)pitch;
    unsigned keep = 0;                                        // bytes of inner columns (0 < x < W - 1)
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (xw + k > 0 && xw + k < W - 1) keep |= 0xffu << (8 * k);
    const unsigned capw = (unsigned)cap * 0x01010101u;
    constexpr unsigned BIAS = 0x01000100u;
    // packed biased differences of row r: (d[x0], d[x0+1]) and (d[x0+2], d[x0+3])
    auto diffs = [&](int r, unsigned& d01, unsigned& d23) {
        const uint8_t* p = img + (size_t)r * pitch;
        const unsigned w = *reinterpret_cast<const unsigned*>(p);
        unsigned wl = __shfl_up_sync(FULL, w, 1), wr = __shfl_down_sync(FULL, w, 1);
        if (nbL) wl = *reinterpret_cast<const unsigned*>(p - 4);
        if (nbR) wr = *reinterpret_cast<const unsigned*>(p + 4);
        const unsigned F = __funnelshift_l(wl, w, 8);        // bytes x0-1, x0, x0+1, x0+2
        const unsigned G = __funnelshift_r(w, wr, 24);       // bytes x0+3, x0+4, ...
        const unsigned X = __byte_perm(F, 0, 0x4140), Y = __byte_perm(F, 0, 0x4342), Z = __byte_perm(G, 0, 0x4140);
        d01 = Y + BIAS - X;
        d23 = Z + BIAS - Y;
    };
    const unsigned lo = (unsigned)(1024 - cap) * 0x10001u, hi = (unsigned)(1024 + cap) * 0x10001u;
    unsigned p01, p23, c01, c23, n01, n23;
    diffs(ya > 0 ? ya - 1 : 1, p01, p23);
    diffs(ya, c01, c23);
    for (int y = ya; y < yb; ++y) {
        diffs(y + 1 < H ? y + 1 : H - 2, n01, n23);
        const unsigned s01 = p01 + 2 * c01 + n01, s23 = p23 + 2 * c23 + n23;     // biased by 1024 per half
        const unsigned q01 = __vminu2(__vmaxu2(s01, lo), hi) - lo, q23 = __vminu2(__vmaxu2(s23, lo), hi) - lo;
        unsigned v = __byte_perm(q01, q23, 0x6420);
        v = (v & keep) | (capw & ~keep);
        if ((H & 1) && y == H - 1) v = capw;
        if (inrow) *reinterpret_cast<unsigned*>(out + (size_t)y * pitch) = v;
        p01 = c01; p23 = c23; c01 = n01; c23 = n23;
    }
}

// texture: window sum of |L - cap| over blockSize x blockSize pixels.
// k_bm_tex_w (blockSize <= 63): a warp owns 128 adjacent columns (128 - 2*w2 of them, rounded down to a multiple of
// four, produce output) and a band of BM_TEX_ROWS rows; a lane slides the vertical sums of its four columns down the
// band (VABSDIFF4 on the entering and the leaving word), the warp turns the 128 column sums of a row into inclusive
// prefix sums (three adds per lane + a shuffle scan of the lanes' totals) in its own piece of shared memory, and an
// output pixel is the difference of two of them.  No CTA barrier.
constexpr int BM_TEX_ROWS = 64;
__global__ void __launch_bounds__(128)
k_bm_tex_w(const uint8_t* __restrict__ preL, size_t pitch, int W, int H, int w2, int cap, int* __restrict__ tex)
{
    __shared__ __align__(16) int pre[4][2][132];              // [warp][copy][1 + 128]: pre[..][0] = 0 stands for P[-1]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nxw = (128 - 2 * w2) & ~3;
    const int X0 = blockIdx.x * nxw;                          // first column of this warp (a multiple of four)
    const int ya = w2 + (blockIdx.y * 4 + warp) * BM_TEX_ROWS, yb = min(ya + BM_TEX_ROWS, H - w2);
    if (ya >= yb) return;
    const int xl = min(X0 + 4 * lane, (int)pitch - 4);        // (lanes past the row feed no output)
    const uint8_t* p = preL + (size_t)blockIdx.z * H * pitch + xl;
    const unsigned capw = (unsigned)cap * 0x01010101u;
    unsigned s01 = 0, s23 = 0;                                // vertical sums of columns (0, 1) and (2, 3), packed u16x2
    for (int dy = -w2; dy <= w2; ++dy) {
        const unsigned a = __vabsdiffu4(*reinterpret_cast<const unsigned*>(p + (size_t)(ya + dy) * pitch), capw);
        s01 += __byte_perm(a, 0, 0x4140); s23 += __byte_perm(a, 0, 0x4342);
    }
    int* P = &pre[warp][0][0];
    if (lane == 0) { pre[warp][0][0] = 0; pre[warp][1][0] = 0; }
    // this lane's output columns: local index j = 4 * lane + k in [w2, w2 + nxw), x = X0 + j < W - w2
    const int j0 = 4 * lane;
    int* o = tex + ((size_t)blockIdx.z * H + ya) * W + X0 + j0;
    const uint8_t* pin = p + (size_t)(ya + w2 + 1) * pitch;   // rows entering / leaving the window of the next output row
    const uint8_t* pout = p + (size_t)(ya - w2) * pitch;
    int alt = 0;
    for (int y = ya; y < yb; ++y) {
        unsigned e = 0, f = 0;
        if (y + 1 < yb) { e = *reinterpret_cast<const unsigned*>(pin); f = *reinterpret_cast<const unsigned*>(pout); pin += pitch; pout += pitch; }
        const int t0 = (int)(s01 & 0xffffu), t1 = t0 + (int)(s01 >> 16), t2 = t1 + (int)(s23 & 0xffffu), t3 = t2 + (int)(s23 >> 16);
        int v = t3;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int u = __shfl_up_sync(FULL, v, d);
            if (lane >= d) v += u;
        }
        const int off = v - t3;                               // sum of the lanes to the left
        int* Pc = P + alt * 132 + 1;
        Pc[j0] = off + t0; Pc[j0 + 1] = off + t1; Pc[j0 + 2] = off + t2; Pc[j0 + 3] = off + t3;
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int j = j0 + k;
            if (j >= w2 && j < w2 + nxw && X0 + j < W - w2) o[k] = Pc[j + w2] - Pc[j - w2 - 1];
        }
        alt ^= 1;                                             // the next row writes the other copy: one warp barrier per row
        o += W;
        const unsigned ae = __vabsdiffu4(e, capw), af = __vabsdiffu4(f, capw);
        s01 += __byte_perm(ae, 0, 0x4140) - __byte_perm(af, 0, 0x4140);
        s23 += __byte_perm(ae, 0, 0x4342) - __byte_perm(af, 0, 0x4342);
    }
}

// k_bm_tex (any blockSize): one CTA = 256 adjacent columns (256 - 2*w2 of them produce output) x BM_TEX_ROWS rows: a
// thread slides the vertical sum of its column down the band; per row the CTA turns the 256 column sums into inclusive
// prefix sums (shuffle scan per warp + the warps' totals) and an output pixel is the difference of two of them.
__global__ void __launch_bounds__(256)
k_bm_tex(const uint8_t* __restrict__ preL, size_t pitch, int W, int H, int w2, int cap, int* __restrict__ tex)
{
    __shared__ int pre[2][256];
    __shared__ int wtot[2][8];
    const int t = threadIdx.x, lane = t & 31, wp = t >> 5;
    const int nx = 256 - 2 * w2;
    const int x0 = w2 + blockIdx.x * nx;                      // first output column of this CTA
    const int xc = min(x0 - w2 + t, W - 1);                   // this thread's column (clamped: the excess feeds no output)
    const int ya = w2 + blockIdx.y * BM_TEX_ROWS, yb = min(ya + BM_TEX_ROWS, H - w2);
    const uint8_t* p = preL + (size_t)blockIdx.z * H * pitch + xc;
    int s = 0;
    for (int dy = -w2; dy <= w2; ++dy) s += abs((int)p[(size_t)(ya + dy) * pitch] - cap);
    const bool outp = t < nx && x0 + t < W - w2;
    int* o = tex + ((size_t)blockIdx.z * H + ya) * W + x0 + t;
    const uint8_t* pin = p + (size_t)(ya + w2 + 1) * pitch;   // row entering / leaving the window of the next output row
    const uint8_t* pout = p + (size_t)(ya - w2) * pitch;
    int e = 0, f = 0;
    for (int y = ya; y < yb; ++y) {
        const int b = (y - ya) & 1;
        if (y + 1 < yb) { e = *pin; f = *pout; pin += pitch; pout += pitch; }    // requested before the scan
        int v = s;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int u = __shfl_up_sync(FULL, v, d);
            if (lane >= d) v += u;
        }
        if (lane == 31) wtot[b][wp] = v;
        __syncthreads();
        int off = 0;
#pragma unroll
        for (int k = 0; k < 7; ++k) off += (k < wp) ? wtot[b][k] : 0;
        pre[b][t] = v + off;
        __syncthreads();
        if (outp) *o = pre[b][t + 2 * w2] - (t > 0 ? pre[b][t - 1] : 0);
        o += W;
        s += abs(e - cap) - abs(f - cap);
    }
}

// column sums: lane (x', q) owns the eight disparity indices k = 8q..8q+7 of column x' and marches down the valid
// rows with a sliding sum.  The eight right-image bytes start at an arbitrary byte address, so they are cut out of
// three aligned words with PRMT (the selector is constant per thread); |L - R| is VABSDIFF4 on four bytes at once,
// widened to packed u16x2 for the running sums; one 128-bit store per row.
struct BmRaw { unsigned l, w0, w1, w2; };       // a row's operands as loaded: the left byte and three aligned right words
__device__ __forceinline__ BmRaw bm_load8(const uint8_t* __restrict__ rowL, const unsigned* __restrict__ rowR)
{
    BmRaw r; r.l = rowL[0]; r.w0 = rowR[0]; r.w1 = rowR[1]; r.w2 = rowR[2];
    return r;
}
__device__ __forceinline__ uint2 bm_ad8(const BmRaw& r, unsigned sel)
{
    const unsigned lb = r.l * 0x01010101u;
    return make_uint2(__vabsdiffu4(lb, __byte_perm(r.w0, r.w1, sel)), __vabsdiffu4(lb, __byte_perm(r.w1, r.w2, sel)));
}
__device__ __forceinline__ uint2 bm_ad8(const uint8_t* __restrict__ rowL, const unsigned* __restrict__ rowR, unsigned sel)
{
    return bm_ad8(bm_load8(rowL, rowR), sel);
}
// acc (packed u16x2) += the eight bytes of e, -= the eight bytes of f
__device__ __forceinline__ void bm_acc(unsigned (&acc)[4], const uint2& e, const uint2& f)
{
    acc[0] += __byte_perm(e.x, 0, 0x4140) - __byte_perm(f.x, 0, 0x4140); acc[1] += __byte_perm(e.x, 0, 0x4342) - __byte_perm(f.x, 0, 0x4342);
    acc[2] += __byte_perm(e.y, 0, 0x4140) - __byte_perm(f.y, 0, 0x4140); acc[3] += __byte_perm(e.y, 0, 0x4342) - __byte_perm(f.y, 0, 0x4342);
}

// The absolute differences of the last blockSize rows stay in a per-thread shared-memory ring (8 bytes per row), so
// the row that leaves the window is not evaluated a second time.
// Threads are numbered (column, octet) with exactly D / 8 octets per column -- not a power of two as in the row scans, so
// no lane idles at D = 80 -- and consecutive threads store consecutive pieces of the volume.
// B8 (blockSize * 2 * cap <= 255, e.g. bm.yml: 21 * 4 = 84): a column sum fits a byte, so the volume is stored as one
// byte per cell and the running sums stay packed four to a register: acc - f + e is exact as plain 32-bit arithmetic
// because every byte of the result is a window sum in 0..255 (no carry leaves a byte).
template <bool B8>
__global__ void __launch_bounds__(128) k_bm_colsum(const uint8_t* __restrict__ preL, const uint8_t* __restrict__ preR,
                                                   size_t pitch, int H, int width1, int D, int lofs, int w2,
                                                   uint16_t* __restrict__ col)
{
    extern __shared__ uint2 bm_ring[];          // [bs][128]
    const int Dp = D;           // pixel stride of the column-sum volume: numDisp (a multiple of 16)
    const int nOct = D >> 3;
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
    const int xp = gtid / nOct, q = gtid - xp * nOct;
    if (xp >= width1) return;
    const size_t fo = (size_t)blockIdx.y * H * pitch;
    const uint8_t* pl = preL + fo + xp + lofs;
    const size_t ra = fo + xp + q * 8;                       // byte address of R[.][x' + 8q]
    const unsigned* pr = reinterpret_cast<const unsigned*>(preR + (ra & ~(size_t)3));
    const unsigned sel = 0x3210u + 0x1111u * (unsigned)(ra & 3);
    const size_t pw = pitch / 4;                             // pitch is a multiple of 16 bytes
    const int bs = 2 * w2 + 1;
    uint2* ring = bm_ring + threadIdx.x;
    unsigned acc[4] = {0, 0, 0, 0};
    uint2 acc8 = make_uint2(0u, 0u);
    for (int y = 0; y < bs; ++y) {
        const uint2 e = bm_ad8(pl + (size_t)y * pitch, pr + (size_t)y * pw, sel);
        ring[y * 128] = e;
        if (B8) { acc8.x += e.x; acc8.y += e.y; }
        else bm_acc(acc, e, make_uint2(0u, 0u));
    }
    const size_t cell0 = ((size_t)blockIdx.y * H * width1 + xp) * Dp + q * 8, rowCells = (size_t)width1 * Dp;
    uint16_t* out = col + cell0 + (size_t)w2 * rowCells;
    uint8_t* out8 = reinterpret_cast<uint8_t*>(col) + cell0 + (size_t)w2 * rowCells;
    // The operands of the entering rows are requested two rows ahead (each row's loads would otherwise be waited for
    // on the spot: ncu showed 24 of 25 stall cycles on the long scoreboard); rows past the image repeat the last one.
    pl += (size_t)(bs - 1) * pitch; pr += (size_t)(bs - 1) * pw;
    const int lastIn = H - 1;                                // last row that ever enters
    int yin = bs - 1;
    if (yin < lastIn) { pl += pitch; pr += pw; ++yin; }
    BmRaw r0 = bm_load8(pl, pr);
    if (yin < lastIn) { pl += pitch; pr += pw; ++yin; }
    BmRaw r1 = bm_load8(pl, pr);
    int slot = 0;                                            // ring slot of the oldest row (y - w2)
    // one output row; `cur` holds the operands of the row that enters and is refilled for the row two further down
    // (two named register sets used in turn: a rotation through moves would wait for the loads it has just issued)
    auto row = [&](int y, BmRaw& cur) {
        if (B8) { *reinterpret_cast<uint2*>(out8) = acc8; out8 += rowCells; }
        else { st128(out, make_uint4(acc[0], acc[1], acc[2], acc[3])); out += rowCells; }
        if (y + 1 < H - w2) {
            const uint2 e = bm_ad8(cur, sel);
            if (yin < lastIn) { pl += pitch; pr += pw; ++yin; }
            cur = bm_load8(pl, pr);
            const uint2 f = ring[slot * 128];
            ring[slot * 128] = e;
            if (B8) { acc8.x += e.x - f.x; acc8.y += e.y - f.y; }
            else bm_acc(acc, e, f);
            if (++slot == bs) slot = 0;
        }
    };
    for (int y = w2; y < H - w2; y += 2) {
        row(y, r0);
        if (y + 1 < H - w2) row(y + 1, r1);
    }
}

struct BmArgs {
    const uint16_t* col; const int* tex; int16_t* disp;
    int W, H, width1, D, Dp, lofs, w2, texThr, uniq, B;
};

// Winner-take-all over the horizontal window sums of `col`.  A row of the volume is scanned left to right by NL
// adjacent lanes, each holding OPL octets (8 * OPL disparities, 4 * OPL packed registers) of the running window sum:
// with 16-bit column sums lane q holds the octets q, q + NL, ..., so that the lanes of a row touch contiguous 16-byte
// pieces; with byte column sums (B8, OPL = 2) lane q holds the sixteen disparities 16q..16q+15, one 16-byte piece.
// bm.yml (D = 80): five lanes per row, six rows per warp.  Per step and lane: the first argmin through
// (SAD << 16) | k keys (one shift-add or mask-or per value, 32-bit min3), a key exchange over the row's NL lanes, and
// the window update from the column that enters and the one that leaves.
//   RING: every column of the volume is read from HBM once.  A lane copies its pieces of column x + w2 + 1 + PF with
//   cp.async into a private shared-memory ring of blockSize + 1 + PF slots and reads both the entering and the leaving
//   column from there (without the ring the leaving column is a second HBM read 2 * w2 + 1 steps later: the rows in
//   flight hold 230 MB of window at bm.yml, twice the L2 -- ncu: 14.5 GB of DRAM reads for a 7.1 GB volume).
// The winner's neighbours S[mind -/+ 1] are read from a shared-memory copy of the row's sums (any lane of the row can
// address any disparity there, no register indexing; two copies used in turn: one warp barrier per step).  The
// per-pixel epilogue (texture test, sub-pixel division, store) is identical on the lanes of a row, so it is deferred:
// lane q keeps the winner of every NL-th step and the lanes of a row finish NL pixels at once; the texture value of a
// lane's pixel is requested one round ahead.  COST: the epilogue also stores the winner's SAD in cost[B][H][W] (the
// left-right check's cost; a parameter of its own after the others, so that the kernels without it stay as they were).
constexpr int BM_PF = 3;       // columns in flight ahead of the window (RING)

template <int OPL, bool RING, bool B8, bool COST>
__global__ void __launch_bounds__(256) k_bm_wta(BmArgs a, int ringSlots, int sumsPerWarp, int* __restrict__ cost)
{
    static_assert(!B8 || OPL == 2, "byte volume: sixteen disparities per lane");
    constexpr int NR = 4 * OPL;                                // packed registers per lane
    constexpr int PC = B8 ? 1 : OPL;                           // 16-byte pieces per lane and column
    extern __shared__ __align__(16) unsigned char bm_smem[];
    // layout: sums[2 copies][warps][sumsPerWarp = RW rows x (D + 8), rounded up to 8] u16 | ring[slots][PC][threads] uint4
    const int nthr = blockDim.x, nwarps = nthr >> 5;
    uint16_t* sums = reinterpret_cast<uint16_t*>(bm_smem);
    uint4* ring = reinterpret_cast<uint4*>(bm_smem + (size_t)2 * nwarps * sumsPerWarp * sizeof(uint16_t)) + threadIdx.x;
    const int nOct = a.D >> 3, NL = nOct / OPL, RW = 32 / NL;  // lanes per row, rows per warp
    const int lane = threadIdx.x & 31, rw = lane / NL, q = lane - rw * NL;
    const int vrows = a.H - 2 * a.w2;
    const long long nrows = (long long)a.B * vrows;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    long long r = warp * RW + rw;
    const bool active = rw < RW && r < nrows;
    if (r >= nrows) r = nrows - 1;
    const int base = min(rw, RW - 1) * NL;                     // first lane of this row's segment
    const int f = (int)(r / vrows), y = (int)(r % vrows) + a.w2;
    // byte offsets into the volume: this lane's first piece of column 0, the next piece, the next column
    const int esz = B8 ? 1 : 2;
    const size_t rowBase = (((size_t)f * a.H + y) * a.width1 * a.Dp + q * (B8 ? 16 : 8)) * esz;
    const unsigned char* cp = reinterpret_cast<const unsigned char*>(a.col) + (rw < RW ? rowBase : 0);
    const int pstep = NL * 16;                                 // bytes between a lane's pieces (16-bit volume)
    const size_t cstep = (size_t)a.Dp * esz;                   // bytes between columns
    const int k00 = B8 ? q * 16 : q * 8, kstep = B8 ? 8 : NL * 8;      // first disparity of octet o: k00 + o * kstep
    const size_t outRow = ((size_t)f * a.H + y) * a.W;
    const int bs = 2 * a.w2 + 1;
    uint16_t* rowsm = sums + (size_t)(threadIdx.x >> 5) * sumsPerWarp + min(rw, RW - 1) * (a.D + 8);
    uint16_t* mine = rowsm + k00;
    const int sumsAlt = nwarps * sumsPerWarp;                  // second copy of the sums area: steps alternate

    // w (a column's pieces) added to / taken off the packed sums
    auto addcol = [&](unsigned (&hs)[NR], const uint4 (&w)[PC]) {
        if (B8) {
            hs[0] += __byte_perm(w[0].x, 0, 0x4140); hs[1] += __byte_perm(w[0].x, 0, 0x4342);
            hs[2] += __byte_perm(w[0].y, 0, 0x4140); hs[3] += __byte_perm(w[0].y, 0, 0x4342);
            hs[4] += __byte_perm(w[0].z, 0, 0x4140); hs[5] += __byte_perm(w[0].z, 0, 0x4342);
            hs[6] += __byte_perm(w[0].w, 0, 0x4140); hs[7] += __byte_perm(w[0].w, 0, 0x4342);
        } else {
#pragma unroll
            for (int o = 0; o < PC; ++o) { hs[4 * o] += w[o].x; hs[4 * o + 1] += w[o].y; hs[4 * o + 2] += w[o].z; hs[4 * o + 3] += w[o].w; }
        }
    };
    auto subcol = [&](unsigned (&hs)[NR], const uint4 (&w)[PC]) {
        if (B8) {
            hs[0] -= __byte_perm(w[0].x, 0, 0x4140); hs[1] -= __byte_perm(w[0].x, 0, 0x4342);
            hs[2] -= __byte_perm(w[0].y, 0, 0x4140); hs[3] -= __byte_perm(w[0].y, 0, 0x4342);
            hs[4] -= __byte_perm(w[0].z, 0, 0x4140); hs[5] -= __byte_perm(w[0].z, 0, 0x4342);
            hs[6] -= __byte_perm(w[0].w, 0, 0x4140); hs[7] -= __byte_perm(w[0].w, 0, 0x4342);
        } else {
#pragma unroll
            for (int o = 0; o < PC; ++o) { hs[4 * o] -= w[o].x; hs[4 * o + 1] -= w[o].y; hs[4 * o + 2] -= w[o].z; hs[4 * o + 3] -= w[o].w; }
        }
    };

    int rot[4];                                                // the other lanes of a five-lane row
#pragma unroll
    for (int k = 0; k < 4; ++k) rot[k] = min(base + (q + k + 1) % NL, 31);
    unsigned hs[NR];
#pragma unroll
    for (int i = 0; i < NR; ++i) hs[i] = 0;
    for (int j = 0; j < bs; ++j) {
        uint4 w[PC];
#pragma unroll
        for (int o = 0; o < PC; ++o) {
            w[o] = ld128(cp + (size_t)j * cstep + o * pstep);
            if (RING) ring[(j * PC + o) * nthr] = w[o];
        }
        addcol(hs, w);
    }
    const int xEnd = a.width1 - a.w2;
    // ring slots (in uint4 units of this lane): column bs + t enters, column t leaves, column bs + BM_PF + t is requested
    const int slotStride = PC * nthr, ringLen = ringSlots * slotStride;
    int sIn = (bs % ringSlots) * slotStride, sOut = 0, sReq = ((bs + BM_PF) % ringSlots) * slotStride;
    if (RING) {
#pragma unroll
        for (int k = 0; k < BM_PF; ++k) {
            if (bs + k < a.width1) {
#pragma unroll
                for (int o = 0; o < PC; ++o)
                    cp_async16(ring + ((bs + k) % ringSlots) * slotStride + o * nthr, cp + (size_t)(bs + k) * cstep + o * pstep);
            }
            cp_async_commit();
        }
    }
    unsigned svKey = 0, svP = 0, svN = 0;
    int svX = -1, sc = 0;
    // texture of the pixel this lane finishes in the current round, and of the next round's
    const int* tp = a.tex + outRow + a.lofs;
    int texCur = tp[min(a.w2 + q, xEnd - 1)], texNext = 0;
    auto flush = [&]() {
        if (svX >= 0 && active && texCur >= a.texThr) {
            const int minsad = (int)(svKey >> 16), mind = (int)(svKey & 0xffffu);
            const int p = (int)svP, n = (int)svN;
            const int den = p + n - 2 * minsad + abs(p - n);
            a.disp[outRow + svX] = (int16_t)((((a.D - 1 - mind) * 256) + (den != 0 ? (p - n) * 256 / den : 0) + 15) >> 4);
            if (COST) cost[outRow + svX] = minsad;
        }
        svX = -1;
    };
    // running pointers to the columns requested / entering / leaving
    const unsigned char* pn = cp + (size_t)(RING ? bs + BM_PF : bs) * cstep;
    const unsigned char* po = cp;
    int colReq = bs + BM_PF, alt = 0;
    for (int xp = a.w2; xp < xEnd; ++xp) {
        uint4 nx[PC], od[PC];
        if (RING) {
            if (colReq < a.width1) {
#pragma unroll
                for (int o = 0; o < PC; ++o) cp_async16(ring + sReq + o * nthr, pn + o * pstep);
            }
            cp_async_commit();
            ++colReq;
            sReq += slotStride; if (sReq == ringLen) sReq = 0;
            cp_async_wait<BM_PF>();                            // column bs + t (requested BM_PF steps ago) has landed
#pragma unroll
            for (int o = 0; o < PC; ++o) { nx[o] = ring[sIn + o * nthr]; od[o] = ring[sOut + o * nthr]; }
            sIn += slotStride; if (sIn == ringLen) sIn = 0;
            sOut += slotStride; if (sOut == ringLen) sOut = 0;
        } else if (xp + 1 < xEnd) {
#pragma unroll
            for (int o = 0; o < PC; ++o) { nx[o] = ld128(pn + o * pstep); od[o] = ld128(po + o * pstep); }
        } else {
#pragma unroll
            for (int o = 0; o < PC; ++o) nx[o] = od[o] = make_uint4(0, 0, 0, 0);
        }
        pn += cstep; po += cstep;
        if (sc == 0) texNext = tp[min(xp + NL + q, xEnd - 1)];
#pragma unroll
        for (int o = 0; o < OPL; ++o)
            if (rw < RW) st128(mine + alt + o * kstep, make_uint4(hs[4 * o], hs[4 * o + 1], hs[4 * o + 2], hs[4 * o + 3]));
        // first argmin: keys (SAD << 16) | k
        unsigned kq[OPL * 2];
#pragma unroll
        for (int o = 0; o < OPL; ++o) {
            const unsigned k0 = (unsigned)(k00 + o * kstep);
            kq[2 * o] = __vimin3_u32((hs[4 * o] << 16) + k0, (hs[4 * o] & 0xffff0000u) | (k0 + 1), (hs[4 * o + 1] << 16) + (k0 + 2));
            kq[2 * o] = __vimin3_u32(kq[2 * o], (hs[4 * o + 1] & 0xffff0000u) | (k0 + 3), (hs[4 * o + 2] << 16) + (k0 + 4));
            kq[2 * o + 1] = __vimin3_u32((hs[4 * o + 2] & 0xffff0000u) | (k0 + 5), (hs[4 * o + 3] << 16) + (k0 + 6),
                                         (hs[4 * o + 3] & 0xffff0000u) | (k0 + 7));
        }
        unsigned key = min(kq[0], kq[1]);
#pragma unroll
        for (int o = 1; o < OPL; ++o) key = __vimin3_u32(key, kq[2 * o], kq[2 * o + 1]);
        if (NL == 5) {
            // all-to-all over the row's five lanes: four independent shuffles instead of a ladder of three plus a broadcast
            const unsigned k1 = __shfl_sync(FULL, key, rot[0]), k2 = __shfl_sync(FULL, key, rot[1]);
            const unsigned k3 = __shfl_sync(FULL, key, rot[2]), k4 = __shfl_sync(FULL, key, rot[3]);
            key = __vimin3_u32(__vimin3_u32(key, k1, k2), k3, k4);
        } else {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                if (o < NL) {                                  // warp-uniform
                    const unsigned other = __shfl_down_sync(FULL, key, o);
                    if (q + o < NL) key = min(key, other);
                }
            }
            if (NL > 1) key = __shfl_sync(FULL, key, base);
        }
        __syncwarp();                                          // the row's sums are in shared memory
        const int minsad = (int)(key >> 16), mind = (int)(key & 0xffffu);
        const int ip = (mind + 1 < a.D) ? mind + 1 : a.D - 2;
        const int in = (mind > 0) ? mind - 1 : 1;
        const unsigned vp = rowsm[alt + ip], vn = rowsm[alt + in];
        alt ^= sumsAlt;                                        // the next step writes the other copy: one warp barrier per step
        bool reject = false;
        if (a.uniq > 0) {
            // another disparity outside mind-1..mind+1 within the margin: count the lane's sums <= thresh and take off
            // those of the three exempt positions that lie in this lane's octets (mind itself always counts)
            const int thresh = minsad + (minsad * a.uniq / 100);
            const unsigned t2 = (unsigned)min(thresh, 0xffff) * 0x10001u;
            unsigned cnt2 = 0;
#pragma unroll
            for (int i = 0; i < NR; ++i) cnt2 += __vsetleu2(hs[i], t2);
            const int cnt = (int)((cnt2 & 0xffffu) + (cnt2 >> 16));
            auto minelane = [&](int k) -> bool { return (B8 ? (k >> 4) : ((k >> 3) % NL)) == q; };
            int exempt = minelane(mind) ? 1 : 0;
            if (mind > 0 && minelane(mind - 1) && (int)vn <= thresh) ++exempt;
            if (mind + 1 < a.D && minelane(mind + 1) && (int)vp <= thresh) ++exempt;
            const unsigned bal = __ballot_sync(FULL, cnt > exempt && rw < RW);
            const unsigned gmask = (NL == 32) ? FULL : (((1u << NL) - 1u) << base);
            reject = (bal & gmask) != 0u;
        }
        if (sc == q) { svKey = key; svP = vp; svN = vn; svX = reject ? -1 : xp + a.lofs; }
        if (++sc == NL) { flush(); sc = 0; texCur = texNext; }
        addcol(hs, nx);
        subcol(hs, od);
    }
    if (RING) cp_async_wait<0>();
    flush();
}

static int bm_sums_per_warp(int D, int opl) { return ((32 / ((D / 8) / opl)) * (D + 8) + 7) / 8 * 8; }
// shared memory of one warp: two copies of its rows' sums + its lanes' ring
static size_t bm_wta_warp_smem(int D, int opl, int pieces, int slots) { return (size_t)2 * bm_sums_per_warp(D, opl) * 2 + (size_t)slots * pieces * 32 * 16; }
// warps per CTA (2..8) that put the most warps on an SM (228 KB, 1 KB reserved per CTA); 0 = not even two warps fit
static int bm_wta_cta_warps(size_t warpBytes, int* warpsPerSm)
{
    int best = 0, bestTotal = 0;
    const int order[] = {4, 5, 6, 3, 7, 8, 2};
    for (int nw : order) {
        const size_t cta = nw * warpBytes + 1024;
        if (nw * warpBytes > 226 * 1024) continue;
        const int total = std::min(64, (int)(228 * 1024 / cta) * nw);
        if (total > bestTotal) { bestTotal = total; best = nw; }
    }
    *warpsPerSm = bestTotal;
    return best;
}

template <int OPL, bool RING, bool B8>
static cudaError_t launch_bm_wta(Engine* c, const BmArgs& a, int* cost, int ringSlots, int ctaWarps)
{
    const int NL = (a.D / 8) / OPL, rowsPerWarp = 32 / NL;
    const long long warps = ((long long)a.B * (a.H - 2 * a.w2) + rowsPerWarp - 1) / rowsPerWarp;
    const auto k = cost ? k_bm_wta<OPL, RING, B8, true> : k_bm_wta<OPL, RING, B8, false>;
    MVSV_TRY(smem_limit((const void*)k, 226 * 1024));
    const size_t smem = ctaWarps * bm_wta_warp_smem(a.D, OPL, B8 ? 1 : OPL, RING ? ringSlots : 0);
    k<<<(unsigned)((warps + ctaWarps - 1) / ctaWarps), ctaWarps * 32, smem, c->stream>>>(a, ringSlots, bm_sums_per_warp(a.D, OPL), cost);
    return cudaGetLastError();
}

// Left-right check of cv::StereoBM (disp12MaxDiff >= 0; semantics SURVEY.md A.4), in place on the x16 map, one CTA per
// row.  cv::StereoBM matches the whole width1 domain, X in [D - 1, W), and runs the check before it clears the columns
// outside the valid rectangle, so the border pixels X in [D, D - 1 + w2) and [W - w2, W) take part in the scatter
// although they end up FILTERED.  The WTA does not evaluate them: phase 1 does, one warp per pixel, from the column
// sums (clamped at the right edge) and, left of column 0 of the volume, from column sums of the clamped left pixel
// against R[0 .. D - 1].  The scatter "x ascending, keep the first strict minimum of the cost at x2" is an atomicMin
// of the keys (cost << 12) | x in shared memory; after one barrier every valid pixel checks itself against the table.
constexpr int BM_LR_THREADS = 256;
constexpr int BM_LR_MAXW = 4096;                                // 12-bit x in the keys; 16 KB of keys

template <bool B8>
__global__ void __launch_bounds__(BM_LR_THREADS)
k_bm_lrcheck(int16_t* __restrict__ disp, const int* __restrict__ cost, const uint16_t* __restrict__ col,
             const uint8_t* __restrict__ preL, const uint8_t* __restrict__ preR, size_t pitch, int W, int H, int width1,
             int D, int w2, int cap, int texThr, int uniq, int d12)
{
    __shared__ unsigned keys[BM_LR_MAXW];
    __shared__ int16_t rowd[BM_LR_MAXW];
    __shared__ int sads[BM_LR_THREADS / 32][256];
    const int f = blockIdx.y, y = blockIdx.x + w2, lofs = D - 1;
    const int xlo = lofs + w2, xhi = W - w2;                  // valid rectangle
    const int FILT = -16;
    const size_t row = ((size_t)f * H + y) * W;
    int16_t* drow = disp + row;
    for (int x = threadIdx.x; x < W; x += BM_LR_THREADS) { keys[x] = 0xffffffffu; rowd[x] = drow[x]; }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // phase 1: the border pixels (w2 - 1 on the left, w2 on the right); x is the column in the width1 domain
    const int nLeft = w2 - 1, nb = nLeft + w2;
    const unsigned char* vol = reinterpret_cast<const unsigned char*>(col);
    const size_t volRow = ((size_t)f * H + y) * width1;
    const uint8_t* pl = preL + (size_t)f * H * pitch;
    const uint8_t* pr = preR + (size_t)f * H * pitch;
    int* sad = sads[warp];
    for (int i = warp; i < nb; i += BM_LR_THREADS / 32) {
        const int X = i < nLeft ? D + i : xhi + (i - nLeft), x = X - lofs;
        int tex = 0;
        for (int t = lane; t < (2 * w2 + 1) * (2 * w2 + 1); t += 32) {
            const int dy = t / (2 * w2 + 1) - w2, dx = t % (2 * w2 + 1) - w2;
            tex += abs((int)pl[(size_t)(y + dy) * pitch + min(max(X + dx, 0), W - 1)] - cap);
        }
        tex = __reduce_add_sync(FULL, tex);
        unsigned best = 0xffffffffu;
        for (int k = lane; k < D; k += 32) {
            int s = 0;
            for (int j = x - w2; j <= x + w2; ++j) {
                if (j >= 0) {
                    const size_t cell = (volRow + min(j, width1 - 1)) * D + k;
                    s += B8 ? (int)vol[cell] : (int)col[cell];
                } else {
                    const int cl = max(j + lofs, 0);
                    for (int dy = -w2; dy <= w2; ++dy)
                        s += abs((int)pl[(size_t)(y + dy) * pitch + cl] - (int)pr[(size_t)(y + dy) * pitch + k]);
                }
            }
            sad[k] = s;
            best = min(best, ((unsigned)s << 8) | (unsigned)k);   // first minimum: smallest k among equal sums
        }
        best = __reduce_min_sync(FULL, best);
        const int minsad = (int)(best >> 8), mind = (int)(best & 0xffu);
        bool reject = tex < texThr;
        if (uniq > 0) {
            const int thresh = minsad + (minsad * uniq / 100);
            bool other = false;
            for (int k = lane; k < D; k += 32) other |= (k < mind - 1 || k > mind + 1) && sad[k] <= thresh;
            reject |= __any_sync(FULL, other);
        }
        __syncwarp();
        if (lane == 0 && !reject) {
            const int p = mind + 1 < D ? sad[mind + 1] : sad[D - 2], n = mind > 0 ? sad[mind - 1] : sad[1];
            const int den = p + n - 2 * minsad + abs(p - n);
            const int d = ((D - 1 - mind) * 256 + (den != 0 ? (p - n) * 256 / den : 0) + 15) >> 4;
            rowd[X] = (int16_t)d;
            atomicMin(&keys[X - ((d + 8) >> 4)], ((unsigned)minsad << 12) | (unsigned)X);
        }
        __syncwarp();
    }
    // phase 2: the valid pixels the WTA matched (FILTERED ones take no part)
    const int* crow = cost + row;
    for (int X = xlo + threadIdx.x; X < xhi; X += BM_LR_THREADS) {
        const int d = rowd[X];
        if (d != FILT) atomicMin(&keys[X - ((d + 8) >> 4)], ((unsigned)crow[X] << 12) | (unsigned)X);
    }
    __syncthreads();
    const int lim = 16 * d12;
    auto inconsistent = [&](int x2, int d) {
        if (x2 < 0 || x2 >= W || keys[x2] == 0xffffffffu) return false;
        return abs((int)rowd[keys[x2] & 0xfffu] - d) > lim;
    };
    for (int X = xlo + threadIdx.x; X < xhi; X += BM_LR_THREADS) {
        const int d = rowd[X];
        if (d != FILT && inconsistent(X - (d >> 4), d) && inconsistent(X - ((d + 15) >> 4), d)) drow[X] = (int16_t)FILT;
    }
}

// n is a multiple of 8 pixels (the image buffers are padded to 16 bytes): one 128-bit store per thread
__global__ void k_fill16(int16_t* p, size_t n, int16_t v)
{
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
    const unsigned vv = (unsigned)(uint16_t)v * 0x10001u;
    if (i + 8 <= n) st128(p + i, make_uint4(vv, vv, vv, vv));
    else for (size_t k = i; k < n; ++k) p[k] = v;
}

}  // namespace

int bm_lrcheck_max_width() { return BM_LR_MAXW; }

// the map after the matcher (and the left-right check) -> the speckle filter -> the slot's disparities
static cudaError_t bm_speckle(Engine* c, int B)
{
    if (c->bm_speckle_win <= 0) return cudaSuccess;
    return launch_speckle(c, c->disp_raw, io(c).disp, B, c->bm.FILT, c->bm_speckle_win, c->bm_speckle_range);
}

cudaError_t launch_bm(Engine* c, int B)
{
    const BmNorm& n = c->bm;
    const bool col8 = n.col8 && !(c->debug_flags & 2u);         // debug bit 1: never keep a volume as bytes
    const int W = c->W, H = c->H;
    const size_t npx = (size_t)B * W * H;
    // with the speckle filter the matcher's map is an intermediate (disp_raw, debug_read 2)
    int16_t* const out = c->bm_speckle_win > 0 ? c->disp_raw : io(c).disp;
    const bool lr = c->bm_d12 >= 0;
    { KernelTimer kt(c, KID_FILL); k_fill16<<<(unsigned)((npx / 8 + 256) / 256), 256, 0, c->stream>>>(out, npx, (int16_t)n.FILT); }
    {
        dim3 blk(128), grd((W + 127) / 128, (H + 4 * BM_PF_ROWS - 1) / (4 * BM_PF_ROWS), 2 * B);
        KernelTimer kt(c, KID_BM_PREFILTER);
        k_bm_prefilter<<<grd, blk, 0, c->stream>>>(io(c).rect[0], io(c).rect[1], c->pitch, W, H, n.cap, c->bm_pre[0], c->bm_pre[1]);
    }
    const bool any = !(n.lofs >= W || n.width1 < 1) && (H - 2 * n.w2 > 0) && (n.width1 - 2 * n.w2 > 0);
    if (!any) {
        MVSV_TRY(cudaGetLastError());
        return bm_speckle(c, B);
    }
    {
        KernelTimer kt(c, KID_BM_TEX);
        if (n.bs <= 63) {
            const int nxw = (128 - 2 * n.w2) & ~3;
            dim3 grd((W - 2 * n.w2 + nxw - 1) / nxw, (H - 2 * n.w2 + 4 * BM_TEX_ROWS - 1) / (4 * BM_TEX_ROWS), B);
            k_bm_tex_w<<<grd, 128, 0, c->stream>>>(c->bm_pre[0], c->pitch, W, H, n.w2, n.cap, c->bm_tex2);
        } else {
            const int nx = 256 - 2 * n.w2;                  // blockSize <= 255: at least two output columns per CTA
            dim3 grd((W - 2 * n.w2 + nx - 1) / nx, (H - 2 * n.w2 + BM_TEX_ROWS - 1) / BM_TEX_ROWS, B);
            k_bm_tex<<<grd, 256, 0, c->stream>>>(c->bm_pre[0], c->pitch, W, H, n.w2, n.cap, c->bm_tex2);
        }
    }
    {
        const long long threads = (long long)n.width1 * (n.D / 8);
        dim3 grd((unsigned)((threads + 127) / 128), B);
        // blockSize^2 * 2 * cap <= 65535 (contract) bounds blockSize by 181: the ring needs at most 181 KB
        const size_t ringBytes = (size_t)n.bs * 128 * sizeof(uint2);
        const auto colsum = col8 ? k_bm_colsum<true> : k_bm_colsum<false>;
        MVSV_TRY(smem_limit((const void*)colsum, 200 * 1024));
        KernelTimer kt(c, KID_BM_COLSUM);
        colsum<<<grd, 128, ringBytes, c->stream>>>(c->bm_pre[0], c->bm_pre[1], c->pitch, H, n.width1, n.D, n.lofs, n.w2, c->bm_col);
    }
    BmArgs a;
    a.col = c->bm_col; a.tex = c->bm_tex2; a.disp = out; a.W = W; a.H = H; a.width1 = n.width1; a.D = n.D; a.Dp = n.Dp;
    a.lofs = n.lofs; a.w2 = n.w2; a.texThr = n.tex; a.uniq = n.uniq; a.B = B;
    int* const cost = lr ? static_cast<int*>(c->d2) : nullptr;                 // the SGBM's disp2 keys buffer: same shape, idle here
    {
        KernelTimer kt(c, KID_BM_WTA);
        // Two octets per lane (numDisp is a multiple of 16) with the window ring while at least eight warps fit an SM
        // (four with the byte volume's smaller ring), one octet per lane while four do, else (blockSize > ~100) no ring.
        const int slots = n.bs + 1 + BM_PF;
        int wps = 0, nw;
        if (col8) {
            nw = bm_wta_cta_warps(bm_wta_warp_smem(n.D, 2, 1, slots), &wps);
            if (wps >= 4) MVSV_TRY((launch_bm_wta<2, true, true>(c, a, cost, slots, nw)));
            else MVSV_TRY((launch_bm_wta<2, false, true>(c, a, cost, slots, 4)));
        } else if (nw = bm_wta_cta_warps(bm_wta_warp_smem(n.D, 2, 2, slots), &wps), wps >= 8) {
            MVSV_TRY((launch_bm_wta<2, true, false>(c, a, cost, slots, nw)));
        } else if (nw = bm_wta_cta_warps(bm_wta_warp_smem(n.D, 1, 1, slots), &wps), wps >= 4) {
            MVSV_TRY((launch_bm_wta<1, true, false>(c, a, cost, slots, nw)));
        } else {
            MVSV_TRY((launch_bm_wta<2, false, false>(c, a, cost, slots, 4)));
        }
    }
    if (lr) {
        KernelTimer kt(c, KID_BM_LRCHECK);
        const auto k = col8 ? k_bm_lrcheck<true> : k_bm_lrcheck<false>;
        k<<<dim3(H - 2 * n.w2, B), BM_LR_THREADS, 0, c->stream>>>(out, c->d2, c->bm_col, c->bm_pre[0], c->bm_pre[1], c->pitch, W, H,
                                                                  n.width1, n.D, n.w2, n.cap, n.tex, n.uniq, c->bm_d12);
        MVSV_TRY(cudaGetLastError());
    }
    return bm_speckle(c, B);
}
