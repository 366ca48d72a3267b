// Fused previous-row sweep of StereoSGBM's path aggregation (SURVEY.md A.2 `step`; cv::StereoSGBM::compute behind
// Disparity::sgbm, reference src/disparity.cpp:6-10): the three paths whose predecessor lies in the previous row,
// r = (-1,dy), (0,dy), (+1,dy) with dy = -1 (top-down) or +1 (bottom-up, second sweep of MODE_HH,
// reference src/disparity.cpp:92-95), added into S in one pass over C and S.
//
// Layout of the work ("disparities in registers"): a pixel's D disparities live in the registers of G = 1, 2 or 4
// adjacent lanes, NR packed u16x2 registers (2*NR disparities) per lane, so that for D <= 64 one lane owns a whole
// pixel: the d-1 / d+1 neighbours of the recurrence are register-to-register byte permutes, the minimum over d is
// an in-register tree, and there are no shuffles at all (G > 1: two neighbour shuffles and log2 G butterfly steps).
// A warp owns 32/G adjacent pixels of a row and marches down the rows of its frame; a CTA is a column strip of up
// to 352/G pixels, a frame is NS strips, and the grid is persistent: NF = floor(#SMs / NS) frames are in flight and
// every CTA walks frames fs, fs + NF, ...
//
// State: the vertical path stays in registers (a lane keeps its column).  The diagonal paths live in shared memory
// at skewed ring slots (lx -/+ t) mod R (t = running row count), so a pixel finds its predecessor in the very slot
// it overwrites: no double buffering, and a slot is only ever touched by one lane per row.  Warps are NOT coupled
// by CTA barriers: warp w+1 needs warp w's last pixel of the previous row (and vice versa for the other diagonal);
// each warp publishes a per-path progress counter in shared memory and its neighbour polls it.  The ring has nw
// spare slots because warps may drift by one row per warp boundary.
//
// Path order inside a row is (diagonal from x-1, fused with the vertical path in one loop body: two independent
// dependency chains) -> (diagonal from x+1): what a neighbour needs first is produced first and what comes from a
// neighbour is consumed last.  (Giving the warp with a strip's first pixel the opposite order -- more slack per border
// on paper -- was measured and rejected: DESIGN.md section 8.)
//
// Strip borders cross CTAs without flags or fences: path costs are at most 0x7fff, so bit 15 of every 16-bit value
// is free; the sender ORs a 4-bit sequence number of the row into those bits of each 8-byte half of a 16-byte chunk,
// and the receiver polls the (four-deep) record itself until every chunk carries the number it expects (the
// low-latency protocol of collective libraries).  With a release/acquire flag the hand-off through global memory
// cost 3.6-4 us per hop and set the pace of the whole frame; with tagged data it is one L2 round trip.  Two
// transports: for one lane per pixel and 2..8 strips the strips of a frame are launched as one thread-block cluster
// and the record is stored straight into the neighbour's shared memory (mapa + st.shared::cluster; template
// parameter DSM); otherwise it goes through global memory (L2) and all CTAs are co-resident by a cooperative launch
// (one CTA per SM).
//
// Operands: a warp's 32/G pixels of a row are one contiguous span of C (and S).  The warp copies it with coalesced
// 16-byte cp.async (LDGSTS) straight into shared memory, transposing on the way: chunk c of the span lands in the
// block of the lane that owns it, blocks padded to an odd number of 16-byte chunks so that every lane can then
// read its own 4*NR bytes with conflict-free 128-bit loads.  Rows are prefetched one (short blocks: up to four)
// rows ahead; S is updated in place in shared memory and written back the same way (coalesced 128-bit stores).
// (A per-lane cp.async.bulk was tried first: UBLKCP is a uniform-datapath instruction, so 32 different addresses
// are serialised by an ELECT loop -- 8.3 ms instead of 4.1 ms at cfg 2.)
#include "mvsv_internal.h"

#include <algorithm>
#include <cstdlib>
#include <type_traits>

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int SW_MAX_THREADS = 352;          // 11 warps = 3 per scheduler: 168 registers per thread
constexpr int SW_SMEM_LIMIT = 227 * 1024;

struct SweepArgs {
    const uint16_t* C; uint16_t* S;
    int H, W1, D, Dp, B;
    int NS, NF, Mmax;            // strips per frame, frames in flight, widest strip
    int bottomUp;
    int dsm;                     // the NS strips of a frame form a thread-block cluster: border records go through
                                 // distributed shared memory instead of global memory
    int mode;                    // 0 saturating adds, 1 plain adds of the row's paths, 2 S as bytes (see k_sweep)
    unsigned one;                // always 1 (see path_step)
    unsigned P1P1, P2P2;
    uint16_t* halo;              // [NF][NS][2][NSLOT][Dp + 8] u16: tagged border records (dir 0: for the strip to the right)
};

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(unsigned dst, const void* src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ int ld_acquire_cta(const int* p)
{
    int v;
    asm volatile("ld.acquire.cta.shared.s32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_cta(int* p, int v)
{
    asm volatile("st.release.cta.shared.s32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ uint4 ld_relaxed128(const void* p)
{
    uint4 v;
    asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed128(void* p, const uint4& v)
{
    asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// distributed shared memory (the strips of a frame launched as one thread-block cluster)
__device__ __forceinline__ unsigned mapa_u32(unsigned addr, unsigned cta)
{
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta));
    return r;
}
__device__ __forceinline__ void st_dsm128(unsigned raddr, const uint4& v)
{
    asm volatile("st.relaxed.cluster.shared::cluster.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(raddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ld_dsm128(const unsigned* p)
{
    uint4 v;
    asm volatile("ld.relaxed.cluster.shared::cta.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(smem_u32(p)) : "memory");
    return v;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
constexpr unsigned TAGMASK = 0x80008000u;
// border records per boundary and direction: with the role-based path order a sender can be three rows ahead of the
// row its neighbour is still receiving
constexpr int NSLOT = 4;

// One step of the path recurrence (A.2 `step`) on the 2*NR disparities of a lane:
//   L[k] = C[k] + min(Lp[k], Lp[k-1]+P1, Lp[k+1]+P1, m+P2) - m ;  mm = packed min_k L[k] (both halves)
// "No predecessor" is the state (L = 0, m = 0), which yields L = C.  Registers j >= jpad of the last lane hold
// padding disparities (numDisp < G*2*NR): they stay at 0x7fff, the out-of-range neighbour value.
// Pipe balance: the packed min / permute instructions (VIMNMX, VIMNMX3, PRMT) issue on the ALU pipe at one warp
// instruction per two cycles per scheduler, and so does IADD3; IMAD has the same rate on the FMA pipe.  The plain
// adds of the recurrence are therefore written as x * one + y with `one` a kernel argument (always 1), which ptxas
// cannot fold and emits as IMAD: three adds per register go to the FMA pipe beside 3 1/3 ALU-pipe instructions.
template <int NR, int G, bool PAD>
__device__ __forceinline__ void path_step(unsigned (&L)[NR], unsigned& mm, const unsigned (&C)[NR], unsigned P1P1, unsigned P2P2,
                                          unsigned one, int q, int jpad)
{
    // min(min(Lp[k-1], Lp[k+1]) + P1, Lp[k], m + P2) == min3(Lp[k-1] + P1, Lp[k+1] + P1, min(Lp[k], m + P2)); P1 is added
    // with a plain 32-bit add (no carry between the halves: L + P1 < 65536)
    unsigned up = 0xffffffffu, dn = 0xffffffffu;          // out-of-range neighbour: larger than any L + P1
    unsigned Pj = L[0] * one + P1P1;
    if (G > 1) {
        const unsigned u = __shfl_up_sync(FULL, L[NR - 1] * one + P1P1, 1, G);
        const unsigned d = __shfl_down_sync(FULL, Pj, 1, G);
        if (q != 0) up = u;
        if (q != G - 1) dn = d;
    }
    const unsigned mP2 = mm + P2P2;
    const unsigned negm = 0u - mm;                        // min3 - m per half never borrows (min3 >= m in both halves)
    unsigned Xj = __byte_perm(up, Pj, 0x5432);            // (d-1 of the low half, d-1 of the high half)
#pragma unroll
    for (int j = 0; j < NR; ++j) {
        const unsigned Pn = (j + 1 < NR) ? L[j + 1] * one + P1P1 : dn;
        const unsigned Xn = __byte_perm(Pj, Pn, 0x5432);  // (d+1 of the low half, d+1 of the high half)
        unsigned n = (__vimin3_u16x2(Xj, Xn, __vminu2(L[j], mP2)) * one + negm) * one + C[j];
        if (PAD && q == G - 1 && j >= jpad) n = MVSV_PK_MAX;
        L[j] = n;
        Xj = Xn; Pj = Pn;
    }
    // minimum over the lane's registers: four independent chains, then one combine
    unsigned a0 = L[0], a1 = L[1], a2 = L[2], a3 = L[3];
#pragma unroll
    for (int j = 4; j < NR; j += 8) {
        if (j + 7 < NR) {
            a0 = __vimin3_u16x2(a0, L[j], L[j + 4]); a1 = __vimin3_u16x2(a1, L[j + 1], L[j + 5]);
            a2 = __vimin3_u16x2(a2, L[j + 2], L[j + 6]); a3 = __vimin3_u16x2(a3, L[j + 3], L[j + 7]);
        } else {
            a0 = __vminu2(a0, L[j]); a1 = __vminu2(a1, L[j + 1]); a2 = __vminu2(a2, L[j + 2]); a3 = __vminu2(a3, L[j + 3]);
        }
    }
    unsigned mv = __vimin3_u16x2(a0, a1, __vminu2(a2, a3));
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) mv = __vminu2(mv, __shfl_xor_sync(FULL, mv, o, G));
    mm = __vminu2(mv, __byte_perm(mv, 0, 0x1032));
}

// Two independent recurrence steps (two paths of the same pixel: same C, separate state) in one loop body, so that the
// two dependency chains interleave and a warp has twice the independent instructions in flight.
template <int NR, int G, bool PAD>
__device__ __forceinline__ void path_step2(unsigned (&L)[NR], unsigned& mm, unsigned (&K)[NR], unsigned& km, const unsigned (&C)[NR],
                                           unsigned P1P1, unsigned P2P2, unsigned one, int q, int jpad)
{
    unsigned upL = 0xffffffffu, dnL = 0xffffffffu, upK = 0xffffffffu, dnK = 0xffffffffu;
    unsigned PjL = L[0] * one + P1P1, PjK = K[0] * one + P1P1;
    if (G > 1) {
        const unsigned uL = __shfl_up_sync(FULL, L[NR - 1] * one + P1P1, 1, G), uK = __shfl_up_sync(FULL, K[NR - 1] * one + P1P1, 1, G);
        const unsigned dL = __shfl_down_sync(FULL, PjL, 1, G), dK = __shfl_down_sync(FULL, PjK, 1, G);
        if (q != 0) { upL = uL; upK = uK; }
        if (q != G - 1) { dnL = dL; dnK = dK; }
    }
    const unsigned mP2L = mm + P2P2, negL = 0u - mm, mP2K = km + P2P2, negK = 0u - km;
    unsigned XjL = __byte_perm(upL, PjL, 0x5432), XjK = __byte_perm(upK, PjK, 0x5432);
#pragma unroll
    for (int j = 0; j < NR; ++j) {
        const unsigned PnL = (j + 1 < NR) ? L[j + 1] * one + P1P1 : dnL;
        const unsigned PnK = (j + 1 < NR) ? K[j + 1] * one + P1P1 : dnK;
        const unsigned XnL = __byte_perm(PjL, PnL, 0x5432), XnK = __byte_perm(PjK, PnK, 0x5432);
        unsigned nL = (__vimin3_u16x2(XjL, XnL, __vminu2(L[j], mP2L)) * one + negL) * one + C[j];
        unsigned nK = (__vimin3_u16x2(XjK, XnK, __vminu2(K[j], mP2K)) * one + negK) * one + C[j];
        if (PAD && q == G - 1 && j >= jpad) { nL = MVSV_PK_MAX; nK = MVSV_PK_MAX; }
        L[j] = nL; K[j] = nK;
        XjL = XnL; PjL = PnL; XjK = XnK; PjK = PnK;
    }
    unsigned a0 = L[0], a1 = L[1], a2 = L[2], a3 = L[3], b0 = K[0], b1 = K[1], b2 = K[2], b3 = K[3];
#pragma unroll
    for (int j = 4; j < NR; j += 8) {
        if (j + 7 < NR) {
            a0 = __vimin3_u16x2(a0, L[j], L[j + 4]); a1 = __vimin3_u16x2(a1, L[j + 1], L[j + 5]);
            a2 = __vimin3_u16x2(a2, L[j + 2], L[j + 6]); a3 = __vimin3_u16x2(a3, L[j + 3], L[j + 7]);
            b0 = __vimin3_u16x2(b0, K[j], K[j + 4]); b1 = __vimin3_u16x2(b1, K[j + 1], K[j + 5]);
            b2 = __vimin3_u16x2(b2, K[j + 2], K[j + 6]); b3 = __vimin3_u16x2(b3, K[j + 3], K[j + 7]);
        } else {
            a0 = __vminu2(a0, L[j]); a1 = __vminu2(a1, L[j + 1]); a2 = __vminu2(a2, L[j + 2]); a3 = __vminu2(a3, L[j + 3]);
            b0 = __vminu2(b0, K[j]); b1 = __vminu2(b1, K[j + 1]); b2 = __vminu2(b2, K[j + 2]); b3 = __vminu2(b3, K[j + 3]);
        }
    }
    unsigned mvL = __vimin3_u16x2(a0, a1, __vminu2(a2, a3)), mvK = __vimin3_u16x2(b0, b1, __vminu2(b2, b3));
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) {
        mvL = __vminu2(mvL, __shfl_xor_sync(FULL, mvL, o, G));
        mvK = __vminu2(mvK, __shfl_xor_sync(FULL, mvK, o, G));
    }
    mm = __vminu2(mvL, __byte_perm(mvL, 0, 0x1032));
    km = __vminu2(mvK, __byte_perm(mvK, 0, 0x1032));
}

template <int NR, int G, bool PAD>
__device__ __forceinline__ void reset_path(unsigned (&L)[NR], unsigned& mm, int q, int jpad)
{
#pragma unroll
    for (int j = 0; j < NR; ++j) L[j] = (PAD && q == G - 1 && j >= jpad) ? MVSV_PK_MAX : 0u;
    mm = 0u;
}

// A lane's block of NR registers in shared memory (blocks are padded to an odd number of 16-byte chunks)
template <int NR>
__device__ __forceinline__ void lds_block(unsigned (&V)[NR], const unsigned* p)
{
#pragma unroll
    for (int j = 0; j < NR; j += 4) {
        const uint4 v = *reinterpret_cast<const uint4*>(p + j);
        V[j] = v.x; V[j + 1] = v.y; V[j + 2] = v.z; V[j + 3] = v.w;
    }
}
template <int NR>
__device__ __forceinline__ void sts_block(unsigned* p, const unsigned (&V)[NR])
{
#pragma unroll
    for (int j = 0; j < NR; j += 4) *reinterpret_cast<uint4*>(p + j) = make_uint4(V[j], V[j + 1], V[j + 2], V[j + 3]);
}

// stages of the C / S operand rings (rows in flight): short lane blocks need more rows to cover the memory latency
__host__ __device__ constexpr int sweep_stages(int NR) { return NR >= 20 ? 1 : NR >= 12 ? 2 : 4; }
// lane-block stride in words: an odd number of 16-byte chunks, so that the 128-bit accesses of eight neighbouring
// lanes fall into eight different bank groups
__host__ __device__ constexpr int sweep_lbw(int NR) { return ((NR / 4) | 1) * 4; }

// MODE 0: every add into S saturates.  MODE 1: 3 * (largest possible path cost) <= 65535 (host-checked), so the three
// paths of a row are summed with plain adds and saturated once when they are added to S.  MODE 2 ("S8"): as MODE 1,
// and the S volume holds one BYTE per cell: (sum of the paths so far) - (paths so far) * C, which is the sum of the
// paths' excesses L - C, each in [0, P2]; the host checks npaths * P2 <= 255.  The sweep then adds the byte
// (L1 + L2 + L3 - 3 C) and moves half as many S bytes.
template <int NR, int G, bool PAD, int MODE, bool DSM>
__global__ void __launch_bounds__(SW_MAX_THREADS, 1) k_sweep(SweepArgs a)
{
    constexpr bool FAST = MODE >= 1, S8 = MODE == 2;
    constexpr int NRC = NR / 4, LBW = sweep_lbw(NR), NSTG = sweep_stages(NR);
    // S blocks: NR registers of packed u16 (LBW words apart), or NR / 2 registers of bytes (S8; NR % 8 == 0)
    constexpr int NRS = S8 ? NR / 2 : NR, NRCS = NRS / 4, LBWS = S8 ? sweep_lbw(NRS) : LBW;
    static_assert(!S8 || NR % 8 == 0, "the byte form of S needs whole 16-byte chunks per lane");
    extern __shared__ __align__(16) unsigned smem[];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nthr = blockDim.x, nw = nthr >> 5;
    const int q = tid % G;
    const int fs = blockIdx.x / a.NS, s = blockIdx.x % a.NS;
    const int x0 = (int)(((long long)a.W1 * s) / a.NS), x1 = (int)(((long long)a.W1 * (s + 1)) / a.NS);
    const int M = x1 - x0;
    const int R = a.Mmax + nw;                       // ring of skewed state slots (nw spare: warps drift by <= 1 row each)
    // layout (words): st1[R*G][LBW] | st2[R*G][LBW] | stgC[NSTG][nthr][LBW] | stgS[NSTG][nthr][LBWS] | m1[R] | m2[R] |
    //                 prog1[nw] | prog2[nw]
    unsigned* const st1 = smem;
    unsigned* const st2 = st1 + (size_t)R * G * LBW;
    unsigned* const stgC = st2 + (size_t)R * G * LBW;
    unsigned* const stgS = stgC + (size_t)NSTG * nthr * LBW;
    unsigned* const m1 = stgS + (size_t)NSTG * nthr * LBWS;
    unsigned* const m2 = m1 + R;
    int* const prog1 = reinterpret_cast<int*>(m2 + R);
    int* const prog2 = prog1 + nw;
    // border records received through distributed shared memory: rec[dir][NSLOT][HBW] words, 16-byte aligned
    const int HBW = a.Dp / 2 + 4;
    unsigned* const rec = smem + (((size_t)(prog2 + nw - reinterpret_cast<int*>(smem)) + 3) & ~(size_t)3);
    constexpr bool dsm = DSM;   // compile time: the extra branches cost the D = 256 instances 5 % when they were run-time

    if (tid < nw) { prog1[tid] = 0; prog2[tid] = 0; }
    if (dsm) {
        for (int i = tid; i < 2 * NSLOT * HBW; i += nthr) rec[i] = 0u;          // tag 0: nothing received yet
        cluster_sync_all();                       // every strip of the frame is resident and cleared before any remote store
    } else {
        __syncthreads();
    }

    const int lxr = tid / G;                          // pixel of this lane inside the strip
    const bool act = lxr < M;
    const int lx = act ? lxr : M - 1;
    const int nact = min(max(M * G - w * 32, 0), 32); // active lanes of this warp
    // (nact == 0 is only possible for trailing warps of a narrower strip: they skip the row loop)
    const int wl = (M * G - 1) >> 5;                  // warp holding the strip's last pixel
    const int jpad = PAD ? (a.D - (G - 1) * 2 * NR) / 2 : NR;
    const int nfr = (a.B - fs + a.NF - 1) / a.NF;     // frames this CTA walks
    const int T = nact > 0 ? nfr * a.H : 0;
    const bool hasL = s > 0, hasR = s + 1 < a.NS;
    const bool firstPx = act && lxr == 0, lastPx = act && lxr == M - 1;
    const int HB = a.Dp + 8;                          // border record: Dp path costs + packed minimum (padded to 16 bytes)
    // tagged border records this strip receives from and sends to
    uint16_t* const haloBase = a.halo + (size_t)fs * a.NS * 2 * NSLOT * HB;
    uint16_t* const sendR = haloBase + ((size_t)(s * 2 + 0) * NSLOT) * HB;            // boundary s | s+1, direction right
    const uint16_t* const recvL = haloBase + ((size_t)((s - 1) * 2 + 0) * NSLOT) * HB; // boundary s-1 | s, direction right
    uint16_t* const sendL = haloBase + ((size_t)((s - 1) * 2 + 1) * NSLOT) * HB;      // boundary s-1 | s, direction left
    const uint16_t* const recvR = haloBase + ((size_t)(s * 2 + 1) * NSLOT) * HB;       // boundary s | s+1, direction left
    const unsigned one = a.one;

    // the warp's span of a row: nact lane blocks, contiguous in global memory.  Chunk c = i*32 + lane of the span
    // belongs to lane c / NRC, position c % NRC.
    const size_t rowElems = (size_t)a.W1 * a.Dp;
    const size_t warpOff = (size_t)(x0 + (w * 32) / G) * a.Dp;       // in cells; the lane's 16-byte chunk is added below
    const int nchunks = nact * NRC;
    // element offset of the warp's span in the row that is k rows ahead of (fi, yi), k < H
    auto row_off = [&](int fi, int yi, int k) -> size_t {
        int y = yi + k;
        if (y >= a.H) { y -= a.H; ++fi; }
        const int f = fs + fi * a.NF;
        return ((size_t)f * a.H + (a.bottomUp ? a.H - 1 - y : y)) * rowElems + warpOff;
    };
    int cdst[NRC];                                    // word offset of chunk i*32 + lane inside a stage (-1: beyond the span)
#pragma unroll
    for (int i = 0; i < NRC; ++i) {
        const int c = i * 32 + lane, o = c / NRC, j = c - o * NRC;
        cdst[i] = c < nchunks ? (w * 32 + o) * LBW + j * 4 : -1;
    }
    int sdst[NRCS];                                   // the same for the S blocks (S8: half as many chunks)
#pragma unroll
    for (int i = 0; i < NRCS; ++i) {
        const int c = i * 32 + lane, o = c / NRCS, j = c - o * NRCS;
        sdst[i] = c < nact * NRCS ? (w * 32 + o) * LBWS + j * 4 : -1;
    }
    const char* const Cbytes = reinterpret_cast<const char*>(a.C) + (size_t)lane * 16;
    char* const Sbytes = reinterpret_cast<char*>(a.S) + (size_t)lane * 16;
    auto issueC = [&](int t, size_t cellOff) {
        if (t < T) {
            const char* src = Cbytes + cellOff * 2;
            unsigned* dst = stgC + (size_t)(t % NSTG) * nthr * LBW;
#pragma unroll
            for (int i = 0; i < NRC; ++i)
                if (cdst[i] >= 0) cp_async16(smem_u32(dst + cdst[i]), src + (size_t)i * 512);
        }
        cp_async_commit();
    };
    auto issueS = [&](int t, size_t cellOff) {
        if (t < T) {
            const char* src = Sbytes + cellOff * (S8 ? 1 : 2);
            unsigned* dst = stgS + (size_t)(t % NSTG) * nthr * LBWS;
#pragma unroll
            for (int i = 0; i < NRCS; ++i)
                if (sdst[i] >= 0) cp_async16(smem_u32(dst + sdst[i]), src + (size_t)i * 512);
        }
        cp_async_commit();
    };
#pragma unroll
    for (int k = 0; k < NSTG; ++k) issueC(k, row_off(k / a.H, k % a.H, 0));
#pragma unroll
    for (int k = 0; k + 1 < NSTG; ++k) issueS(k, row_off(k / a.H, k % a.H, 0));
    cp_async_wait<2 * (NSTG - 1)>();                  // C of row 0 has landed
    __syncwarp();

    unsigned Lv[NR], mv;
    reset_path<NR, G, PAD>(Lv, mv, q, jpad);
    int s1 = lx, s2 = lx;                             // (lx - t) mod R, (lx + t) mod R
    int yi = 0, fi = 0;
    for (int t = 0; t < T; ++t) {
        const int st = t % NSTG;
        const bool firstRow = yi == 0, lastRow = yi == a.H - 1;
        // ---- C of this row: shared memory -> registers (it landed before the end of the previous row), then refill
        //      the stage with row t + NSTG
        unsigned Cc[NR];
        lds_block<NR>(Cc, stgC + ((size_t)st * nthr + tid) * LBW);
        __syncwarp();

        unsigned Ss[NR];                              // sum of the three paths of this row
        // tag of the records received in this row / sent for the next one: 4 bits in the free top bits of the first
        // two registers of every 8-byte half (see the header)
        const unsigned seqR = (unsigned)(t / NSLOT + 1), seqS = (unsigned)((t + 1) / NSLOT + 1);
        const unsigned tagRx = ((seqR & 1u) << 15) | ((seqR & 2u) << 30), tagRy = ((seqR & 4u) << 13) | ((seqR & 8u) << 28);
        const unsigned tagSx = ((seqS & 1u) << 15) | ((seqS & 2u) << 30), tagSy = ((seqS & 4u) << 13) | ((seqS & 8u) << 28);

        // One diagonal path.  DIR 0: predecessor (x-1, previous row), state flows to the right; DIR 1: predecessor
        // (x+1, previous row), state flows to the left.  The result is left in L.
        auto diag = [&](auto dirTag, auto fuseTag, unsigned (&L)[NR]) {
            constexpr int DIR = decltype(dirTag)::value;
            constexpr bool FUSE_V = decltype(fuseTag)::value;    // run the vertical path's step interleaved with this one
            const int sidx = DIR ? s2 : s1;
            unsigned* const slot = (DIR ? st2 : st1) + (size_t)(sidx * G + q) * LBW;
            unsigned* const mArr = DIR ? m2 : m1;
            int* const prog = DIR ? prog2 : prog1;
            const bool recvPx = DIR ? lastPx : firstPx, sendPx = DIR ? firstPx : lastPx;
            const bool nbStripR = DIR ? hasR : hasL, nbStripS = DIR ? hasL : hasR;   // strip we receive from / send to
            unsigned mm;
            // Pace against the neighbouring warp on every row -- also on a frame's first row, which needs no data from
            // it: the slot ring only has room for a drift of one row per warp boundary.
            if (DIR ? (w < wl) : (w > 0)) {
                const int* nb = prog + (DIR ? w + 1 : w - 1);
                while (ld_acquire_cta(nb) < t) {}
            }
            if (firstRow) {
                reset_path<NR, G, PAD>(L, mm, q, jpad);
            } else {
                if (recvPx) {
                    // the strip's border pixel: predecessor is off the cost domain (state 0) or in the next strip (record)
                    if (nbStripR) {
                        // all chunks of the record are requested together; the whole set is re-read until every
                        // 8-byte half carries this row's tag (one L2 round trip once the record is there)
                        const uint16_t* hb = (DIR ? recvR : recvL) + (size_t)(t % NSLOT) * HB;
                        const uint16_t* hp = hb + (size_t)q * 2 * NR;
                        const unsigned* rb = rec + (size_t)(DIR * NSLOT + t % NSLOT) * HBW;     // the same record in shared memory
                        unsigned bad;
                        uint4 mrec = make_uint4(tagRx, tagRy, 0u, 0u);
                        do {
#pragma unroll
                            for (int j = 0; j < NR; j += 4) {
                                const uint4 v = dsm ? ld_dsm128(rb + q * NR + j) : ld_relaxed128(hp + 2 * j);
                                L[j] = v.x; L[j + 1] = v.y; L[j + 2] = v.z; L[j + 3] = v.w;
                            }
                            if (q == 0) mrec = dsm ? ld_dsm128(rb + a.Dp / 2) : ld_relaxed128(hb + a.Dp);
                            bad = ((mrec.x & TAGMASK) ^ tagRx) | ((mrec.y & TAGMASK) ^ tagRy);
#pragma unroll
                            for (int j = 0; j < NR; j += 2) bad |= ((L[j] & TAGMASK) ^ tagRx) | ((L[j + 1] & TAGMASK) ^ tagRy);
                        } while (bad);
#pragma unroll
                        for (int j = 0; j < NR; ++j) L[j] &= MVSV_PK_MAX;
                        sts_block<NR>(slot, L);
                        if (q == 0) mArr[sidx] = mrec.x & MVSV_PK_MAX;
                    } else {
                        reset_path<NR, G, PAD>(L, mm, q, jpad);
                        sts_block<NR>(slot, L);
                        if (q == 0) mArr[sidx] = 0u;
                    }
                }
                if (G > 1) __syncwarp();              // the pixel's other lanes read the minimum written by lane q == 0
                lds_block<NR>(L, slot);
                mm = mArr[sidx];
            }
            if (FUSE_V) {
                if (firstRow) reset_path<NR, G, PAD>(Lv, mv, q, jpad);
                path_step2<NR, G, PAD>(L, mm, Lv, mv, Cc, a.P1P1, a.P2P2, one, q, jpad);
            } else {
                path_step<NR, G, PAD>(L, mm, Cc, a.P1P1, a.P2P2, one, q, jpad);
            }
            if (act) {
                sts_block<NR>(slot, L);
                if (q == 0) mArr[sidx] = mm;
                if (sendPx && nbStripS && !lastRow) {
                    if (dsm) {
                        // the neighbour strip is CTA s -/+ 1 of this cluster; its rec[DIR] takes what we send in direction DIR
                        const unsigned rb = mapa_u32(smem_u32(rec + (size_t)(DIR * NSLOT + (t + 1) % NSLOT) * HBW), (unsigned)(DIR ? s - 1 : s + 1));
#pragma unroll
                        for (int j = 0; j < NR; j += 4)
                            st_dsm128(rb + (unsigned)(q * NR + j) * 4u, make_uint4(L[j] | tagSx, L[j + 1] | tagSy, L[j + 2] | tagSx, L[j + 3] | tagSy));
                        if (q == 0) st_dsm128(rb + (unsigned)(a.Dp / 2) * 4u, make_uint4(mm | tagSx, tagSy, tagSx, tagSy));
                    } else {
                        uint16_t* hp = (DIR ? sendL : sendR) + (size_t)((t + 1) % NSLOT) * HB;
#pragma unroll
                        for (int j = 0; j < NR; j += 4)
                            st_relaxed128(hp + (size_t)q * 2 * NR + 2 * j, make_uint4(L[j] | tagSx, L[j + 1] | tagSy, L[j + 2] | tagSx, L[j + 3] | tagSy));
                        if (q == 0) st_relaxed128(hp + a.Dp, make_uint4(mm | tagSx, tagSy, tagSx, tagSy));
                    }
                }
            }
            __syncwarp();
            if (lane == 0) st_release_cta(prog + w, t + 1);
        };

        // ---- diagonal from x-1 first: it feeds the warp / strip to the right
        diag(std::integral_constant<int, 0>(), std::true_type(), Ss);
        // ---- prefetches, issued after the first diagonal so that its border record does not queue behind them:
        //      C of row t + NSTG into the stage just read; S of row t + NSTG - 1 into the stage whose write-back (row
        //      t - 1) has been read out
        issueC(t + NSTG, row_off(fi + NSTG / a.H, yi, NSTG % a.H));
        issueS(t + NSTG - 1, row_off(fi + (NSTG - 1) / a.H, yi, (NSTG - 1) % a.H));
        // ---- vertical path (state in registers): its step ran interleaved with the first diagonal's
#pragma unroll
        for (int j = 0; j < NR; ++j) Ss[j] = FAST ? Ss[j] * one + Lv[j] : __viaddmin_u16x2(Ss[j], Lv[j], MVSV_PK_MAX);
        // ---- diagonal from x+1 last: it needs the warp / strip to the right
        {
            unsigned L[NR];
            diag(std::integral_constant<int, 1>(), std::false_type(), L);
#pragma unroll
            for (int j = 0; j < NR; ++j) Ss[j] = FAST ? Ss[j] * one + L[j] : __viaddmin_u16x2(Ss[j], L[j], MVSV_PK_MAX);
        }
        // ---- S += the three paths, in place in shared memory, then coalesced write-back of the warp's span
        {
            unsigned* const stage = stgS + (size_t)st * nthr * LBWS;
            unsigned* const sb = stage + (size_t)tid * LBWS;
            cp_async_wait<2 * (NSTG - 1)>();          // S of this row (and C of the next) have landed
            __syncwarp();
            unsigned Sin[NRS];
            lds_block<NRS>(Sin, sb);
            if (S8) {
                // bytes of L1 + L2 + L3 - 3 C (each path's excess is in [0, P2], the byte sums stay below 256)
#pragma unroll
                for (int j = 0; j < NR; ++j) Ss[j] -= 3u * Cc[j];
#pragma unroll
                for (int j = 0; j < NRS; ++j) Sin[j] += __byte_perm(Ss[2 * j], Ss[2 * j + 1], 0x6420);
            } else {
#pragma unroll
                for (int j = 0; j < NR; ++j)  // FAST: the plain sum of three paths may exceed 0x7fff (but not 0xffff)
                    Sin[j] = __viaddmin_u16x2(FAST ? __vminu2(Ss[j], MVSV_PK_MAX) : Ss[j], Sin[j], MVSV_PK_MAX);
            }
            sts_block<NRS>(sb, Sin);
            __syncwarp();
            char* dst = Sbytes + row_off(fi, yi, 0) * (S8 ? 1 : 2);
#pragma unroll
            for (int i = 0; i < NRCS; ++i)
                if (sdst[i] >= 0) *reinterpret_cast<uint4*>(dst + (size_t)i * 512) = *reinterpret_cast<const uint4*>(stage + sdst[i]);
        }
        if (--s1 < 0) s1 += R;
        if (++s2 >= R) s2 -= R;
        if (++yi == a.H) { yi = 0; ++fi; }
    }
    cp_async_wait<0>();
    if (dsm) cluster_sync_all();                  // no strip may exit while a neighbour can still store into its shared memory
}

size_t sweep_smem_bytes(int NR, int G, int Mmax, int nthr)
{
    const int LBW = sweep_lbw(NR), NSTG = sweep_stages(NR), nw = nthr / 32, R = Mmax + nw;
    size_t words = (size_t)2 * R * G * LBW + (size_t)2 * NSTG * nthr * LBW + 2 * R + 2 * nw;
    words = ((words + 3) & ~(size_t)3) + (size_t)2 * NSLOT * (G * NR + 4);      // + border records (cluster hand-off)
    return words * 4;
}

// One launch.  DSM: the strips of a frame as one thread-block cluster (co-scheduled by the hardware; frames are
// independent), border records through distributed shared memory -- used only if as many clusters fit at once as frames
// are planned to be in flight: a GPC holds a whole number of clusters, and e.g. clusters of 4 strand 16 of the 148 SMs,
// which would cost a whole extra wave of frames (*fits reports it).  Otherwise: cooperative launch (all CTAs
// co-resident: they wait on one another), records through global memory.
template <int NR, int G, bool PAD, int MODE, bool DSM>
cudaError_t launch_one(const SweepArgs& a, int nthr, size_t smem, cudaStream_t st, bool* fits)
{
    MVSV_TRY(smem_limit((const void*)k_sweep<NR, G, PAD, MODE, DSM>, SW_SMEM_LIMIT));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(a.NS * a.NF, 1, 1); cfg.blockDim = dim3(nthr, 1, 1); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    if (DSM) {
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = a.NS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int nmax = 0;
        MVSV_TRY(cudaOccupancyMaxActiveClusters(&nmax, k_sweep<NR, G, PAD, MODE, DSM>, &cfg));
        *fits = nmax >= a.NF;
        if (!*fits) return cudaSuccess;
    } else {
        at[0].id = cudaLaunchAttributeCooperative; at[0].val.cooperative = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
    }
    return cudaLaunchKernelEx(&cfg, k_sweep<NR, G, PAD, MODE, DSM>, a);
}

template <int NR, int G, bool PAD, int MODE>
cudaError_t launch_fast(const SweepArgs& a, int nthr, size_t smem, cudaStream_t st)
{
    // the cluster variant only exists for one lane per pixel (D <= 64: cfg 2 and the reference's other 752x480 uses)
    if constexpr (G == 1) {
        if (a.dsm) {
            bool fits = false;
            const cudaError_t e = launch_one<NR, G, PAD, MODE, true>(a, nthr, smem, st, &fits);
            if (e != cudaSuccess || fits) return e;
        }
    }
    bool unused = true;
    return launch_one<NR, G, PAD, MODE, false>(a, nthr, smem, st, &unused);
}

template <int NR, int G, bool PAD>
cudaError_t launch_inst(const SweepArgs& a, int nthr, size_t smem, cudaStream_t st)
{
    if constexpr (NR % 8 == 0) {
        if (a.mode == 2) return launch_fast<NR, G, PAD, 2>(a, nthr, smem, st);
    }
    return a.mode >= 1 ? launch_fast<NR, G, PAD, 1>(a, nthr, smem, st) : launch_fast<NR, G, PAD, 0>(a, nthr, smem, st);
}

template <int G, bool PAD>
cudaError_t launch_nr(int NR, const SweepArgs& a, int nthr, size_t smem, cudaStream_t st)
{
    switch (NR) {
        case 4: if constexpr (G == 1) return launch_inst<4, G, PAD>(a, nthr, smem, st); break;
        case 8: if constexpr (G == 1) return launch_inst<8, G, PAD>(a, nthr, smem, st); break;
        case 12: if constexpr (G == 1) return launch_inst<12, G, PAD>(a, nthr, smem, st); break;
        case 16: if constexpr (G == 1) return launch_inst<16, G, PAD>(a, nthr, smem, st); break;
        case 20: return launch_inst<20, G, PAD>(a, nthr, smem, st);
        case 24: return launch_inst<24, G, PAD>(a, nthr, smem, st);
        case 28: return launch_inst<28, G, PAD>(a, nthr, smem, st);
        case 32: return launch_inst<32, G, PAD>(a, nthr, smem, st);
    }
    return cudaErrorInvalidValue;
}

}  // namespace

// Lane layout of the sweep for numDisp = D: G lanes per pixel, NR packed registers per lane; the volumes' pixel
// stride is Dp = G * 2 * NR >= D (a multiple of 8; equal to D whenever D is a multiple of 8 * G).
void sweep_layout(int D, int* G, int* NR)
{
    const int g = D <= 64 ? 1 : D <= 128 ? 2 : 4;
    const int per = (D + g - 1) / g;                  // disparities per lane
    *G = g; *NR = (per + 7) / 8 * 4;
}

// Chooses the strip decomposition for a batch of B frames: NS strips per frame (0 = the sweep cannot run: use the
// independent passes), NF frames in flight, CTA size.  `forcedNS` > 0 pins the strip count, 0xfe only rules out the
// independent passes (test hooks).
void sweep_plan(const Engine* c, int B, int forcedNS, SweepPlan* p)
{
    const SgbmNorm& n = c->sg;
    *p = SweepPlan();
    if (n.W1 <= 0 || B < 1) return;
    int G, NR;
    sweep_layout(n.D, &G, &NR);
    if (G * 2 * NR != n.Dp) return;                   // volumes are laid out with another pixel stride
    const int capThreads = SW_MAX_THREADS / 32 * 32;
    // Time model (measured on B200, profiles/r02_sweep_row_time.txt): a CTA's row takes about c0 + c1 * warps -- a
    // latency floor plus the warps' share of the SM -- plus the border hand-off when a frame has several strips
    // (~0.5 us through a cluster's shared memory, ~1.6 us through global memory), and a batch takes waves * H rows,
    // waves = ceil(B / NF).  Fewer, wider strips amortise the floor; more strips keep a small batch in one wave.
    const double c0 = 1.1, c1 = 0.2, hoCluster = 0.5, hoGlobal = 1.6;
    double best = 1e300;
    for (int NS = 1; NS <= std::min(n.W1, c->num_sms); ++NS) {
        if (forcedNS > 0 && forcedNS != 0xfe && NS != forcedNS) continue;
        const int Mmax = (n.W1 + NS - 1) / NS;
        const int nthr = (Mmax * G + 31) / 32 * 32;
        if (nthr > capThreads) continue;
        const size_t smem = sweep_smem_bytes(NR, G, Mmax, nthr);
        if (smem > (size_t)SW_SMEM_LIMIT) continue;
        const int NF = std::min(B, c->num_sms / NS);
        const int waves = (B + NF - 1) / NF;
        const double handoff = NS == 1 ? 0.0 : (G == 1 && NS <= 8 && NF * NS <= c->num_sms - 16) ? hoCluster : hoGlobal;
        const double cost = waves * (c0 + c1 * (nthr / 32) + handoff) + 1e-6 * NS;   // us per row; ties: fewer strips
        if (cost < best) { best = cost; p->NS = NS; p->NF = NF; p->Mmax = Mmax; p->threads = nthr; p->smem = smem; }
    }
    p->G = G; p->NR = NR;
    // Small batches: the three independent one-direction passes (k_sgbm_vdir: every column of every frame in parallel,
    // 6 B/cell each at HBM speed plus ~0.1 ms of latency per pass) beat a sweep that is paced row by row -- a single
    // 752x480 pair takes 0.4 ms that way and 1.1-2.5 ms in the sweep.  Not when the strip count is forced (tests).
    if (p->NS > 0 && forcedNS <= 0) {        // forcedNS: a strip count, or 0xfe = "the sweep, strips chosen as usual"
        const double sweepMs = best * c->H * 1e-3;
        const double cells = (double)B * c->H * n.W1 * n.Dp;
        const double vdirMs = 3.0 * (0.1 + cells * 6.0 / 5.5e12 * 1e3);
        if (vdirMs < sweepMs) *p = SweepPlan();
    }
}

size_t sweep_scratch_bytes(const Engine* c)
{
    // worst case over all plans and disparity ranges: NF * NS <= num_sms CTAs, 2 directions x NSLOT records each
    return (size_t)c->num_sms * 2 * NSLOT * (256 + 8) * sizeof(uint16_t);
}

// 3 * (largest possible path cost) <= 65535: the three paths of a row can be summed in 16 bits without saturation
static bool sweep_fast_ok(const SgbmNorm& n)
{
    const long long bs = 2 * n.SH2 + 1, lmax = bs * bs * (2 * n.ftzero + 63) + n.P2;
    return 3 * lmax <= 65535;
}

// S as bytes: all npaths excesses (each <= P2) fit a byte, plain 16-bit row sums, whole 16-byte chunks per lane
bool sweep_s8_ok(const Engine* c, const SweepPlan& p)
{
    const SgbmNorm& n = c->sg;
    return p.NS > 0 && p.NR % 8 == 0 && sweep_fast_ok(n) && (long long)n.npaths * n.P2 <= 255;
}

cudaError_t launch_sweep(Engine* c, int B, const SweepPlan& p, int bottomUp, bool s8)
{
    const SgbmNorm& n = c->sg;
    SweepArgs a;
    a.C = c->C; a.S = c->S; a.H = c->H; a.W1 = n.W1; a.D = n.D; a.Dp = n.Dp; a.B = B;
    a.NS = p.NS; a.NF = p.NF; a.Mmax = p.Mmax; a.bottomUp = bottomUp;
    a.dsm = (p.NS >= 2 && p.NS <= 8 && !getenv("MVSV_NO_DSM")) ? 1 : 0;
    a.P1P1 = ((unsigned)n.P1 & 0xffffu) * 0x10001u; a.P2P2 = ((unsigned)n.P2 & 0xffffu) * 0x10001u;
    a.halo = c->sweep_halo;
    a.one = 1u;
    a.mode = s8 ? 2 : (sweep_fast_ok(n) ? 1 : 0);
    // tag 0 everywhere: no record of an earlier launch can be mistaken for one of this launch
    cudaError_t e = cudaMemsetAsync(c->sweep_halo, 0, (size_t)p.NS * p.NF * 2 * NSLOT * (n.Dp + 8) * sizeof(uint16_t), c->stream);
    if (e != cudaSuccess) return e;
    const bool pad = n.D != n.Dp;
    KernelTimer kt(c, KID_SGBM_TD);
    switch (p.G) {
        case 1: return launch_nr<1, false>(p.NR, a, p.threads, p.smem, c->stream);
        case 2: return pad ? launch_nr<2, true>(p.NR, a, p.threads, p.smem, c->stream) : launch_nr<2, false>(p.NR, a, p.threads, p.smem, c->stream);
        default: return pad ? launch_nr<4, true>(p.NR, a, p.threads, p.smem, c->stream) : launch_nr<4, false>(p.NR, a, p.threads, p.smem, c->stream);
    }
}
