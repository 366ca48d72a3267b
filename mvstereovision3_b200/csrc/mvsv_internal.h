// Internal declarations shared by the sm_100a kernels and the C-ABI glue (libmvsv.so).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <string>
#include <vector>

#include "../../include/mvsv.h"

#define MVSV_MAX_COST 32767
#define MVSV_PK_MAX 0x7fff7fffu

// Normalised StereoSGBM parameters (SURVEY.md 8a-3; OpenCV's own normalisation of the values that
// Disparity::loadSGBMParameters hands over, reference src/disparity.cpp:83-95).
struct SgbmNorm {
    int minD, D, Dp, G;          // Dp = G*8 padded disparity count, G = lanes per pixel (power of two)
    int bs, SW2, SH2, ftzero, uniq, d12, P1, P2;
    int maxD, minX1, maxX1, W1, INV, mode, npaths;
    int speckleWin, speckleRange;
    int vsWide;                  // cost kernel with 768 compute threads (D > 128 and the row ring fits shared memory)
};

struct BmNorm {
    int D, Dp, G, bs, w2, cap, tex, uniq;
    int lofs, width1, FILT;
    int col8;                   // column sums fit a byte (blockSize * 2 * cap <= 255): the volume is one byte per cell
};

// kernel ids for the optional per-launch CUDA-event timing (mvsv_profile_*)
enum KernelId {
    KID_REMAP = 0, KID_SGBM_PREFILTER, KID_SGBM_VSUM, KID_SGBM_H1, KID_SGBM_VDIR, KID_SGBM_TD, KID_SGBM_H2_WTA, KID_MEDIAN,
    KID_CCL_ROWS, KID_CCL_VMERGE, KID_CCL_FLATTEN, KID_CCL_APPLY, KID_BM_PREFILTER, KID_BM_TEX, KID_BM_COLSUM,
    KID_BM_WTA, KID_XYZ, KID_MEANS, KID_FILL, KID_MINMAX, KID_TM, KID_BM_LRCHECK, KID_COUNT
};
extern const char* const kKernelNames[KID_COUNT];

struct ProfBracket { int kid; cudaEvent_t a, b; };

// I/O slot (mvsv_set_io_slots): the buffers a compute call reads its inputs into and leaves its results in.  They
// exist once or twice; with two, the host->device copy of the next batch and the device->host copy of the previous
// one overlap the kernels of the current batch inside ONE engine (one set of cost volumes).  The slot is the only
// owner of these buffers; the launchers reach the slot of the compute in progress through io(c).
struct IoSlot {
    uint8_t* rect[2] = {nullptr, nullptr};    // [B][H][pitch]
    uint8_t* raw[2] = {nullptr, nullptr};     // [B][fh][raw_pitch], once rectification maps are installed
    int16_t* disp = nullptr;                  // final disparities [B][H][W]
    float* xyz = nullptr;                     // [B][H][W][3], allocated by the first compute with MVSV_STAGE_XYZ
    float* means = nullptr;                   // [B][nrois], once mean-disparity ROIs are set
    cudaEvent_t done = nullptr;               // all kernels of the slot's last compute have finished
    int B = 0;                                // frames of the slot's last compute; 0: it holds no results
    unsigned stages = 0;
};

struct mvsv_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    // host->device input copies run on their own stream so that they overlap the kernels of the other I/O slot's
    // compute
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_h2d = nullptr, ev_done = nullptr;
    // second kernel stream: the first row scan of one chunk of frames runs beside the cost kernel of the next chunk
    // (sgbm.cu, launch_sgbm_g); joined back into `stream` before the sweep
    cudaStream_t aux_stream = nullptr;
    static constexpr int kMaxChunks = 16;
    cudaEvent_t ev_chunk[kMaxChunks] = {}, ev_join = nullptr;
    int fw = 0, fh = 0;          // raw frame
    int W = 0, H = 0;            // rectified/cropped pair
    int maxB = 0;
    unsigned long long launches = 0;
    unsigned debug_flags = 0;   // bit0: h2 pass stores the final S volume (test hook); bit1: never use the byte form of S;
                                // bit2: the scalar median kernel only; bits 8..15: sweep strips; bits 16..23: frames per
                                // chunk of the vsum / h1 overlap (mvsv.h)
    bool last_s8 = false;       // the last SGBM compute kept S as bytes (S8)
    bool prof = false;
    std::vector<ProfBracket> brackets;      // pending (unread) timed launches
    std::vector<cudaEvent_t> ev_free;       // recycled events
    cudaEvent_t timer_a = nullptr, timer_b = nullptr;
    std::string err;

    // rectification (device): per camera, fixed-point maps for the ROI only
    bool has_maps[2] = {false, false};
    int roi[4] = {0, 0, 0, 0};
    int2* map_xy[2] = {nullptr, nullptr};     // (ix, iy) = rint(map*32), saturated int32
    size_t raw_pitch = 0;
    // cv::resize(.., factor, factor) after the crop (Stereosystem::getRectifiedImagepair(sip, factor),
    // reference src/Stereosystem.cpp:279-315); off when resize_factor == 0
    double resize_factor = 0.0;
    uint8_t* tm_out = nullptr;                // [B][H][pitch], Disparity::tm
    uint8_t* crop[2] = {nullptr, nullptr};    // [B][roi_h][crop_pitch]: remap output when a resize follows
    size_t crop_pitch = 0;

    size_t pitch = 0;                         // row pitch of the rectified images

    int nslots = 1, cur = 0;                  // I/O slots in use; the slot of the last (or current) compute
    IoSlot slot[2];
    cudaStream_t dl_stream = nullptr;         // device->host result copies

    bool has_sgbm = false, has_bm = false;
    mvsv_sgbm_params sgbm_raw{};
    SgbmNorm sg{};
    int td_nc = 0;               // strips per frame of the fused previous-row sweep at max_batch (0: independent passes)
    uint16_t* sweep_halo = nullptr;   // tagged border-pixel records of the strip hand-off (csrc/sweep.cu)
    int num_sms = 148;
    mvsv_bm_params bm_raw{};
    BmNorm bm{};
    // mvsv_set_bm_filters, kept across mvsv_set_bm_params and geometry changes: -1 / 0 = off
    int bm_d12 = -1, bm_speckle_win = 0, bm_speckle_range = 0;

    uint2* recL = nullptr;                    // left prefilter records [B][H][W] (a_s,lo_s,hi_s,a_r,lo_r,hi_r)
    uint16_t* plR = nullptr;                  // right prefilter planes, reversed + padded: [6][B][H][vsRP]
    int vsNV = 0, vsRP = 0, vsJOFF = 0;
    uint16_t* VS = nullptr;                   // [B][H][W1][Dp] vertical box sums of the pixel cost
    uint16_t* C = nullptr;                    // [B][H][W1][Dp] block cost
    uint16_t* S = nullptr;                    // [B][H][W1][Dp] aggregated cost
    size_t vol_elems = 0;                     // elements allocated per volume
    int* d2 = nullptr;                        // [B][H][W] (disp2cost<<16 | disp2)
    int16_t* disp_raw = nullptr;              // [B][H][W]
    int16_t* disp_med = nullptr;              // [B][H][W]
    int* labels = nullptr;                    // [B][H][W]
    int* sizes = nullptr;                     // [B][H][W]

    uint8_t* bm_pre[2] = {nullptr, nullptr};  // [B][H][pitch]
    int* bm_tex2 = nullptr;                   // [B][H][W] texture: window sums of |L - cap|
    size_t bm_vol_elems = 0;
    uint16_t* bm_col = nullptr;               // [B][H][width1][Dp]

    bool has_Q = false;
    float Q[16];
    int nrois = 0;
    int* rois = nullptr;                      // device [n][4]
    int* minmax = nullptr;                    // device [B][2]
};

// the I/O slot of the compute in progress (or of the last one)
inline IoSlot& io(mvsv_ctx* c) { return c->slot[c->cur]; }

// RAII bracket: records CUDA events on the ctx stream around one kernel launch when profiling is on.
struct KernelTimer {
    mvsv_ctx* c; int idx;
    cudaStream_t st;
    KernelTimer(mvsv_ctx* ctx, int kid, cudaStream_t on = nullptr) : c(ctx), idx(-1), st(on ? on : ctx->stream)
    {
        ++c->launches;
        if (!c->prof) return;
        ProfBracket b; b.kid = kid;
        for (cudaEvent_t* e : {&b.a, &b.b}) {
            if (!c->ev_free.empty()) { *e = c->ev_free.back(); c->ev_free.pop_back(); }
            else cudaEventCreate(e);
        }
        cudaEventRecord(b.a, st);
        c->brackets.push_back(b);
        idx = (int)c->brackets.size() - 1;
    }
    ~KernelTimer() { if (idx >= 0) cudaEventRecord(c->brackets[idx].b, st); }
};

// ---- kernel launchers (launch counting happens in KernelTimer) ------------------------------------------
// Each returns the first error of its launches and of the CUDA calls it makes on the way; MVSV_TRY passes one on.
#define MVSV_TRY(call)                                                                          \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) return e_;                                                       \
    } while (0)
// Sets a kernel's cudaFuncAttributeMaxDynamicSharedMemorySize on the current device when it differs from the value set
// there before (function attributes are per device; engines on several devices and threads share this state).
cudaError_t smem_limit(const void* kernel, int bytes);
cudaError_t launch_remap(mvsv_ctx* c, int cam, int B);
cudaError_t launch_resize(mvsv_ctx* c, int cam, int B);
// inverse of P[:, :3]*R, camera matrix and distortion of one camera (cv::initUndistortRectifyMap's inputs)
struct RectifyCoef { double iR[9]; double k1, k2, p1, p2, k3; double fx, fy, cx, cy; };
cudaError_t launch_rectify_maps(mvsv_ctx* c, int cam, const RectifyCoef& q);
cudaError_t launch_convert_maps(mvsv_ctx* c, int cam, const float* dmapx, const float* dmapy, size_t stride_elems);
cudaError_t launch_sgbm(mvsv_ctx* c, int B);
cudaError_t launch_bm(mvsv_ctx* c, int B);
int bm_lrcheck_max_width();
size_t tm_smem_bytes(int W, int k);
int tm_max_width();
cudaError_t launch_tm(mvsv_ctx* c, int B, int k, uint8_t* out, size_t opitch);
cudaError_t launch_xyz(mvsv_ctx* c, int B);
cudaError_t launch_means(mvsv_ctx* c, int B);
cudaError_t launch_minmax(mvsv_ctx* c, int B);
cudaError_t launch_median(mvsv_ctx* c, const int16_t* in, int16_t* out, int B);
cudaError_t launch_speckle(mvsv_ctx* c, const int16_t* img, int16_t* out, int B, int newVal, int maxSize, int maxDiff);
// fused previous-row sweep (csrc/sweep.cu): strip decomposition of a batch, scratch sizes, launch
struct SweepPlan { int NS = 0, NF = 0, Mmax = 0, threads = 0, G = 0, NR = 0; size_t smem = 0; };
void sweep_layout(int D, int* G, int* NR);
void sweep_plan(const mvsv_ctx* c, int B, int forcedNS, SweepPlan* p);
size_t sweep_scratch_bytes(const mvsv_ctx* c);
bool sweep_s8_ok(const mvsv_ctx* c, const SweepPlan& p);
cudaError_t launch_sweep(mvsv_ctx* c, int B, const SweepPlan& p, int bottomUp, bool s8);
int sgbm_choose_td_cluster(mvsv_ctx* c);
void sgbm_plane_geometry(const SgbmNorm& n, int W, int* NV, int* RP, int* JOFF);
bool sgbm_vsum_wide(const SgbmNorm& n);

#ifdef __CUDACC__
// ---- packed 16x2 helpers -----------------------------------------------------------------------------
__device__ __forceinline__ unsigned pk16(int v) { return ((unsigned)v & 0xffffu) * 0x10001u; }
__device__ __forceinline__ uint4 ld128(const void* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void st128(void* p, const uint4& v) { *reinterpret_cast<uint4*>(p) = v; }
#endif
