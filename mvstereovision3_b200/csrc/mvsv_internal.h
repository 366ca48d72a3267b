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
    int minD, D, Dp, G;          // Dp = padded disparity count (pixel stride), G = lanes per pixel (power of two)
    int dpl;                     // disparities per lane in the row scans: 8, or 16 when D > 256 (G = 32, Dp <= 16 G)
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
    KID_BM_WTA, KID_XYZ, KID_MEANS, KID_FILL, KID_MINMAX, KID_TM, KID_BM_LRCHECK, KID_POINTS, KID_DETECT, KID_COUNT
};
// a launch counted in mvsv_launch_count but never timed: the per-kernel timing brackets the engine's stream only
// (mvsv_profile_read waits for that stream), and the device downloads launch on the download stream
constexpr int KID_UNTIMED = -1;
extern const char* const kKernelNames[KID_COUNT];

struct ProfBracket { int kid; cudaEvent_t a, b; };

// One device allocation of T elements, the only owner of it: freed by reset() and by the destructor, on the current
// device (whoever releases an engine's buffer has made the engine's device current).  Converts to T* for the launchers.
template <class T>
class DeviceBuffer {
public:
    DeviceBuffer() = default;
    DeviceBuffer(DeviceBuffer&& o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
    DeviceBuffer& operator=(DeviceBuffer&& o) noexcept
    {
        if (this != &o) { reset(); p_ = o.p_; n_ = o.n_; o.p_ = nullptr; o.n_ = 0; }
        return *this;
    }
    ~DeviceBuffer() { reset(); }

    // exactly n elements, in place of what it held
    cudaError_t alloc(size_t n)
    {
        reset();
        const cudaError_t e = cudaMalloc(&p_, n * sizeof(T));
        if (e == cudaSuccess) n_ = n;
        else p_ = nullptr;
        return e;
    }
    // at least n elements: reallocates only when it holds fewer
    cudaError_t ensure(size_t n) { return p_ && n_ >= n ? cudaSuccess : alloc(n); }
    void reset()
    {
        if (p_) cudaFree(p_);
        p_ = nullptr;
        n_ = 0;
    }
    operator T*() const { return p_; }

private:
    T* p_ = nullptr;
    size_t n_ = 0;
};

// I/O slot (mvsv_set_io_slots): the buffers a compute call reads its inputs into and leaves its results in.  They
// exist once or twice; with two, the host->device copy of the next batch and the device->host copy of the previous
// one overlap the kernels of the current batch inside ONE engine (one set of cost volumes).  The slot is the only
// owner of these buffers; the launchers reach the slot of the compute in progress through io(c).
struct IoSlot {
    DeviceBuffer<uint8_t> rect[2];            // [B][H][pitch]
    DeviceBuffer<uint8_t> raw[2];             // [B][fh][raw_pitch], once rectification maps are installed
    DeviceBuffer<int16_t> disp;               // final disparities [B][H][W]
    DeviceBuffer<float> xyz;                  // [B][H][W][3], allocated by the first compute with MVSV_STAGE_XYZ
    // MVSV_STAGE_POINTS, allocated by the first compute with it: the packed point list ([B*H*W][3] at most) and the
    // frame offsets into it ([B+1]).  In the slot, because a download at age 1 reads them while the next compute runs.
    DeviceBuffer<float> points;
    DeviceBuffer<long long> offsets;
    DeviceBuffer<float> means;                // [B][nrois], once mean-disparity ROIs are set
    // MVSV_STAGE_DETECT, allocated by the first compute with it: the packed found obstacles ([B*nrois] at most) and the
    // frame offsets into them ([B+1]); in the slot for the same reason as the points
    DeviceBuffer<mvsv_obstacle> obstacles;
    DeviceBuffer<long long> det_offsets;
    cudaEvent_t done = nullptr;               // all kernels of the slot's last compute have finished
    // recorded on dl_stream after every download of the slot's results: a device download (mvsv_download_device) may
    // still be copying when its call returns, so whatever writes the slot next waits for it
    cudaEvent_t dl_done = nullptr;
    // mvsv_download_minmax_device: the reduction of the slot's disparities ([maxB][2]) and its int16 pairs.  Per slot, so that it never races with mvsv_download_minmax (Engine::minmax, on the engine's
    // stream) or with the download of the other slot.
    DeviceBuffer<int> minmax;
    DeviceBuffer<int16_t> minmax16;
    int B = 0;                                // frames of the slot's last compute; 0: it holds no results
    unsigned stages = 0;
};

// frames per thread of the remap kernel (csrc/filters.cu), and the largest chunk of one rig's frames it takes
constexpr int RM_FRAMES = 8;

// Device tables of mvsv_set_frame_rigs (one allocation of max_batch entries each), built on the host from the frame ->
// rig table.  The remap kernel expands a map entry once for up to RM_FRAMES frames, which must then share the rig: it
// walks `chunk`, runs of at most RM_FRAMES frames of one rig in `order`.
struct RigFrames {
    DeviceBuffer<int4> chunk;                 // (rig, first index into order, count <= RM_FRAMES, 0)
    DeviceBuffer<int> order;                  // frames sorted by rig, ascending within a rig
    DeviceBuffer<int> rig;                    // rig of each frame
    int nchunks = 0;
};

// What the rig-aware kernels read of every rig: the fixed-point maps and Q widened to double (k_xyz's QMat).
struct RigTables {
    const int2* map[2][MVSV_MAX_RIGS];
    double Q[MVSV_MAX_RIGS][16];
    // MVSV_STAGE_DETECT: (first, second) disparity range of every (rig, detector), Engine::det_range
    float det_range[MVSV_MAX_RIGS][MVSV_MAX_DETECTORS][2];
};

// one ROI of the detection table (mvsv_set_detection): its detector (-1: not tested) and calcCoordinate's image_x, image_y
struct DetRoi { int det; float x, y; int pad; };

// One engine on one device: its streams, events, volumes and I/O slots.  An mvsv_ctx (csrc/api.cu) splits every batch
// across one or more of them.
struct Engine {
    ~Engine();                                // destroys the streams and events; the buffers free themselves
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

    // rectification (device): per rig and camera, fixed-point maps for the rig's display ROI only.  All rigs share the
    // ROI size; rig r's ROI starts at roi_xy[r] of the frame.  Rig 0 is the single-rig engine.
    bool has_maps[MVSV_MAX_RIGS][2] = {};
    int roi_w = 0, roi_h = 0;
    int roi_xy[MVSV_MAX_RIGS][2] = {};
    DeviceBuffer<int2> map_xy[MVSV_MAX_RIGS][2];   // (ix, iy) = rint(map*32), saturated int32
    size_t raw_pitch = 0;
    // cv::resize(.., factor, factor) after the crop (Stereosystem::getRectifiedImagepair(sip, factor),
    // reference src/Stereosystem.cpp:279-315); off when resize_factor == 0
    double resize_factor = 0.0;
    DeviceBuffer<uint8_t> tm_out;             // [B][H][pitch], Disparity::tm
    DeviceBuffer<uint8_t> crop[2];            // [B][roi_h][crop_pitch]: remap output when a resize follows
    size_t crop_pitch = 0;

    size_t pitch = 0;                         // row pitch of the rectified images

    int nslots = 1, cur = 0;                  // I/O slots in use; the slot of the last (or current) compute
    IoSlot slot[2];
    cudaStream_t dl_stream = nullptr;         // result copies to host or device memory (mvsv_download*)

    bool has_sgbm = false, has_bm = false;
    mvsv_sgbm_params sgbm_raw{};
    SgbmNorm sg{};
    int td_nc = 0;               // strips per frame of the fused previous-row sweep at max_batch (0: independent passes)
    DeviceBuffer<uint16_t> sweep_halo;        // tagged border-pixel records of the strip hand-off (csrc/sweep.cu)
    int num_sms = 148;
    mvsv_bm_params bm_raw{};
    BmNorm bm{};
    // mvsv_set_bm_filters, kept across mvsv_set_bm_params and geometry changes: -1 / 0 = off
    int bm_d12 = -1, bm_speckle_win = 0, bm_speckle_range = 0;

    DeviceBuffer<uint2> recL;                 // left prefilter records [B][H][W] (a_s,lo_s,hi_s,a_r,lo_r,hi_r)
    DeviceBuffer<uint16_t> plR;               // right prefilter planes, reversed + padded: [6][B][H][vsRP]
    int vsNV = 0, vsRP = 0, vsJOFF = 0;
    DeviceBuffer<uint16_t> VS;                // [B][H][W1][Dp] vertical box sums of the pixel cost
    DeviceBuffer<uint16_t> C;                 // [B][H][W1][Dp] block cost
    DeviceBuffer<uint16_t> S;                 // [B][H][W1][Dp] aggregated cost
    DeviceBuffer<int> d2;                     // [B][H][W] (disp2cost<<16 | disp2)
    DeviceBuffer<int16_t> disp_raw;           // [B][H][W]
    DeviceBuffer<int16_t> disp_med;           // [B][H][W]
    DeviceBuffer<int> labels;                 // [B][H][W]
    DeviceBuffer<int> sizes;                  // [B][H][W]

    DeviceBuffer<uint8_t> bm_pre[2];          // [B][H][pitch]
    DeviceBuffer<int> bm_tex2;                // [B][H][W] texture: window sums of |L - cap|
    DeviceBuffer<uint16_t> bm_col;            // [B][H][width1][Dp]

    bool has_Q[MVSV_MAX_RIGS] = {};
    float Q[MVSV_MAX_RIGS][16];

    // mvsv_set_frame_rigs: frame i of a compute comes from rig frame_rig[i] (frames past its end: rig 0).  While every
    // frame of a compute comes from rig 0 the single-rig kernels run; otherwise the rig-aware ones, which read the
    // device tables below.
    std::vector<int> frame_rig;
    RigFrames rig_frames;
    DeviceBuffer<RigTables> rig_tables;       // device mirror of map_xy and Q; refreshed by a compute when rig_tables_dirty
    bool rig_tables_dirty = true;

    int nrois = 0;
    DeviceBuffer<int> rois;                   // [n][4]
    DeviceBuffer<int> minmax;                 // [B][2]
    DeviceBuffer<long long> pt_tiles;         // MVSV_STAGE_POINTS: per tile, its count, then its base (points_tiles)
    // mvsv_download_points_stream on a multi-device ctx: the point totals of the parts before this one, copied from
    // their slots on dl_stream (one entry per part of the ctx); k_points_out adds them up into this part's base
    DeviceBuffer<long long> pt_base;

    // mvsv_set_detection: the table (device copy of det_rois_h) of the nrois ROIs, the detectors' distances and the
    // disparity ranges they give with each rig's Q (recomputed when a Q or the table changes)
    bool has_det = false;
    int det_n = 0, ndet = 0;
    std::vector<DetRoi> det_rois_h;
    float det_dist[MVSV_MAX_DETECTORS][2] = {};
    float det_range[MVSV_MAX_RIGS][MVSV_MAX_DETECTORS][2] = {};
    DeviceBuffer<DetRoi> det_rois;
    DeviceBuffer<long long> det_counts;       // per frame: its number of hits, then its base (launch_detect)
};

// the I/O slot of the compute in progress (or of the last one)
inline IoSlot& io(Engine* c) { return c->slot[c->cur]; }

// RAII bracket: records CUDA events on the engine's stream around one kernel launch when profiling is on.
struct KernelTimer {
    Engine* c; int idx;
    cudaStream_t st;
    KernelTimer(Engine* ctx, int kid, cudaStream_t on = nullptr) : c(ctx), idx(-1), st(on ? on : ctx->stream)
    {
        ++c->launches;
        if (!c->prof || kid == KID_UNTIMED) return;
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
cudaError_t launch_remap(Engine* c, int cam, int B);
cudaError_t launch_remap_rigs(Engine* c, int cam, int B);      // frames of several rigs (mvsv_set_frame_rigs)
cudaError_t launch_resize(Engine* c, int cam, int B);
// inverse of P[:, :3]*R, camera matrix and distortion of one camera (cv::initUndistortRectifyMap's inputs)
struct RectifyCoef { double iR[9]; double k1, k2, p1, p2, k3; double fx, fy, cx, cy; };
cudaError_t launch_rectify_maps(Engine* c, int rig, int cam, const RectifyCoef& q);
cudaError_t launch_convert_maps(Engine* c, int rig, int cam, const float* dmapx, const float* dmapy, size_t stride_elems);
cudaError_t launch_sgbm(Engine* c, int B);
cudaError_t launch_bm(Engine* c, int B);
int bm_lrcheck_max_width();
size_t tm_smem_bytes(int W, int k);
int tm_max_width();
cudaError_t launch_tm(Engine* c, int B, int k, uint8_t* out, size_t opitch);
cudaError_t launch_xyz(Engine* c, int B);
cudaError_t launch_xyz_rigs(Engine* c, int B);                 // frames of several rigs (mvsv_set_frame_rigs)
cudaError_t launch_means(Engine* c, int B);
// MVSV_STAGE_POINTS of the current I/O slot: the point tiles of B frames of W x H (the size of Engine::pt_tiles), and the
// launch; `rigs`: frames of several rigs (mvsv_set_frame_rigs)
size_t points_tiles(int W, int H, int B);
cudaError_t launch_points(Engine* c, int B, bool rigs);
// MVSV_STAGE_DETECT of the current I/O slot, after launch_means: the found obstacles of B frames and their offsets;
// `rigs`: frames of several rigs (Q and ranges from Engine::rig_tables)
cudaError_t launch_detect(Engine* c, int B, bool rigs);
// Utility::calcMinMaxDisparity of slot s's disparities into mm ([s.B][2] int: lo, hi) on stream st; the fold turns B
// such pairs into the int16 pairs of mvsv_download_minmax
cudaError_t launch_minmax(Engine* c, const IoSlot& s, int* mm, cudaStream_t st);
cudaError_t launch_minmax_fold(Engine* c, const int* mm, int16_t* out, int B, cudaStream_t st);
// mvsv_download_points_stream, one part: slot s's frame offsets (nout of them) rebased by the sum of bases[0 .. nbases)
// into dst_offs, and the points that fit below `capacity` into dst (NULL: the offsets only), on dl_stream
cudaError_t launch_points_out(Engine* c, const IoSlot& s, const long long* bases, int nbases, long long* dst_offs, int nout,
                              float* dst, long long capacity);
// mvsv_download_obstacles_stream, one part: launch_points_out for slot s's found obstacles
cudaError_t launch_obstacles_out(Engine* c, const IoSlot& s, const long long* bases, int nbases, long long* dst_offs, int nout,
                                 mvsv_obstacle* dst, long long capacity);
cudaError_t launch_median(Engine* c, const int16_t* in, int16_t* out, int B);
cudaError_t launch_speckle(Engine* c, const int16_t* img, int16_t* out, int B, int newVal, int maxSize, int maxDiff);
// fused previous-row sweep (csrc/sweep.cu): strip decomposition of a batch, scratch sizes, launch
struct SweepPlan { int NS = 0, NF = 0, Mmax = 0, threads = 0, G = 0, NR = 0; size_t smem = 0; };
void sweep_layout(int D, int* G, int* NR);
void sweep_plan(const Engine* c, int B, int forcedNS, SweepPlan* p);
size_t sweep_scratch_bytes(const Engine* c);
bool sweep_s8_ok(const Engine* c, const SweepPlan& p);
cudaError_t launch_sweep(Engine* c, int B, const SweepPlan& p, int bottomUp, bool s8);
int sgbm_choose_td_cluster(Engine* c);
void sgbm_plane_geometry(const SgbmNorm& n, int W, int* NV, int* RP, int* JOFF);
bool sgbm_vsum_wide(const SgbmNorm& n);

#ifdef __CUDACC__
// ---- packed 16x2 helpers -----------------------------------------------------------------------------
__device__ __forceinline__ unsigned pk16(int v) { return ((unsigned)v & 0xffffu) * 0x10001u; }
__device__ __forceinline__ uint4 ld128(const void* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void st128(void* p, const uint4& v) { *reinterpret_cast<uint4*>(p) = v; }
#endif
