// C-ABI glue of libmvsv.so (include/mvsv.h): context, device buffers, parameter normalisation, stage sequencing.
#include "mvsv_internal.h"
#include <cmath>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <numeric>

const char* const kKernelNames[KID_COUNT] = {
    "remap", "sgbm_prefilter", "sgbm_vsum", "sgbm_h1", "sgbm_vdir", "sgbm_td", "sgbm_h2_wta", "median3", "ccl_rows", "ccl_vmerge",
    "ccl_flatten", "ccl_apply", "bm_prefilter", "bm_tex", "bm_colsum", "bm_wta", "xyz", "means", "fill", "minmax", "tm",
    "bm_lrcheck", "points"};

cudaError_t smem_limit(const void* kernel, int bytes)
{
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, int> limits;   // (kernel, device) -> bytes set there
    int dev = 0;
    MVSV_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    int& set = limits[{kernel, dev}];
    if (set == bytes) return cudaSuccess;
    MVSV_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    set = bytes;
    return cudaSuccess;
}

namespace {

thread_local std::string g_init_error;

inline size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

#define MVSV_CK(ctx, call)                                                                      \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                    \
            return e_ == cudaErrorMemoryAllocation ? MVSV_ERR_NOMEM : MVSV_ERR_CUDA;            \
        }                                                                                       \
    } while (0)

template <class C>    // an Engine, or the mvsv_ctx handle
int fail(C* c, int code, const std::string& msg)
{
    c->err = msg;
    return code;
}

// some rig holds (or is getting) a rectification map
bool any_maps(const Engine* c)
{
    for (int r = 0; r < MVSV_MAX_RIGS; ++r)
        if (c->has_maps[r][0] || c->has_maps[r][1] || c->map_xy[r][0] || c->map_xy[r][1]) return true;
    return false;
}

// the rigs frames 0 .. B-1 of a compute come from (bit r = rig r; frames past the mvsv_set_frame_rigs table: rig 0)
uint64_t rigs_of_batch(const Engine* c, int B)
{
    const int n = std::min(B, (int)c->frame_rig.size());
    uint64_t m = B > n ? 1u : 0u;
    for (int i = 0; i < n; ++i) m |= (uint64_t)1 << c->frame_rig[i];
    return m;
}

// The rig-aware kernels read every rig's map and Q from c->rig_tables.  The copy is queued on the engine's stream, so
// that a compute sees the Q's set before it was submitted, as the single-rig k_xyz does with its by-value Q.
int upload_rig_tables(Engine* c)
{
    if (!c->rig_tables_dirty) return MVSV_OK;
    RigTables t;
    for (int r = 0; r < MVSV_MAX_RIGS; ++r) {
        for (int cam = 0; cam < 2; ++cam) t.map[cam][r] = c->map_xy[r][cam];
        for (int i = 0; i < 16; ++i) t.Q[r][i] = (double)c->Q[r][i];
    }
    MVSV_CK(c, cudaMemcpyAsync(c->rig_tables, &t, sizeof(t), cudaMemcpyHostToDevice, c->stream));   // pageable: staged before it returns
    c->rig_tables_dirty = false;
    return MVSV_OK;
}

// Releases the slot's buffers sized by the image geometry (rectified images, disparities, XYZ, points, ROI means), and with
// `staging` the raw-frame staging too (the slot goes away).  The slot then holds no results.
void release_slot(IoSlot& s, bool staging)
{
    for (int i = 0; i < 2; ++i) {
        s.rect[i].reset();
        if (staging) s.raw[i].reset();
    }
    s.disp.reset(); s.xyz.reset(); s.points.reset(); s.offsets.reset(); s.means.reset();
    s.B = 0; s.stages = 0;
}

// Allocates what each live slot needs in the engine's present state and does not have yet: the rectified images and
// the (zeroed) disparities always, the raw-frame staging once rectification maps are installed, the ROI means once ROIs
// are set.  The XYZ and point buffers are left to the first compute that asks for them.
int ensure_slots(Engine* c)
{
    const size_t B = (size_t)c->maxB, npx = B * c->H * c->W, nimg = B * c->H * c->pitch;
    const bool maps = any_maps(c);
    for (int k = 0; k < c->nslots; ++k) {
        IoSlot& s = c->slot[k];
        for (int i = 0; i < 2; ++i) {
            MVSV_CK(c, s.rect[i].ensure(nimg));
            if (maps) MVSV_CK(c, s.raw[i].ensure(B * c->fh * c->raw_pitch));
        }
        if (!s.disp) {
            MVSV_CK(c, s.disp.alloc(npx));
            MVSV_CK(c, cudaMemsetAsync(s.disp, 0, npx * sizeof(int16_t), c->stream));
        }
        if (c->nrois > 0) MVSV_CK(c, s.means.ensure((size_t)c->nrois * B));
    }
    return MVSV_OK;
}

// StereoSGBM parameters p normalised for W x H images
int normalise_sgbm(Engine* c, const mvsv_sgbm_params* p, int W, int H, SgbmNorm* n)
{
    n->minD = p->minDisp;
    n->D = p->numDisp;
    if (n->D <= 0 || n->D % 8 != 0 || n->D > 256)
        return fail(c, MVSV_ERR_INVALID, "numDisp must be a positive multiple of 8 and <= 256");
    // pixel stride of the volumes = the sweep's lane layout (csrc/sweep.cu): numDisp rounded up to 8, 16 or 32;
    // the row-scan and cost kernels spread a pixel over the next power of two of lanes (8 disparities each)
    {
        int sg, snr;
        sweep_layout(n->D, &sg, &snr);
        n->Dp = sg * 2 * snr;
    }
    int g = 1;
    while (g * 8 < n->Dp) g <<= 1;
    n->G = g;
    n->bs = p->blockSize > 0 ? p->blockSize : 5;
    n->SW2 = n->SH2 = n->bs / 2;
    n->ftzero = std::max(p->preFilterCap, 15) | 1;
    n->uniq = p->uniquenessRatio >= 0 ? p->uniquenessRatio : 10;
    n->d12 = p->disp12MaxDiff > 0 ? p->disp12MaxDiff : 1;
    n->P1 = p->P1 > 0 ? p->P1 : 2;
    n->P2 = std::max(p->P2 > 0 ? p->P2 : 5, n->P1 + 1);
    n->maxD = n->minD + n->D;
    n->minX1 = std::max(n->maxD, 0);
    n->maxX1 = W + std::min(n->minD, 0);
    n->W1 = n->maxX1 - n->minX1;
    n->INV = (n->minD - 1) * 16;
    n->mode = p->disparityMode == 1 ? 1 : 0;   // reference src/disparity.cpp:92-95
    n->npaths = n->mode ? 8 : 5;
    n->speckleWin = p->speckleWindowSize;
    n->speckleRange = p->speckleRange;
    n->vsWide = 0;
    if (n->ftzero > 127) return fail(c, MVSV_ERR_INVALID, "preFilterCap > 127 is outside the supported range");
    if (n->uniq > 100) return fail(c, MVSV_ERR_INVALID, "uniquenessRatio > 100");
    const long long eff = 2 * n->SH2 + 1;
    if (eff * eff * (2 * n->ftzero + 63) + n->P2 > 32767)
        return fail(c, MVSV_ERR_INVALID,
                    "blockSize^2*(2*ftzero+63)+P2 > 32767: int16 overflow regime of OpenCV is outside the bit-exact contract");
    if (n->INV < -32768 || (n->maxD) * 16 > 32767) return fail(c, MVSV_ERR_INVALID, "disparity range does not fit CV_16S");
    n->vsWide = sgbm_vsum_wide(*n) ? 1 : 0;
    if (n->W1 > 0 && (long long)H * n->W1 * n->Dp >= (1ll << 31))
        return fail(c, MVSV_ERR_UNSUPPORTED, "cost volume of one frame exceeds 2^31 cells");
    return MVSV_OK;
}

int ensure_sgbm_volumes(Engine* c)
{
    const SgbmNorm& n = c->sg;
    if (n.W1 <= 0) return MVSV_OK;
    int nv, rp, joff;
    sgbm_plane_geometry(n, c->W, &nv, &rp, &joff);
    const size_t need = (size_t)c->maxB * c->H * n.W1 * n.Dp;
    for (DeviceBuffer<uint16_t>* v : {&c->VS, &c->C, &c->S}) MVSV_CK(c, v->ensure(need));
    MVSV_CK(c, c->sweep_halo.ensure(sweep_scratch_bytes(c) / sizeof(uint16_t)));   // strip-border records of the fused sweep
    if (!c->plR || nv != c->vsNV || rp != c->vsRP || joff != c->vsJOFF) {
        const size_t elems = (size_t)6 * c->maxB * c->H * rp;
        MVSV_CK(c, c->plR.alloc(elems));
        MVSV_CK(c, cudaMemsetAsync(c->plR, 0, elems * sizeof(uint16_t), c->stream));   // the padding around each row stays zero
        c->vsNV = nv; c->vsRP = rp; c->vsJOFF = joff;
    }
    return MVSV_OK;
}

// StereoBM parameters p normalised for images W wide
int normalise_bm(Engine* c, const mvsv_bm_params* p, int W, BmNorm* n)
{
    n->D = p->numDisp; n->bs = p->blockSize; n->cap = p->preFilterCap; n->tex = p->textureThreshold; n->uniq = p->uniquenessRatio;
    if (n->D <= 0 || n->D % 16 != 0 || n->D > 256) return fail(c, MVSV_ERR_INVALID, "BM numDisp must be a positive multiple of 16 and <= 256");
    if (n->bs < 5 || n->bs > 255 || n->bs % 2 == 0) return fail(c, MVSV_ERR_INVALID, "BM blockSize must be odd, 5..255");
    if (n->cap < 1 || n->cap > 63) return fail(c, MVSV_ERR_INVALID, "BM preFilterCap must be 1..63");
    if (n->tex < 0 || n->uniq < 0) return fail(c, MVSV_ERR_INVALID, "BM textureThreshold/uniquenessRatio must be >= 0");
    if ((long long)n->bs * n->bs * 2 * n->cap > 65535) return fail(c, MVSV_ERR_INVALID, "BM blockSize^2*2*cap > 65535 unsupported");
    int g = 2;
    while (g * 8 < n->D) g <<= 1;
    n->G = g; n->Dp = n->D; n->w2 = n->bs / 2;      // lanes: next power of two; storage stride: numDisp itself
    n->lofs = n->D - 1; n->width1 = W - n->D + 1; n->FILT = -16;
    n->col8 = n->bs * 2 * n->cap <= 255;
    return MVSV_OK;
}

int ensure_bm_volumes(Engine* c)
{
    const BmNorm& n = c->bm;
    if (n.width1 < 1) return MVSV_OK;
    MVSV_CK(c, c->bm_col.ensure((size_t)c->maxB * c->H * n.width1 * n.Dp));
    return MVSV_OK;
}

// What the matcher sees under a geometry (the frame, or the display ROI, possibly resized)
struct Geometry {
    int W, H;
    SgbmNorm sg;     // the matcher parameters normalised for W x H (while set)
    BmNorm bm;
};

// The size of the images the matcher would see with display ROI roi_w x roi_h once some rig holds maps (`maps`; the
// frame otherwise), resized by `factor` when that is on, and the matcher parameters normalised for it.  Every check
// that can reject a geometry runs here, before the caller changes anything: a rejected geometry leaves the engine as
// it was.
int plan_geometry(Engine* c, bool maps, int roi_w, int roi_h, double factor, Geometry* g)
{
    g->W = maps ? roi_w : c->fw;
    g->H = maps ? roi_h : c->fh;
    if (maps && factor > 0.0) {
        // cv::resize: dsize = Size(saturate_cast<int>(w*fx), saturate_cast<int>(h*fy)), round half to even
        g->W = (int)lrint((double)g->W * factor);
        g->H = (int)lrint((double)g->H * factor);
        if (g->W < 2 || g->H < 1 || g->W > 16384 || g->H > 16384) return fail(c, MVSV_ERR_INVALID, "resized image out of range");
    }
    g->sg = c->sg;
    g->bm = c->bm;
    int rc = MVSV_OK;
    if (c->has_sgbm) rc = normalise_sgbm(c, &c->sgbm_raw, g->W, g->H, &g->sg);
    if (!rc && c->has_bm) rc = normalise_bm(c, &c->bm_raw, g->W, &g->bm);
    if (rc) return rc;
    // the connected-components labels of the speckle filter are int indices over the whole batch
    if ((size_t)c->maxB * g->H * round_up((size_t)g->W, 16) >= ((size_t)1 << 31))
        return fail(c, MVSV_ERR_UNSUPPORTED, "max_batch * height * width must stay below 2^31 pixels");
    return MVSV_OK;
}

// Installs geometry g (plan_geometry) once the engine's ROI, maps and resize factor describe it, with the engine's stream
// synchronised.  A new image size reallocates every buffer sized by it and drops the mean-disparity ROIs; the crop
// buffers follow the display ROI.
int apply_geometry(Engine* c, const Geometry& g)
{
    if (g.W != c->W || g.H != c->H) {
        c->W = g.W; c->H = g.H;
        // mean-disparity ROIs are coordinates of the old map: drop them (run() asks for new ones)
        c->rois.reset();
        c->nrois = 0;
        for (IoSlot& s : c->slot) release_slot(s, false);
        for (auto& b : c->bm_pre) b.reset();
        c->recL.reset(); c->d2.reset(); c->disp_raw.reset(); c->disp_med.reset(); c->labels.reset(); c->sizes.reset();
        c->bm_tex2.reset(); c->minmax.reset(); c->tm_out.reset(); c->pt_tiles.reset();
        // 16-byte aligned rows; when the width already is (752, 1920, 3840, ...) a batch is one contiguous block and
        // host <-> device transfers are single linear copies instead of strided 2-D copies of many short rows
        c->pitch = round_up((size_t)c->W, 16);
        const size_t B = (size_t)c->maxB, npx = B * c->H * c->W, nimg = B * c->H * c->pitch;
        // the slot buffers first: allocated after the scratch buffers below, the StereoBM configuration ran 0.4 % slower
        // (49.35 K against 49.55 K frames/s on a B200 at 1000 W)
        int rc = ensure_slots(c);
        if (rc) return rc;
        for (auto& b : c->bm_pre) MVSV_CK(c, b.alloc(nimg + 64));   // the BM column-sum kernel reads whole aligned words
        MVSV_CK(c, c->recL.alloc(npx));
        MVSV_CK(c, c->d2.alloc(npx));
        MVSV_CK(c, c->disp_raw.alloc(npx));
        MVSV_CK(c, c->disp_med.alloc(npx));
        MVSV_CK(c, c->labels.alloc(npx));
        MVSV_CK(c, c->sizes.alloc(npx));
        MVSV_CK(c, c->bm_tex2.alloc(npx));
        // the volumes grow within one geometry; a new one starts them afresh
        for (DeviceBuffer<uint16_t>* v : {&c->VS, &c->C, &c->S, &c->plR, &c->sweep_halo, &c->bm_col}) v->reset();
        if (c->has_sgbm) {
            c->sg = g.sg;
            c->td_nc = sgbm_choose_td_cluster(c);
            rc = ensure_sgbm_volumes(c);
            if (rc) { c->has_sgbm = false; return rc; }
        }
        if (c->has_bm) {
            c->bm = g.bm;
            rc = ensure_bm_volumes(c);
            if (rc) { c->has_bm = false; return rc; }
        }
    }
    for (auto& b : c->crop) b.reset();
    if (any_maps(c) && c->resize_factor > 0.0) {
        c->crop_pitch = round_up((size_t)c->roi_w, 16);
        for (auto& b : c->crop) MVSV_CK(c, b.alloc((size_t)c->maxB * c->roi_h * c->crop_pitch));
    }
    return MVSV_OK;
}

int bind(Engine* c)
{
    MVSV_CK(c, cudaSetDevice(c->device));
    return MVSV_OK;
}

// host -> device copy of `batch` images (w bytes wide, h rows) into dst[b][h][dpitch]
int upload_images(Engine* c, uint8_t* dst, size_t dpitch, const uint8_t* src, size_t sstride, size_t frame_stride, int w,
                  int h, int batch, bool device_src)
{
    // device inputs may live on another device than the engine (the parts of a multi-device ctx all read one batch):
    // cudaMemcpyDefault lets unified addressing find both ends, and copies peer to peer where they differ
    const cudaMemcpyKind kind = device_src ? cudaMemcpyDefault : cudaMemcpyHostToDevice;
    cudaStream_t st = device_src ? c->stream : c->copy_stream;
    if (sstride == (size_t)w && dpitch == (size_t)w && (batch == 1 || frame_stride == (size_t)w * h)) {
        MVSV_CK(c, cudaMemcpyAsync(dst, src, (size_t)w * h * batch, kind, st));
    } else if (frame_stride == sstride * (size_t)h) {
        MVSV_CK(c, cudaMemcpy2DAsync(dst, dpitch, src, sstride, (size_t)w, (size_t)h * batch, kind, st));
    } else {
        for (int b = 0; b < batch; ++b)
            MVSV_CK(c, cudaMemcpy2DAsync(dst + (size_t)b * h * dpitch, dpitch, src + (size_t)b * frame_stride, sstride, (size_t)w,
                                         (size_t)h, kind, st));
    }
    return MVSV_OK;
}

static int inputs_uploaded(Engine* c, bool device_src)
{
    if (device_src) return MVSV_OK;
    MVSV_CK(c, cudaEventRecord(c->ev_h2d, c->copy_stream));
    MVSV_CK(c, cudaStreamWaitEvent(c->stream, c->ev_h2d, 0));
    return MVSV_OK;
}

// the I/O slot the next compute takes; its previous results must have been downloaded by then (mvsv_set_io_slots)
IoSlot& next_slot(Engine* c) { return c->slot[(c->cur + 1) % c->nslots]; }

// Takes it, empty: the compute fills in its frames once every step has been queued, so that if a step fails a download
// reports the failure instead of returning the frames of an older compute.
void take_slot(Engine* c)
{
    c->cur = (c->cur + 1) % c->nslots;
    io(c).B = 0;
    io(c).stages = 0;
}

// what the XYZ, POINTS and MEANS stages need of the engine and of the slot they write to; `rigs`: the rigs of the batch's
// frames
int check_consumers(Engine* c, const IoSlot& slot, unsigned stages, uint64_t rigs)
{
    if (stages & (MVSV_STAGE_XYZ | MVSV_STAGE_POINTS))
        for (int r = 0; r < MVSV_MAX_RIGS; ++r)
            if (((rigs >> r) & 1) && !c->has_Q[r])
                return fail(c, MVSV_ERR_STATE, r == 0 ? "mvsv_set_Q not called" : "no Q for rig " + std::to_string(r) + " (mvsv_set_Q_rig)");
    if ((stages & MVSV_STAGE_MEANS) && (c->nrois < 1 || !c->rois || !slot.means))
        return fail(c, MVSV_ERR_STATE, "no mean-disparity ROIs (mvsv_set_mean_rois; a geometry change drops them)");
    return MVSV_OK;
}

// The buffers the XYZ and POINTS stages write, in the slot they write to (and the engine's point tiles)
int ensure_consumers(Engine* c, IoSlot& slot, unsigned stages)
{
    const size_t npx = (size_t)c->maxB * c->H * c->W;
    if (stages & MVSV_STAGE_XYZ) MVSV_CK(c, slot.xyz.ensure(npx * 3));
    if (stages & MVSV_STAGE_POINTS) {
        MVSV_CK(c, slot.points.ensure(npx * 3));
        MVSV_CK(c, slot.offsets.ensure((size_t)c->maxB + 1));
        MVSV_CK(c, c->pt_tiles.ensure(points_tiles(c->W, c->H, c->maxB)));
    }
    return MVSV_OK;
}

// What a compute of `batch` frames needs of engine c: arguments, state, the rigs of its frames, allocations.  It takes
// no I/O slot, so that a rejected compute leaves the results of earlier ones downloadable.
int compute_check(Engine* c, size_t lstride, size_t rstride, int batch, unsigned stages)
{
    int rc = bind(c);
    if (rc) return rc;
    IoSlot& slot = next_slot(c);
    const bool rectify = stages & MVSV_STAGE_RECTIFY;
    if ((stages & MVSV_STAGE_SGBM) && (stages & MVSV_STAGE_BM)) return fail(c, MVSV_ERR_INVALID, "choose SGBM or BM, not both");
    if ((stages & MVSV_STAGE_SGBM) && !c->has_sgbm) return fail(c, MVSV_ERR_STATE, "mvsv_set_sgbm_params not called");
    if ((stages & MVSV_STAGE_BM) && !c->has_bm) return fail(c, MVSV_ERR_STATE, "mvsv_set_bm_params not called");
    const uint64_t rigs = rigs_of_batch(c, batch);
    rc = check_consumers(c, slot, stages, rigs);
    if (rc) return rc;
    if (rectify)
        for (int r = 0; r < MVSV_MAX_RIGS; ++r)
            if (((rigs >> r) & 1) && (!c->has_maps[r][0] || !c->has_maps[r][1]))
                return fail(c, MVSV_ERR_STATE, r == 0 ? "rectify maps missing (mvsv_upload_rectify_maps)"
                                                      : "rectify maps of rig " + std::to_string(r) + " missing (mvsv_upload_rectify_maps_rig)");
    if ((stages & MVSV_STAGE_BM) && c->bm_d12 >= 0 && c->W > bm_lrcheck_max_width())
        return fail(c, MVSV_ERR_UNSUPPORTED, "BM left-right check (disp12MaxDiff >= 0): image wider than 4096");
    const int iw = rectify ? c->fw : c->W;
    if (lstride < (size_t)iw || rstride < (size_t)iw)
        return fail(c, MVSV_ERR_INVALID, rectify ? "stride smaller than frame width" : "stride smaller than image width");
    if (stages & MVSV_STAGE_SGBM) rc = ensure_sgbm_volumes(c);
    else if (stages & MVSV_STAGE_BM) rc = ensure_bm_volumes(c);
    if (rc) return rc;
    return ensure_consumers(c, slot, stages);
}

// Queues engine c's copies and kernels of a compute of `batch` frames; they fill the I/O slot it has taken (take_slot).
int compute_submit(Engine* c, const uint8_t* left, size_t lstride, const uint8_t* right, size_t rstride, size_t frame_stride,
                   int batch, unsigned stages, bool device_src)
{
    const IoSlot& slot = io(c);
    const bool rectify = stages & MVSV_STAGE_RECTIFY;
    const int iw = rectify ? c->fw : c->W, ih = rectify ? c->fh : c->H;
    // frames of rigs other than 0: the rig-aware remap, XYZ and point kernels
    const bool multi = rigs_of_batch(c, batch) != 1;
    int rc = bind(c);
    if (rc) return rc;
    // host inputs: the copies wait for the slot's previous compute (which may still read the input buffers), the
    // kernels wait for the copies
    if (!device_src) MVSV_CK(c, cudaStreamWaitEvent(c->copy_stream, slot.done, 0));
    const DeviceBuffer<uint8_t>* dst = rectify ? slot.raw : slot.rect;
    const size_t dpitch = rectify ? c->raw_pitch : c->pitch;
    rc = upload_images(c, dst[0], dpitch, left, lstride, frame_stride, iw, ih, batch, device_src);
    if (!rc) rc = upload_images(c, dst[1], dpitch, right, rstride, frame_stride, iw, ih, batch, device_src);
    if (!rc) rc = inputs_uploaded(c, device_src);
    if (rc) return rc;
    if (multi && (rectify || (stages & (MVSV_STAGE_XYZ | MVSV_STAGE_POINTS)))) {
        rc = upload_rig_tables(c);
        if (rc) return rc;
    }
    if (rectify)
        for (int cam = 0; cam < 2; ++cam) {
            MVSV_CK(c, multi ? launch_remap_rigs(c, cam, batch) : launch_remap(c, cam, batch));
            if (c->resize_factor > 0.0) MVSV_CK(c, launch_resize(c, cam, batch));
        }
    if (stages & MVSV_STAGE_SGBM) MVSV_CK(c, launch_sgbm(c, batch));
    else if (stages & MVSV_STAGE_BM) MVSV_CK(c, launch_bm(c, batch));
    if (stages & MVSV_STAGE_XYZ) MVSV_CK(c, multi ? launch_xyz_rigs(c, batch) : launch_xyz(c, batch));
    if (stages & MVSV_STAGE_POINTS) MVSV_CK(c, launch_points(c, batch, multi));
    if (stages & MVSV_STAGE_MEANS) MVSV_CK(c, launch_means(c, batch));
    MVSV_CK(c, cudaEventRecord(slot.done, c->stream));
    MVSV_CK(c, cudaEventRecord(c->ev_done, c->stream));
    return MVSV_OK;
}

// Queues the copies of the results a compute left in I/O slot `k` to the host on the download stream (so that they
// overlap kernels submitted later); download_wait waits for them.
int download_enqueue(Engine* c, int k, int16_t* disp, size_t dstride, uint8_t* rectL, uint8_t* rectR, size_t rstride,
                     float* xyz, float* means)
{
    int rc = bind(c);
    if (rc) return rc;
    IoSlot& s = c->slot[k];
    const int B = s.B;
    cudaStream_t st = c->dl_stream;
    MVSV_CK(c, cudaStreamWaitEvent(st, s.done, 0));
    if (disp) {
        if (dstride < (size_t)c->W * 2) return fail(c, MVSV_ERR_INVALID, "disparity stride too small");
        if (dstride == (size_t)c->W * 2)
            MVSV_CK(c, cudaMemcpyAsync(disp, s.disp, (size_t)c->W * 2 * c->H * B, cudaMemcpyDeviceToHost, st));
        else
            MVSV_CK(c, cudaMemcpy2DAsync(disp, dstride, s.disp, (size_t)c->W * 2, (size_t)c->W * 2, (size_t)c->H * B,
                                         cudaMemcpyDeviceToHost, st));
    }
    uint8_t* r[2] = {rectL, rectR};
    for (int i = 0; i < 2; ++i)
        if (r[i]) {
            if (rstride < (size_t)c->W) return fail(c, MVSV_ERR_INVALID, "rectified stride too small");
            MVSV_CK(c, cudaMemcpy2DAsync(r[i], rstride, s.rect[i], c->pitch, (size_t)c->W, (size_t)c->H * B, cudaMemcpyDeviceToHost, st));
        }
    if (xyz) {
        if (!s.xyz || !(s.stages & MVSV_STAGE_XYZ)) return fail(c, MVSV_ERR_STATE, "XYZ stage was not computed");
        MVSV_CK(c, cudaMemcpyAsync(xyz, s.xyz, (size_t)B * c->H * c->W * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    if (means) {
        if (!s.means || !(s.stages & MVSV_STAGE_MEANS)) return fail(c, MVSV_ERR_STATE, "MEANS stage was not computed");
        MVSV_CK(c, cudaMemcpyAsync(means, s.means, (size_t)B * c->nrois * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    return MVSV_OK;
}

int download_wait(Engine* c)
{
    MVSV_CK(c, cudaStreamSynchronize(c->dl_stream));
    return MVSV_OK;
}

// mvsv_download_points, first phase: the frame offsets of the point list in I/O slot `k` (B + 1 values) into `offsets`.
// The copy is a few bytes to pageable memory, which the CUDA runtime completes before it returns.
int points_offsets(Engine* c, int k, std::vector<long long>& offsets)
{
    int rc = bind(c);
    if (rc) return rc;
    const IoSlot& s = c->slot[k];
    offsets.resize((size_t)s.B + 1);
    MVSV_CK(c, cudaStreamWaitEvent(c->dl_stream, s.done, 0));
    MVSV_CK(c, cudaMemcpyAsync(offsets.data(), s.offsets, offsets.size() * sizeof(long long), cudaMemcpyDeviceToHost, c->dl_stream));
    return download_wait(c);
}

// second phase: queues the copy of the slot's n points to `points` on the download stream (download_wait waits for it)
int points_enqueue(Engine* c, int k, float* points, long long n)
{
    int rc = bind(c);
    if (rc) return rc;
    if (n > 0) MVSV_CK(c, cudaMemcpyAsync(points, c->slot[k].points, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->dl_stream));
    return MVSV_OK;
}

// mvsv_download_minmax of the current I/O slot = minmax_launch + minmax_read
int minmax_launch(Engine* c)
{
    int rc = bind(c);
    if (rc) return rc;
    MVSV_CK(c, c->minmax.ensure((size_t)c->maxB * 2));
    MVSV_CK(c, launch_minmax(c, io(c).B));
    return MVSV_OK;
}

int minmax_read(Engine* c, int16_t* minmax)
{
    int rc = bind(c);
    if (rc) return rc;
    const int B = io(c).B;
    std::vector<int> h((size_t)2 * B);
    MVSV_CK(c, cudaMemcpyAsync(h.data(), c->minmax, h.size() * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < B; ++i) {
        const bool none = h[2 * i + 1] <= 0;
        minmax[2 * i] = none ? 0 : (int16_t)h[2 * i];
        minmax[2 * i + 1] = none ? 0 : (int16_t)h[2 * i + 1];
    }
    return MVSV_OK;
}

// Engine c's frame -> rig table (frames past its end: rig 0) and the device tables built from it.  Waits for c's
// stream, so that computes already submitted keep their assignment.
int set_rigs(Engine* c, const std::vector<int>& rig_of_frame)
{
    int rc = bind(c);
    if (rc) return rc;
    // every frame of max_batch: the given rig, rig 0 past the table; the order sorted by rig (stable), cut into remap chunks
    const int B = c->maxB;
    std::vector<int> rig(B, 0);
    std::copy(rig_of_frame.begin(), rig_of_frame.end(), rig.begin());
    std::vector<int> order(B);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return rig[a] < rig[b]; });
    std::vector<int4> chunk;
    for (int i = 0; i < B; ++i) {
        const int r = rig[order[i]];
        if (chunk.empty() || chunk.back().x != r || chunk.back().z == RM_FRAMES) chunk.push_back(make_int4(r, i, 0, 0));
        ++chunk.back().z;
    }
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    RigFrames& t = c->rig_frames;
    MVSV_CK(c, t.chunk.ensure(B));
    MVSV_CK(c, t.order.ensure(B));
    MVSV_CK(c, t.rig.ensure(B));
    if (!c->rig_tables) {
        MVSV_CK(c, c->rig_tables.alloc(1));
        c->rig_tables_dirty = true;
    }
    // Until the copies below have all been queued the engine holds a table longer than any it accepts, which its
    // computes read as rig 0 and which equals no slice a compute hands it (send_rigs): after a failure here the next
    // compute sends the table again rather than trusting device tables that were only half written.
    c->frame_rig.assign((size_t)B + 1, 0);
    MVSV_CK(c, cudaMemcpyAsync(t.chunk, chunk.data(), chunk.size() * sizeof(int4), cudaMemcpyHostToDevice, c->stream));
    MVSV_CK(c, cudaMemcpyAsync(t.order, order.data(), (size_t)B * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    MVSV_CK(c, cudaMemcpyAsync(t.rig, rig.data(), (size_t)B * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    t.nchunks = (int)chunk.size();
    c->frame_rig = rig_of_frame;
    return MVSV_OK;
}

}  // namespace

// The handle of include/mvsv.h: the engines ("parts") a ctx splits its batches across, one for an mvsv_init ctx.  It
// holds no device state of its own.
struct mvsv_ctx {
    std::vector<Engine*> parts;              // part k: an engine of ceil(max_batch / n) frames on device[k]
    std::vector<int> device;
    int maxB = 0;                            // frames of all parts
    std::vector<int> frame_rig;              // the whole frame -> rig table (mvsv_set_frame_rigs)
    bool broken = false;                     // a setter failed in a way that can have left the parts different
    std::string err;
};

namespace {

int usable(mvsv_ctx* c)
{
    if (!c) return MVSV_ERR_INVALID;
    if (c->broken)
        return fail(c, MVSV_ERR_STATE, "an earlier call failed on one part only, so the parts no longer hold the same state ("
                                       "only mvsv_destroy, mvsv_last_error and mvsv_get_info remain): " + c->err);
    return MVSV_OK;
}

// Runs f on part k.  The part's error text becomes the ctx's: with several parts that of a failure, prefixed with the
// part and its device; with one, any text f set, so that a rejection without text leaves the previous one in place.
template <class F>
auto on_part(mvsv_ctx* c, int k, F&& f) -> decltype(f(c->parts[k]))
{
    Engine* p = c->parts[k];
    p->err.clear();
    const auto rc = f(p);
    if (c->parts.size() == 1) {
        if (!p->err.empty()) c->err = p->err;
    } else if (rc < 0) {
        c->err = "part " + std::to_string(k) + " (device " + std::to_string(c->device[k]) + "): " + p->err;
    }
    return rc;
}

// Runs f on every part in order, up to the first failure.  `setter`: f changes engine state.  The parts hold the same
// state, so an argument or state rejection comes from part 0 before any part changed; a CUDA or allocation error can
// leave part 0 half changed, and any failure past part 0 leaves the parts before it changed.  Such a failure marks a
// ctx of several parts broken.
template <class F>
int each(mvsv_ctx* c, bool setter, F&& f)
{
    int rc = usable(c);
    if (rc) return rc;
    for (int k = 0; k < (int)c->parts.size() && !rc; ++k) {
        rc = on_part(c, k, f);
        if (rc && setter && c->parts.size() > 1 && (k > 0 || rc == MVSV_ERR_CUDA || rc == MVSV_ERR_NOMEM)) c->broken = true;
    }
    return rc;
}

// mvsv_tm, profiling and the test hooks: on the only part; a ctx of several parts does not offer them
template <class F>
auto single(mvsv_ctx* c, const char* what, F&& f) -> decltype(f(c->parts[0]))
{
    const int rc = usable(c);
    if (rc) return rc;
    if (c->parts.size() > 1)
        return fail(c, MVSV_ERR_UNSUPPORTED, std::string(what) + " is not available on a multi-device ctx (mvsv_init_devices); "
                                                                  "call it on a single-device engine");
    return on_part(c, 0, f);
}

// Part k holds frames [first[k], first[k + 1]) of the compute in I/O slot s: every compute advances the slots of all
// parts, so they hold the same one.
std::vector<int> firsts(const mvsv_ctx* c, int s)
{
    std::vector<int> first(c->parts.size() + 1, 0);
    for (size_t k = 0; k < c->parts.size(); ++k) first[k + 1] = first[k] + c->parts[k]->slot[s].B;
    return first;
}

// Part k, whose frames of a compute start at frame `first` of the batch, holds the ctx's table from that frame on, as
// far as the part's capacity reaches (a single part: the whole table).  It receives it unless it holds it already.
int send_rigs(mvsv_ctx* c, int k, int first)
{
    const std::vector<int>& all = c->frame_rig;
    const int n = (int)all.size();
    const auto a = all.begin() + std::min(first, n), b = all.begin() + std::min(first + c->parts[k]->maxB, n);
    if (std::equal(a, b, c->parts[k]->frame_rig.begin(), c->parts[k]->frame_rig.end())) return MVSV_OK;
    const std::vector<int> slice(a, b);
    return on_part(c, k, [&](Engine* p) { return set_rigs(p, slice); });
}

// Part k computes the frames [floor(k*b/n), floor((k+1)*b/n)) of a batch of b: contiguous shares keep every host copy
// one bulk or 2-D copy per buffer and part.
int run(mvsv_ctx* c, const uint8_t* left, size_t lstride, const uint8_t* right, size_t rstride, size_t frame_stride, int batch,
        unsigned stages, bool device_src)
{
    int rc = usable(c);
    if (rc) return rc;
    if (!left || !right || batch < 1 || batch > c->maxB) return fail(c, MVSV_ERR_INVALID, "bad image pointers or batch size");
    const int n = (int)c->parts.size();
    std::vector<int> first(n + 1);
    for (int k = 0; k <= n; ++k) first[k] = (int)((long long)k * batch / n);
    // every part that gets frames checks them (and allocates what they need) before any part takes an I/O slot
    for (int k = 0; k < n && !rc; ++k)
        if (first[k] < first[k + 1]) {
            rc = send_rigs(c, k, first[k]);
            if (!rc)
                rc = on_part(c, k, [&](Engine* p) { return compute_check(p, lstride, rstride, first[k + 1] - first[k], stages); });
        }
    if (rc) return rc;
    // every part takes its next slot, one without frames too, so that the slots of all parts hold the same compute
    for (Engine* p : c->parts) take_slot(p);
    for (int k = 0; k < n; ++k)
        if (first[k] < first[k + 1]) {
            rc = on_part(c, k, [&](Engine* p) {
                return compute_submit(p, left + first[k] * frame_stride, lstride, right + first[k] * frame_stride, rstride,
                                      frame_stride, first[k + 1] - first[k], stages, device_src);
            });
            if (rc) return rc;
        }
    for (int k = 0; k < n; ++k) {
        IoSlot& s = io(c->parts[k]);
        s.B = first[k + 1] - first[k];
        s.stages = s.B ? stages : 0;
    }
    return MVSV_OK;
}

}  // namespace

Engine::~Engine()
{
    for (auto& b : brackets) { cudaEventDestroy(b.a); cudaEventDestroy(b.b); }
    for (cudaEvent_t ev : ev_free) cudaEventDestroy(ev);
    for (cudaEvent_t ev : ev_chunk)
        if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : {timer_a, timer_b, ev_h2d, ev_done, ev_join, slot[0].done, slot[1].done})
        if (ev) cudaEventDestroy(ev);
    for (cudaStream_t st : {aux_stream, copy_stream, dl_stream, stream})
        if (st) cudaStreamDestroy(st);
}

extern "C" {

static void destroy_engine(Engine* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->dl_stream) cudaStreamSynchronize(c->dl_stream);
    if (c->stream) cudaStreamSynchronize(c->stream);
    delete c;
}

// an engine on `device`; the text of a failure goes to mvsv_last_error(NULL)
static int init_engine(int device, int frame_width, int frame_height, int max_batch, Engine** out)
{
    if (frame_width < 2 || frame_height < 1 || frame_width > 16384 || frame_height > 16384 || max_batch < 1 || max_batch > 32767) {
        g_init_error = "mvsv_init: invalid frame size or batch";
        return MVSV_ERR_INVALID;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0) {
        g_init_error = std::string("mvsv_init: no CUDA device (") + cudaGetErrorString(e) + "); this engine has no CPU fallback";
        return MVSV_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) {
        g_init_error = "mvsv_init: device index out of range";
        return MVSV_ERR_INVALID;
    }
    Engine* c = new (std::nothrow) Engine();
    if (!c) return MVSV_ERR_NOMEM;
    c->device = device; c->fw = frame_width; c->fh = frame_height; c->maxB = max_batch;
    c->raw_pitch = round_up((size_t)frame_width, 16);
    auto bail = [&](cudaError_t ee, const char* what) {
        g_init_error = std::string("mvsv_init: ") + what + ": " + cudaGetErrorString(ee);
        destroy_engine(c);
        return ee == cudaErrorMemoryAllocation ? MVSV_ERR_NOMEM : MVSV_ERR_CUDA;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail(e, "cudaSetDevice");
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail(e, "cudaGetDeviceProperties");
    c->num_sms = prop.multiProcessorCount;
    if (prop.major != 10 || prop.minor != 0) {
        // the library holds sm_100a code only (arch-specific, no PTX): other devices have no kernel image
        g_init_error = "mvsv_init: this library is built for sm_100a (B200, compute capability 10.0) only; device reports " +
                       std::to_string(prop.major) + "." + std::to_string(prop.minor);
        destroy_engine(c);
        return MVSV_ERR_UNSUPPORTED;
    }
    if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
    if ((e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
    if ((e = cudaStreamCreateWithFlags(&c->dl_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
    if ((e = cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
    for (cudaEvent_t& ev : c->ev_chunk)
        if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return bail(e, "cudaEventCreate");
    if ((e = cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming)) != cudaSuccess) return bail(e, "cudaEventCreate");
    for (auto& sl : c->slot)
        if ((e = cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming)) != cudaSuccess) return bail(e, "cudaEventCreate");
    for (cudaEvent_t* ev : {&c->ev_h2d, &c->ev_done})
        if ((e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming)) != cudaSuccess) return bail(e, "cudaEventCreate");
    Geometry g;
    int rc = plan_geometry(c, false, 0, 0, 0.0, &g);
    if (!rc) rc = apply_geometry(c, g);
    if (rc) { g_init_error = c->err; destroy_engine(c); return rc; }
    *out = c;
    return MVSV_OK;
}

// a ctx of one part per listed device, each of ceil(max_batch / n) frames
static int init(const int* devices, int n, int frame_width, int frame_height, int max_batch, mvsv_ctx** out)
{
    mvsv_ctx* c = new (std::nothrow) mvsv_ctx();
    if (!c) return MVSV_ERR_NOMEM;
    const int cap = (max_batch + n - 1) / n;
    for (int k = 0; k < n; ++k) {
        Engine* p = nullptr;
        const int rc = init_engine(devices[k], frame_width, frame_height, cap, &p);
        if (rc) {
            mvsv_destroy(c);
            if (n > 1)
                g_init_error = "mvsv_init_devices: part " + std::to_string(k) + " (device " + std::to_string(devices[k]) + "): " +
                               g_init_error;
            return rc;
        }
        c->parts.push_back(p);
        c->device.push_back(devices[k]);
    }
    c->maxB = cap * n;
    *out = c;
    return MVSV_OK;
}

int mvsv_init(int device, int frame_width, int frame_height, int max_batch, mvsv_ctx** out)
{
    if (!out) return MVSV_ERR_INVALID;
    *out = nullptr;
    return init(&device, 1, frame_width, frame_height, max_batch, out);
}

int mvsv_init_devices(const int* devices, int n, int frame_width, int frame_height, int max_batch, mvsv_ctx** out)
{
    if (!out) return MVSV_ERR_INVALID;
    *out = nullptr;
    if (!devices || n < 1 || n > max_batch) {
        g_init_error = "mvsv_init_devices: the device list must name between 1 and max_batch devices";
        return MVSV_ERR_INVALID;
    }
    return init(devices, n, frame_width, frame_height, max_batch, out);
}

void mvsv_destroy(mvsv_ctx* c)
{
    if (!c) return;
    for (Engine* p : c->parts) destroy_engine(p);
    delete c;
}

int mvsv_get_devices(const mvsv_ctx* c, int* devices, int n)
{
    if (!c || n < 0 || (n > 0 && !devices)) return MVSV_ERR_INVALID;
    std::copy(c->device.begin(), c->device.begin() + std::min(n, (int)c->device.size()), devices);
    return (int)c->device.size();
}

const char* mvsv_last_error(const mvsv_ctx* c) { return c ? c->err.c_str() : g_init_error.c_str(); }

int mvsv_set_sgbm_params(mvsv_ctx* ctx, const mvsv_sgbm_params* p)
{
    return each(ctx, true, [&](Engine* c) -> int {
        if (!p) return MVSV_ERR_INVALID;
        int rc = bind(c);
        if (rc) return rc;
        SgbmNorm n;
        rc = normalise_sgbm(c, p, c->W, c->H, &n);
        if (rc) return rc;
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        c->sg = n; c->sgbm_raw = *p; c->has_sgbm = true;
        c->td_nc = sgbm_choose_td_cluster(c);
        return ensure_sgbm_volumes(c);
    });
}

int mvsv_set_bm_params(mvsv_ctx* ctx, const mvsv_bm_params* p)
{
    return each(ctx, true, [&](Engine* c) -> int {
        if (!p) return MVSV_ERR_INVALID;
        int rc = bind(c);
        if (rc) return rc;
        BmNorm n;
        rc = normalise_bm(c, p, c->W, &n);
        if (rc) return rc;
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        c->bm = n; c->bm_raw = *p; c->has_bm = true;
        return ensure_bm_volumes(c);
    });
}

int mvsv_set_bm_filters(mvsv_ctx* ctx, int disp12MaxDiff, int speckleWindowSize, int speckleRange)
{
    return each(ctx, true, [&](Engine* c) -> int {
        if (speckleWindowSize < 0) return fail(c, MVSV_ERR_INVALID, "BM speckleWindowSize must be >= 0");
        if (speckleWindowSize > 0 && speckleRange < 0) return fail(c, MVSV_ERR_INVALID, "BM speckleRange must be >= 0");
        if (disp12MaxDiff >= 0 && c->W > bm_lrcheck_max_width())
            return fail(c, MVSV_ERR_UNSUPPORTED, "BM left-right check (disp12MaxDiff >= 0): image wider than 4096");
        int rc = bind(c);
        if (rc) return rc;
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        c->bm_d12 = disp12MaxDiff < 0 ? -1 : disp12MaxDiff;
        c->bm_speckle_win = speckleWindowSize;
        c->bm_speckle_range = speckleWindowSize > 0 ? speckleRange : 0;
        return MVSV_OK;
    });
}

// shared by the two ways of installing a camera's maps: checks the display ROI, sizes the rectified images and
// the raw-frame staging, allocates the fixed-point map
static int prepare_maps(Engine* c, int rig, int cam, int roi_x, int roi_y, int roi_w, int roi_h)
{
    if (roi_x < 0 || roi_y < 0 || roi_w < 2 || roi_h < 1 || roi_x + roi_w > c->fw || roi_y + roi_h > c->fh)
        return fail(c, MVSV_ERR_INVALID, "display ROI outside the frame");
    const int other = 1 - cam;
    if (c->has_maps[rig][other] &&
        (c->roi_xy[rig][0] != roi_x || c->roi_xy[rig][1] != roi_y || c->roi_w != roi_w || c->roi_h != roi_h))
        return fail(c, MVSV_ERR_INVALID, "both cameras must share one display ROI (mDisplayROI)");
    for (int r = 0; r < MVSV_MAX_RIGS; ++r)
        if (r != rig && (c->has_maps[r][0] || c->has_maps[r][1]) && (c->roi_w != roi_w || c->roi_h != roi_h))
            return fail(c, MVSV_ERR_INVALID, "all rigs share the display-ROI size (rig " + std::to_string(r) + " holds maps of another size)");
    Geometry g;
    int rc = plan_geometry(c, true, roi_w, roi_h, c->resize_factor, &g);
    if (rc) return rc;
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    c->roi_xy[rig][0] = roi_x; c->roi_xy[rig][1] = roi_y; c->roi_w = roi_w; c->roi_h = roi_h;
    c->has_maps[rig][cam] = false;
    c->rig_tables_dirty = true;
    MVSV_CK(c, c->map_xy[rig][cam].alloc((size_t)roi_w * roi_h));
    rc = apply_geometry(c, g);
    if (rc) return rc;
    return ensure_slots(c);
}

int mvsv_upload_rectify_maps(mvsv_ctx* c, int cam, const float* mapx, const float* mapy, size_t stride_bytes, int roi_x,
                             int roi_y, int roi_w, int roi_h)
{
    return mvsv_upload_rectify_maps_rig(c, 0, cam, mapx, mapy, stride_bytes, roi_x, roi_y, roi_w, roi_h);
}

int mvsv_upload_rectify_maps_rig(mvsv_ctx* ctx, int rig, int cam, const float* mapx, const float* mapy, size_t stride_bytes,
                                 int roi_x, int roi_y, int roi_w, int roi_h)
{
    return each(ctx, true, [&](Engine* c) -> int {
        if (!mapx || !mapy || cam < 0 || cam > 1) return MVSV_ERR_INVALID;
        if (rig < 0 || rig >= MVSV_MAX_RIGS) return fail(c, MVSV_ERR_INVALID, "rig outside [0, MVSV_MAX_RIGS)");
        int rc = bind(c);
        if (rc) return rc;
        if (stride_bytes < (size_t)c->fw * sizeof(float) || stride_bytes % sizeof(float)) return fail(c, MVSV_ERR_INVALID, "bad map stride");
        rc = prepare_maps(c, rig, cam, roi_x, roi_y, roi_w, roi_h);
        if (rc) return rc;
        // the float maps, staged on the device for the conversion
        DeviceBuffer<float> dx, dy;
        MVSV_CK(c, dx.alloc((size_t)c->fw * c->fh));
        MVSV_CK(c, dy.alloc((size_t)c->fw * c->fh));
        const size_t w = (size_t)c->fw * sizeof(float);
        MVSV_CK(c, cudaMemcpy2DAsync(dx, w, mapx, stride_bytes, w, c->fh, cudaMemcpyHostToDevice, c->stream));
        MVSV_CK(c, cudaMemcpy2DAsync(dy, w, mapy, stride_bytes, w, c->fh, cudaMemcpyHostToDevice, c->stream));
        MVSV_CK(c, launch_convert_maps(c, rig, cam, dx, dy, (size_t)c->fw));
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        c->has_maps[rig][cam] = true;
        return MVSV_OK;
    });
}

int mvsv_set_rectification(mvsv_ctx* c, int cam, const double K[9], const double* dist, int n_dist, const double R[9],
                           const double P[12], int roi_x, int roi_y, int roi_w, int roi_h)
{
    return mvsv_set_rectification_rig(c, 0, cam, K, dist, n_dist, R, P, roi_x, roi_y, roi_w, roi_h);
}

int mvsv_set_rectification_rig(mvsv_ctx* ctx, int rig, int cam, const double K[9], const double* dist, int n_dist,
                               const double R[9], const double P[12], int roi_x, int roi_y, int roi_w, int roi_h)
{
    return each(ctx, true, [&](Engine* c) -> int {
        if (!K || !R || !P || cam < 0 || cam > 1 || n_dist < 0 || (n_dist > 0 && !dist)) return MVSV_ERR_INVALID;
        if (rig < 0 || rig >= MVSV_MAX_RIGS) return fail(c, MVSV_ERR_INVALID, "rig outside [0, MVSV_MAX_RIGS)");
        int rc = bind(c);
        if (rc) return rc;
        if (n_dist != 0 && n_dist != 4 && n_dist != 5)
            return fail(c, MVSV_ERR_UNSUPPORTED, "distortion model: 0, 4 or 5 coefficients (k1 k2 p1 p2 [k3])");
        // iR = (P[:, :3] * R)^-1, the 3x3 closed form (cofactors / determinant)
        double A[9];
        for (int r = 0; r < 3; ++r)
            for (int k = 0; k < 3; ++k) {
                double acc = 0;
                for (int m = 0; m < 3; ++m) acc += P[r * 4 + m] * R[m * 3 + k];
                A[r * 3 + k] = acc;
            }
        const double c00 = A[4] * A[8] - A[5] * A[7], c01 = A[3] * A[8] - A[5] * A[6], c02 = A[3] * A[7] - A[4] * A[6];
        const double det = A[0] * c00 - A[1] * c01 + A[2] * c02;
        if (!(det != 0.0) || !std::isfinite(det)) return fail(c, MVSV_ERR_INVALID, "P[:, :3]*R is singular");
        const double d = 1.0 / det;
        RectifyCoef q;
        q.iR[0] = c00 * d;                         q.iR[1] = (A[2] * A[7] - A[1] * A[8]) * d;  q.iR[2] = (A[1] * A[5] - A[2] * A[4]) * d;
        q.iR[3] = (A[5] * A[6] - A[3] * A[8]) * d;  q.iR[4] = (A[0] * A[8] - A[2] * A[6]) * d;  q.iR[5] = (A[2] * A[3] - A[0] * A[5]) * d;
        q.iR[6] = c02 * d;                         q.iR[7] = (A[1] * A[6] - A[0] * A[7]) * d;  q.iR[8] = (A[0] * A[4] - A[1] * A[3]) * d;
        q.k1 = n_dist > 0 ? dist[0] : 0; q.k2 = n_dist > 1 ? dist[1] : 0; q.p1 = n_dist > 2 ? dist[2] : 0;
        q.p2 = n_dist > 3 ? dist[3] : 0; q.k3 = n_dist > 4 ? dist[4] : 0;
        q.fx = K[0]; q.fy = K[4]; q.cx = K[2]; q.cy = K[5];
        rc = prepare_maps(c, rig, cam, roi_x, roi_y, roi_w, roi_h);
        if (rc) return rc;
        MVSV_CK(c, launch_rectify_maps(c, rig, cam, q));
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        c->has_maps[rig][cam] = true;
        return MVSV_OK;
    });
}

int mvsv_reset_rectification(mvsv_ctx* ctx)
{
    return each(ctx, true, [&](Engine* c) -> int {
        int rc = bind(c);
        if (rc) return rc;
        Geometry g;
        rc = plan_geometry(c, false, 0, 0, c->resize_factor, &g);
        if (rc) return rc;
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        for (int r = 0; r < MVSV_MAX_RIGS; ++r)
            for (int i = 0; i < 2; ++i) {
                c->has_maps[r][i] = false;
                c->map_xy[r][i].reset();
            }
        c->rig_tables_dirty = true;
        return apply_geometry(c, g);
    });
}

int mvsv_set_resize(mvsv_ctx* ctx, double factor)
{
    return each(ctx, true, [&](Engine* c) -> int {
        int rc = bind(c);
        if (rc) return rc;
        if (!(factor == factor) || factor > 8.0) return fail(c, MVSV_ERR_INVALID, "resize factor must be in (0, 8]");
        const double f = (factor <= 0.0 || factor == 1.0) ? 0.0 : factor;   // off: cv::resize by 1 is the identity
        if (f > 0.0 && f < 1.0 / 64) return fail(c, MVSV_ERR_INVALID, "resize factor must be in (0, 8]");
        Geometry g;
        rc = plan_geometry(c, any_maps(c), c->roi_w, c->roi_h, f, &g);
        if (rc) return rc;
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        c->resize_factor = f;
        return apply_geometry(c, g);
    });
}

int mvsv_tm(mvsv_ctx* ctx, const uint8_t* left, size_t lstride, const uint8_t* right, size_t rstride, size_t frame_stride,
            int batch, unsigned kernel_size, uint8_t* out, size_t ostride)
{
    return single(ctx, "mvsv_tm", [&](Engine* c) -> int {
        if (!left || !right || !out) return MVSV_ERR_INVALID;
        int rc = bind(c);
        if (rc) return rc;
        const int W = c->W, H = c->H;
        if (batch < 1 || batch > c->maxB) return fail(c, MVSV_ERR_INVALID, "bad batch size");
        if (lstride < (size_t)W || rstride < (size_t)W || ostride < (size_t)W) return fail(c, MVSV_ERR_INVALID, "stride smaller than image width");
        if (kernel_size < 1 || kernel_size > 31) return fail(c, MVSV_ERR_UNSUPPORTED, "tm: kernelSize must be in [1, 31]");
        if (W > tm_max_width()) return fail(c, MVSV_ERR_UNSUPPORTED, "tm: image wider than 4096");
        if (tm_smem_bytes(W, (int)kernel_size) > 200 * 1024) return fail(c, MVSV_ERR_UNSUPPORTED, "tm: kernelSize x width exceeds shared memory");
        MVSV_CK(c, cudaStreamWaitEvent(c->copy_stream, c->ev_done, 0));
        rc = upload_images(c, io(c).rect[0], c->pitch, left, lstride, frame_stride, W, H, batch, false);
        if (rc) return rc;
        rc = upload_images(c, io(c).rect[1], c->pitch, right, rstride, frame_stride, W, H, batch, false);
        if (rc) return rc;
        rc = inputs_uploaded(c, false);
        if (rc) return rc;
        MVSV_CK(c, c->tm_out.ensure((size_t)c->maxB * H * c->pitch));
        MVSV_CK(c, cudaMemsetAsync(c->tm_out, 0, (size_t)batch * H * c->pitch, c->stream));   // cv::Scalar::all(0)
        // the reference's loops are `i < rows - kernelSize` in unsigned arithmetic: nothing to do unless k < rows, cols
        if ((int)kernel_size < H && (int)kernel_size < W) MVSV_CK(c, launch_tm(c, batch, (int)kernel_size, c->tm_out, c->pitch));
        MVSV_CK(c, cudaMemcpy2DAsync(out, ostride, c->tm_out, c->pitch, (size_t)W, (size_t)H * batch, cudaMemcpyDeviceToHost, c->stream));
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        return MVSV_OK;
    });
}

int mvsv_set_Q(mvsv_ctx* c, const float q[16]) { return mvsv_set_Q_rig(c, 0, q); }

int mvsv_set_Q_rig(mvsv_ctx* ctx, int rig, const float q[16])
{
    return each(ctx, true, [&](Engine* c) -> int {
        if (!q) return MVSV_ERR_INVALID;
        if (rig < 0 || rig >= MVSV_MAX_RIGS) return fail(c, MVSV_ERR_INVALID, "rig outside [0, MVSV_MAX_RIGS)");
        std::memcpy(c->Q[rig], q, sizeof(float) * 16);
        c->has_Q[rig] = true;
        c->rig_tables_dirty = true;
        return MVSV_OK;
    });
}

int mvsv_set_frame_rigs(mvsv_ctx* c, const int* rig_of_frame, int n)
{
    int rc = usable(c);
    if (rc) return rc;
    if (n < 0 || (n > 0 && !rig_of_frame)) return MVSV_ERR_INVALID;
    if (n > c->maxB) return fail(c, MVSV_ERR_INVALID, "more frames than max_batch");
    for (int i = 0; i < n; ++i)
        if (rig_of_frame[i] < 0 || rig_of_frame[i] >= MVSV_MAX_RIGS)
            return fail(c, MVSV_ERR_INVALID, "rig of frame " + std::to_string(i) + " outside [0, MVSV_MAX_RIGS)");
    std::vector<int> table(rig_of_frame, rig_of_frame + n);
    // A single part's slice is the whole table, which no batch size changes: it goes now, so that a compute never waits
    // for it.  Several parts receive theirs when a compute needs them (send_rigs).
    if (c->parts.size() == 1) {
        rc = on_part(c, 0, [&](Engine* p) { return set_rigs(p, table); });
        if (rc) return rc;
    }
    c->frame_rig.swap(table);
    return MVSV_OK;
}

int mvsv_set_mean_rois(mvsv_ctx* ctx, const int* xywh, int n)
{
    return each(ctx, true, [&](Engine* c) -> int {
        if (n < 0 || (n > 0 && !xywh)) return MVSV_ERR_INVALID;
        int rc = bind(c);
        if (rc) return rc;
        for (int i = 0; i < n; ++i) {
            const int* r = xywh + 4 * i;
            if (r[0] < 0 || r[1] < 0 || r[2] < 1 || r[3] < 1 || r[0] + r[2] > c->W || r[1] + r[3] > c->H)
                return fail(c, MVSV_ERR_INVALID, "ROI outside the disparity map");
        }
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        c->rois.reset();
        for (IoSlot& s : c->slot) {
            s.means.reset();
            s.stages &= ~(unsigned)MVSV_STAGE_MEANS;
        }
        c->nrois = n;
        if (n == 0) return MVSV_OK;
        MVSV_CK(c, c->rois.alloc((size_t)n * 4));
        rc = ensure_slots(c);
        if (rc) return rc;
        MVSV_CK(c, cudaMemcpy(c->rois, xywh, (size_t)n * 4 * sizeof(int), cudaMemcpyHostToDevice));
        return MVSV_OK;
    });
}

int mvsv_compute(mvsv_ctx* c, const uint8_t* left, size_t lstride, const uint8_t* right, size_t rstride, size_t frame_stride,
                 int batch, unsigned stages)
{
    return run(c, left, lstride, right, rstride, frame_stride, batch, stages, false);
}

int mvsv_compute_device(mvsv_ctx* c, const uint8_t* dleft, size_t lstride, const uint8_t* dright, size_t rstride,
                        size_t frame_stride, int batch, unsigned stages)
{
    return run(c, dleft, lstride, dright, rstride, frame_stride, batch, stages, true);
}

int mvsv_download(mvsv_ctx* c, int16_t* disp, size_t dstride, uint8_t* rectL, uint8_t* rectR, size_t rstride, float* xyz,
                  float* means)
{
    return mvsv_download_age(c, 0, disp, dstride, rectL, rectR, rstride, xyz, means);
}

int mvsv_download_age(mvsv_ctx* c, int age, int16_t* disp, size_t dstride, uint8_t* rectL, uint8_t* rectR, size_t rstride,
                      float* xyz, float* means)
{
    int rc = usable(c);
    if (rc) return rc;
    const Engine* p0 = c->parts[0];
    if (age < 0 || age >= p0->nslots) return fail(c, MVSV_ERR_INVALID, "age must be below the number of I/O slots");
    const int s = (p0->cur + p0->nslots - age) % p0->nslots, n = (int)c->parts.size();
    const std::vector<int> first = firsts(c, s);
    if (first[n] < 1) return fail(c, MVSV_ERR_STATE, "nothing computed yet");
    // every part's copies are queued before the first wait, so that the parts' downloads run side by side
    int queued = 0;
    for (; queued < n && !rc; ++queued)
        if (first[queued] < first[queued + 1])
            rc = on_part(c, queued, [&](Engine* p) {
                const size_t rows = (size_t)first[queued] * p->H;
                return download_enqueue(p, s, disp ? (int16_t*)((uint8_t*)disp + rows * dstride) : nullptr, dstride,
                                        rectL ? rectL + rows * rstride : nullptr, rectR ? rectR + rows * rstride : nullptr,
                                        rstride, xyz ? xyz + rows * p->W * 3 : nullptr,
                                        means ? means + (size_t)first[queued] * p->nrois : nullptr);
            });
    // wait also after a failure: the caller's buffers must not be written once the call has returned
    for (int k = 0; k < queued; ++k)
        if (first[k] < first[k + 1]) {
            if (rc) cudaStreamSynchronize(c->parts[k]->dl_stream);
            else rc = on_part(c, k, download_wait);
        }
    return rc;
}

int mvsv_download_points(mvsv_ctx* c, int age, int64_t* offsets, float* points, size_t capacity_points)
{
    int rc = usable(c);
    if (rc) return rc;
    if (!offsets) return fail(c, MVSV_ERR_INVALID, "offsets must not be NULL");
    const Engine* p0 = c->parts[0];
    if (age < 0 || age >= p0->nslots) return fail(c, MVSV_ERR_INVALID, "age must be below the number of I/O slots");
    const int s = (p0->cur + p0->nslots - age) % p0->nslots, n = (int)c->parts.size();
    const std::vector<int> first = firsts(c, s);
    if (first[n] < 1) return fail(c, MVSV_ERR_STATE, "nothing computed yet");
    for (int k = 0; k < n; ++k)
        if (first[k] < first[k + 1] && (!c->parts[k]->slot[s].offsets || !(c->parts[k]->slot[s].stages & MVSV_STAGE_POINTS)))
            return fail(c, MVSV_ERR_STATE, "POINTS stage was not computed");
    // phase 1: every part's frame offsets; part k's list goes after the points of the parts before it
    std::vector<std::vector<long long>> part(n);
    std::vector<long long> base(n + 1, 0);
    for (int k = 0; k < n; ++k) {
        if (first[k] < first[k + 1]) {
            rc = on_part(c, k, [&](Engine* p) { return points_offsets(p, s, part[k]); });
            if (rc) return rc;
        }
        base[k + 1] = base[k] + (part[k].empty() ? 0 : part[k].back());
    }
    for (int k = 0; k < n; ++k)
        for (int f = first[k]; f < first[k + 1]; ++f) offsets[f] = base[k] + part[k][f - first[k]];
    offsets[first[n]] = base[n];
    if (!points) return MVSV_OK;
    if (capacity_points < (size_t)base[n])
        return fail(c, MVSV_ERR_INVALID, "points buffer holds " + std::to_string(capacity_points) + " points, the list has " +
                                             std::to_string(base[n]));
    // phase 2: every part's copy is queued before the first wait, so that the parts' copies run side by side
    int queued = 0;
    for (; queued < n && !rc; ++queued)
        if (first[queued] < first[queued + 1])
            rc = on_part(c, queued, [&](Engine* p) { return points_enqueue(p, s, points + 3 * (size_t)base[queued], base[queued + 1] - base[queued]); });
    // wait also after a failure: the caller's buffer must not be written once the call has returned
    for (int k = 0; k < queued; ++k)
        if (first[k] < first[k + 1]) {
            if (rc) cudaStreamSynchronize(c->parts[k]->dl_stream);
            else rc = on_part(c, k, download_wait);
        }
    return rc;
}

int mvsv_set_io_slots(mvsv_ctx* ctx, int n)
{
    return each(ctx, true, [&](Engine* c) -> int {
        int rc = bind(c);
        if (rc) return rc;
        if (n != 1 && n != 2) return fail(c, MVSV_ERR_INVALID, "1 or 2 I/O slots");
        if (n == c->nslots) return MVSV_OK;
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        MVSV_CK(c, cudaStreamSynchronize(c->copy_stream));
        if (n < c->nslots) release_slot(c->slot[1], true);
        c->nslots = n;
        c->cur = 0;
        rc = ensure_slots(c);
        if (rc) { release_slot(c->slot[1], true); c->nslots = 1; }
        return rc;
    });
}

int mvsv_download_minmax(mvsv_ctx* c, int16_t* minmax)
{
    if (!c || !minmax) return MVSV_ERR_INVALID;
    int rc = usable(c);
    if (rc) return rc;
    const int n = (int)c->parts.size();
    const std::vector<int> first = firsts(c, c->parts[0]->cur);
    if (first[n] < 1) return fail(c, MVSV_ERR_STATE, "nothing computed yet");
    // the reductions of all parts are launched before the first result is read back
    for (int pass = 0; pass < 2 && !rc; ++pass)
        for (int k = 0; k < n && !rc; ++k)
            if (first[k] < first[k + 1])
                rc = on_part(c, k, [&](Engine* p) {
                    return pass == 0 ? minmax_launch(p) : minmax_read(p, minmax + 2 * (size_t)first[k]);
                });
    return rc;
}

int mvsv_sync(mvsv_ctx* ctx)
{
    return each(ctx, false, [&](Engine* c) -> int {
        int rc = bind(c);
        if (rc) return rc;
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        return MVSV_OK;
    });
}

int mvsv_get_info(const mvsv_ctx* ctx, mvsv_info* info)
{
    if (!ctx || !info) return MVSV_ERR_INVALID;
    const Engine* c = ctx->parts[0];
    std::memset(info, 0, sizeof(*info));
    info->frame_width = c->fw; info->frame_height = c->fh; info->width = c->W; info->height = c->H; info->max_batch = ctx->maxB;
    if (c->has_sgbm) {
        info->sgbm_minX1 = c->sg.minX1; info->sgbm_W1 = c->sg.W1; info->sgbm_D = c->sg.D; info->sgbm_Dpad = c->sg.Dp;
        info->sgbm_npaths = c->sg.npaths;
    }
    info->num_rois = c->nrois; info->device = c->device; info->sgbm_td_cluster = c->has_sgbm ? c->td_nc : 0;
    info->last_batch = firsts(ctx, c->cur).back();
    info->sgbm_s8 = c->last_s8 ? 1 : 0;
    info->bm_col8 = (c->has_bm && c->bm.col8 && !(c->debug_flags & 2u)) ? 1 : 0;
    return MVSV_OK;
}

void* mvsv_stream(mvsv_ctx* c) { return c && c->parts.size() == 1 ? (void*)c->parts[0]->stream : nullptr; }
unsigned long long mvsv_launch_count(const mvsv_ctx* c)
{
    unsigned long long n = 0;
    if (c)
        for (const Engine* p : c->parts) n += p->launches;
    return n;
}

int mvsv_host_alloc(void** p, size_t bytes)
{
    if (!p) return MVSV_ERR_INVALID;
    return cudaHostAlloc(p, bytes, cudaHostAllocDefault) == cudaSuccess ? MVSV_OK : MVSV_ERR_NOMEM;
}
int mvsv_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? MVSV_OK : MVSV_ERR_CUDA; }

int mvsv_timer_start(mvsv_ctx* ctx)
{
    return each(ctx, false, [&](Engine* c) -> int {
        int rc = bind(c);
        if (rc) return rc;
        if (!c->timer_a) { MVSV_CK(c, cudaEventCreate(&c->timer_a)); MVSV_CK(c, cudaEventCreate(&c->timer_b)); }
        MVSV_CK(c, cudaEventRecord(c->timer_a, c->stream));
        return MVSV_OK;
    });
}

// the longest part's interval
int mvsv_timer_stop(mvsv_ctx* ctx, float* ms)
{
    int rc = usable(ctx);
    if (rc) return rc;
    if (!ms) return MVSV_ERR_INVALID;
    float longest = 0.f;
    rc = each(ctx, false, [&](Engine* c) -> int {
        if (!c->timer_a) return MVSV_ERR_INVALID;
        const int bound = bind(c);
        if (bound) return bound;
        float t = 0.f;
        MVSV_CK(c, cudaEventRecord(c->timer_b, c->stream));
        MVSV_CK(c, cudaEventSynchronize(c->timer_b));
        MVSV_CK(c, cudaEventElapsedTime(&t, c->timer_a, c->timer_b));
        longest = std::max(longest, t);
        return MVSV_OK;
    });
    if (!rc) *ms = longest;
    return rc;
}

int mvsv_profile_enable(mvsv_ctx* ctx, int enable)
{
    return single(ctx, "mvsv_profile_enable", [&](Engine* c) -> int {
        c->prof = enable != 0;
        return MVSV_OK;
    });
}

int mvsv_profile_read(mvsv_ctx* ctx, float* ms, int* counts, int n)
{
    return single(ctx, "mvsv_profile_read", [&](Engine* c) -> int {
        if (!ms || !counts || n < KID_COUNT) return MVSV_ERR_INVALID;
        int rc = bind(c);
        if (rc) return rc;
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        for (int i = 0; i < n; ++i) { ms[i] = 0.f; counts[i] = 0; }
        for (auto& b : c->brackets) {
            float t = 0.f;
            if (cudaEventElapsedTime(&t, b.a, b.b) == cudaSuccess) { ms[b.kid] += t; counts[b.kid] += 1; }
            c->ev_free.push_back(b.a); c->ev_free.push_back(b.b);
        }
        c->brackets.clear();
        return KID_COUNT;
    });
}

const char* mvsv_kernel_name(int kid) { return (kid >= 0 && kid < KID_COUNT) ? kKernelNames[kid] : ""; }

int mvsv_debug_set_flags(mvsv_ctx* ctx, unsigned flags)
{
    return single(ctx, "mvsv_debug_set_flags", [&](Engine* c) -> int {
        c->debug_flags = flags;
        if (c->has_sgbm) c->td_nc = sgbm_choose_td_cluster(c);
        return MVSV_OK;
    });
}

int mvsv_debug_postfilter(mvsv_ctx* ctx, const int16_t* maps, size_t stride, int batch, int median, int newVal,
                          int maxSpeckleSize, int maxDiff, unsigned stages)
{
    return single(ctx, "mvsv_debug_postfilter", [&](Engine* c) -> int {
        int rc = bind(c);
        if (rc) return rc;
        if (!maps || batch < 1 || batch > c->maxB) return fail(c, MVSV_ERR_INVALID, "bad map pointer or batch size");
        if (stride < (size_t)c->W * sizeof(int16_t)) return fail(c, MVSV_ERR_INVALID, "stride smaller than the map width");
        if (stages & ~(unsigned)(MVSV_STAGE_XYZ | MVSV_STAGE_POINTS | MVSV_STAGE_MEANS))
            return fail(c, MVSV_ERR_INVALID, "post-filter hook: only MVSV_STAGE_XYZ, MVSV_STAGE_POINTS and MVSV_STAGE_MEANS");
        if (maxSpeckleSize > 0 && (newVal < -32768 || newVal > 32767)) return fail(c, MVSV_ERR_INVALID, "newVal does not fit CV_16S");
        const uint64_t rigs = rigs_of_batch(c, batch);
        const bool multi = rigs != 1;
        // the next I/O slot, taken as a compute takes it
        IoSlot& slot = next_slot(c);
        rc = check_consumers(c, slot, stages, rigs);
        if (!rc) rc = ensure_consumers(c, slot, stages);
        if (rc) return rc;

        take_slot(c);
        const size_t row = (size_t)c->W * sizeof(int16_t), npx = (size_t)batch * c->H * c->W;
        MVSV_CK(c, cudaMemcpy2DAsync(c->disp_raw, row, maps, stride, row, (size_t)c->H * batch, cudaMemcpyHostToDevice, c->stream));
        const bool speckle = maxSpeckleSize > 0;
        if (median) MVSV_CK(c, launch_median(c, c->disp_raw, speckle ? c->disp_med : slot.disp, batch));
        if (speckle)
            MVSV_CK(c, launch_speckle(c, median ? c->disp_med : c->disp_raw, slot.disp, batch, newVal, maxSpeckleSize, maxDiff));
        if (!median && !speckle)
            MVSV_CK(c, cudaMemcpyAsync(slot.disp, c->disp_raw, npx * sizeof(int16_t), cudaMemcpyDeviceToDevice, c->stream));
        if (multi && (stages & (MVSV_STAGE_XYZ | MVSV_STAGE_POINTS))) {
            rc = upload_rig_tables(c);
            if (rc) return rc;
        }
        if (stages & MVSV_STAGE_XYZ) MVSV_CK(c, multi ? launch_xyz_rigs(c, batch) : launch_xyz(c, batch));
        if (stages & MVSV_STAGE_POINTS) MVSV_CK(c, launch_points(c, batch, multi));
        if (stages & MVSV_STAGE_MEANS) MVSV_CK(c, launch_means(c, batch));
        MVSV_CK(c, cudaEventRecord(slot.done, c->stream));
        MVSV_CK(c, cudaEventRecord(c->ev_done, c->stream));
        slot.B = batch;
        slot.stages = stages;
        return MVSV_OK;
    });
}

long long mvsv_debug_read(mvsv_ctx* ctx, int which, void* host, size_t cap)
{
    return single(ctx, "mvsv_debug_read", [&](Engine* c) -> long long {
        if (!host) return MVSV_ERR_INVALID;
        int rc = bind(c);
        if (rc) return rc;
        const void* src = nullptr;
        size_t bytes = 0;
        if (which == 7 || which == 8) {
            const int cam = which - 7;
            if (!c->has_maps[0][cam]) return fail(c, MVSV_ERR_STATE, "no rectification map for this camera");
            src = c->map_xy[0][cam];
            bytes = (size_t)c->roi_w * c->roi_h * sizeof(int2);
            if (bytes > cap) return fail(c, MVSV_ERR_INVALID, "host buffer too small");
            MVSV_CK(c, cudaMemcpyAsync(host, src, bytes, cudaMemcpyDeviceToHost, c->stream));
            MVSV_CK(c, cudaStreamSynchronize(c->stream));
            return (long long)bytes;
        }
        const int B = io(c).B;
        if (B < 1) return fail(c, MVSV_ERR_STATE, "nothing computed yet");
        const size_t vol = c->has_sgbm && c->sg.W1 > 0 ? (size_t)B * c->H * c->sg.W1 * c->sg.Dp * 2 : 0;
        const size_t img16 = (size_t)B * c->H * c->W * 2;
        switch (which) {
            case 0: src = c->C; bytes = vol; break;
            case 1:
                // with S kept as bytes (S8) the complete 16-bit S only exists when the test hook asked the last scan to
                // store it (debug flag bit 0); it then lives in the VS volume, which is dead by that time
                if (c->last_s8 && !(c->debug_flags & 1)) return fail(c, MVSV_ERR_STATE, "S is held as bytes: set debug flag bit 0 before the compute");
                src = c->last_s8 ? c->VS : c->S; bytes = vol; break;
            case 2: src = c->disp_raw; bytes = img16; break;
            case 3:
                if (c->last_s8 && (c->debug_flags & 1)) return fail(c, MVSV_ERR_STATE, "the VS volume was reused for the final S (debug flag bit 0)");
                src = c->VS; bytes = vol; break;
            case 4: src = (c->has_sgbm && c->sg.speckleWin > 0) ? c->disp_med : io(c).disp; bytes = img16; break;
            case 5: src = c->bm_pre[0]; bytes = (size_t)B * c->H * c->pitch; break;
            case 6: src = c->bm_pre[1]; bytes = (size_t)B * c->H * c->pitch; break;
            default: return fail(c, MVSV_ERR_INVALID, "unknown debug buffer");
        }
        if (!src || bytes == 0) return fail(c, MVSV_ERR_STATE, "buffer not available");
        if (bytes > cap) return fail(c, MVSV_ERR_INVALID, "host buffer too small");
        MVSV_CK(c, cudaMemcpyAsync(host, src, bytes, cudaMemcpyDeviceToHost, c->stream));
        MVSV_CK(c, cudaStreamSynchronize(c->stream));
        return (long long)bytes;
    });
}

}  // extern "C"
