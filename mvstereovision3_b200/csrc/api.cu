// C-ABI glue of libmvsv.so (include/mvsv.h): context, device buffers, parameter normalisation, stage sequencing.
#include "mvsv_internal.h"
#include <cmath>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <new>

const char* const kKernelNames[KID_COUNT] = {
    "remap", "sgbm_prefilter", "sgbm_vsum", "sgbm_h1", "sgbm_vdir", "sgbm_td", "sgbm_h2_wta", "median3", "ccl_rows", "ccl_vmerge",
    "ccl_flatten", "ccl_apply", "bm_prefilter", "bm_tex", "bm_colsum", "bm_wta", "xyz", "means", "fill", "minmax", "tm",
    "bm_lrcheck"};

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

template <class T>
void dfree(T*& p)
{
    if (p) cudaFree(p);
    p = nullptr;
}

int fail(mvsv_ctx* c, int code, const std::string& msg)
{
    if (c) c->err = msg;
    return code;
}

// What free_slot releases; each level includes the ones before it.
enum SlotBuffers {
    SLOT_MEANS,     // the ROI means (the ROIs change)
    SLOT_SIZED,     // + rectified images, disparities, XYZ (the image size changes): the slot then holds no results
    SLOT_ALL        // + the raw-frame staging (the slot goes away)
};

void free_slot(mvsv_ctx* c, int k, SlotBuffers what)
{
    IoSlot& s = c->slot[k];
    dfree(s.means);
    s.stages &= ~(unsigned)MVSV_STAGE_MEANS;
    if (what == SLOT_MEANS) return;
    for (int i = 0; i < 2; ++i) dfree(s.rect[i]);
    dfree(s.disp); dfree(s.xyz);
    s.B = 0; s.stages = 0;
    if (what == SLOT_ALL)
        for (int i = 0; i < 2; ++i) dfree(s.raw[i]);
}

// Allocates what each live slot needs in the ctx's present state and does not have yet: the rectified images and the
// (zeroed) disparities always, the raw-frame staging once rectification maps are installed, the ROI means once ROIs
// are set.  The XYZ buffer is left to the first compute that asks for it.
int ensure_slots(mvsv_ctx* c)
{
    const size_t B = (size_t)c->maxB, npx = B * c->H * c->W, nimg = B * c->H * c->pitch;
    const bool maps = c->map_xy[0] || c->map_xy[1];
    for (int k = 0; k < c->nslots; ++k) {
        IoSlot& s = c->slot[k];
        for (int i = 0; i < 2; ++i) {
            if (!s.rect[i]) MVSV_CK(c, cudaMalloc(&s.rect[i], nimg));
            if (maps && !s.raw[i]) MVSV_CK(c, cudaMalloc(&s.raw[i], B * c->fh * c->raw_pitch));
        }
        if (!s.disp) {
            MVSV_CK(c, cudaMalloc(&s.disp, npx * sizeof(int16_t)));
            MVSV_CK(c, cudaMemsetAsync(s.disp, 0, npx * sizeof(int16_t), c->stream));
        }
        if (c->nrois > 0 && !s.means) MVSV_CK(c, cudaMalloc(&s.means, (size_t)c->nrois * B * sizeof(float)));
    }
    return MVSV_OK;
}

void free_images(mvsv_ctx* c)
{
    for (int k = 0; k < 2; ++k) free_slot(c, k, SLOT_SIZED);
    for (int i = 0; i < 2; ++i) dfree(c->bm_pre[i]);
    dfree(c->recL);
    dfree(c->d2); dfree(c->disp_raw); dfree(c->disp_med); dfree(c->labels); dfree(c->sizes);
    dfree(c->bm_tex2); dfree(c->minmax); dfree(c->tm_out);
}
void free_sgbm_volumes(mvsv_ctx* c)
{
    dfree(c->VS); dfree(c->C); dfree(c->S); dfree(c->plR); dfree(c->sweep_halo);
    c->vol_elems = 0;
}
void free_bm_volumes(mvsv_ctx* c) { dfree(c->bm_col); c->bm_vol_elems = 0; }

int alloc_images(mvsv_ctx* c)
{
    free_images(c);
    // 16-byte aligned rows; when the width already is (752, 1920, 3840, ...) a batch is one contiguous block and
    // host <-> device transfers are single linear copies instead of strided 2-D copies of many short rows
    c->pitch = round_up((size_t)c->W, 16);
    const size_t B = (size_t)c->maxB, npx = B * c->H * c->W, nimg = B * c->H * c->pitch;
    // the connected-components labels of the speckle filter are int indices over the whole batch
    if (nimg >= ((size_t)1 << 31)) return fail(c, MVSV_ERR_UNSUPPORTED, "max_batch * height * width must stay below 2^31 pixels");
    // the slot buffers first: allocated after the scratch buffers below, the StereoBM configuration ran 0.4 % slower
    // (49.35 K against 49.55 K frames/s on a B200 at 1000 W)
    const int rc = ensure_slots(c);
    if (rc) return rc;
    for (int i = 0; i < 2; ++i) MVSV_CK(c, cudaMalloc(&c->bm_pre[i], nimg + 64));   // the BM column-sum kernel reads whole aligned words
    MVSV_CK(c, cudaMalloc(&c->recL, npx * sizeof(uint2)));
    MVSV_CK(c, cudaMalloc(&c->d2, npx * sizeof(int)));
    MVSV_CK(c, cudaMalloc(&c->disp_raw, npx * sizeof(int16_t)));
    MVSV_CK(c, cudaMalloc(&c->disp_med, npx * sizeof(int16_t)));
    MVSV_CK(c, cudaMalloc(&c->labels, npx * sizeof(int)));
    MVSV_CK(c, cudaMalloc(&c->sizes, npx * sizeof(int)));
    MVSV_CK(c, cudaMalloc(&c->bm_tex2, npx * sizeof(int)));
    return MVSV_OK;
}

int normalise_sgbm(mvsv_ctx* c, const mvsv_sgbm_params* p, SgbmNorm* n)
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
    n->maxX1 = c->W + std::min(n->minD, 0);
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
    if (n->W1 > 0 && (long long)c->H * n->W1 * n->Dp >= (1ll << 31))
        return fail(c, MVSV_ERR_UNSUPPORTED, "cost volume of one frame exceeds 2^31 cells");
    return MVSV_OK;
}

int ensure_sgbm_volumes(mvsv_ctx* c)
{
    const SgbmNorm& n = c->sg;
    if (n.W1 <= 0) return MVSV_OK;
    int nv, rp, joff;
    sgbm_plane_geometry(n, c->W, &nv, &rp, &joff);
    const size_t need = (size_t)c->maxB * c->H * n.W1 * n.Dp;
    if (!(need <= c->vol_elems && c->VS)) {
        dfree(c->VS); dfree(c->C); dfree(c->S);
        c->vol_elems = 0;
        MVSV_CK(c, cudaMalloc(&c->VS, need * 2));
        MVSV_CK(c, cudaMalloc(&c->C, need * 2));
        MVSV_CK(c, cudaMalloc(&c->S, need * 2));
        c->vol_elems = need;
    }
    if (!c->sweep_halo) MVSV_CK(c, cudaMalloc(&c->sweep_halo, sweep_scratch_bytes(c)));   // strip-border records of the fused sweep
    if (!c->plR || nv != c->vsNV || rp != c->vsRP || joff != c->vsJOFF) {
        dfree(c->plR);
        const size_t bytes = (size_t)6 * c->maxB * c->H * rp * sizeof(uint16_t);
        MVSV_CK(c, cudaMalloc(&c->plR, bytes));
        MVSV_CK(c, cudaMemsetAsync(c->plR, 0, bytes, c->stream));   // the padding around each row stays zero
        c->vsNV = nv; c->vsRP = rp; c->vsJOFF = joff;
    }
    return MVSV_OK;
}

int normalise_bm(mvsv_ctx* c, const mvsv_bm_params* p, BmNorm* n)
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
    n->lofs = n->D - 1; n->width1 = c->W - n->D + 1; n->FILT = -16;
    n->col8 = n->bs * 2 * n->cap <= 255;
    return MVSV_OK;
}

int ensure_bm_volumes(mvsv_ctx* c)
{
    const BmNorm& n = c->bm;
    if (n.width1 < 1) return MVSV_OK;
    const size_t need = (size_t)c->maxB * c->H * n.width1 * n.Dp;
    if (need <= c->bm_vol_elems && c->bm_col) return MVSV_OK;
    free_bm_volumes(c);
    MVSV_CK(c, cudaMalloc(&c->bm_col, need * 2));
    c->bm_vol_elems = need;
    return MVSV_OK;
}

int bind(mvsv_ctx* c)
{
    MVSV_CK(c, cudaSetDevice(c->device));
    return MVSV_OK;
}

// host -> device copy of `batch` images (w bytes wide, h rows) into dst[b][h][dpitch]
int upload_images(mvsv_ctx* c, uint8_t* dst, size_t dpitch, const uint8_t* src, size_t sstride, size_t frame_stride, int w,
                  int h, int batch, bool device_src)
{
    const cudaMemcpyKind kind = device_src ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
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

static int inputs_uploaded(mvsv_ctx* c, bool device_src)
{
    if (device_src) return MVSV_OK;
    MVSV_CK(c, cudaEventRecord(c->ev_h2d, c->copy_stream));
    MVSV_CK(c, cudaStreamWaitEvent(c->stream, c->ev_h2d, 0));
    return MVSV_OK;
}

// what the XYZ and MEANS stages need of the ctx and of the slot they write to
int check_consumers(mvsv_ctx* c, const IoSlot& slot, unsigned stages)
{
    if ((stages & MVSV_STAGE_XYZ) && !c->has_Q) return fail(c, MVSV_ERR_STATE, "mvsv_set_Q not called");
    if ((stages & MVSV_STAGE_MEANS) && (c->nrois < 1 || !c->rois || !slot.means))
        return fail(c, MVSV_ERR_STATE, "no mean-disparity ROIs (mvsv_set_mean_rois; a geometry change drops them)");
    return MVSV_OK;
}

int run(mvsv_ctx* c, const uint8_t* left, size_t lstride, const uint8_t* right, size_t rstride, size_t frame_stride, int batch,
        unsigned stages, bool device_src)
{
    if (!c) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    // next I/O slot; its previous results must have been downloaded by now (mvsv_set_io_slots)
    const int k = (c->cur + 1) % c->nslots;
    IoSlot& slot = c->slot[k];
    const bool rectify = stages & MVSV_STAGE_RECTIFY;
    if (!left || !right || batch < 1 || batch > c->maxB) return fail(c, MVSV_ERR_INVALID, "bad image pointers or batch size");
    if ((stages & MVSV_STAGE_SGBM) && (stages & MVSV_STAGE_BM)) return fail(c, MVSV_ERR_INVALID, "choose SGBM or BM, not both");
    if ((stages & MVSV_STAGE_SGBM) && !c->has_sgbm) return fail(c, MVSV_ERR_STATE, "mvsv_set_sgbm_params not called");
    if ((stages & MVSV_STAGE_BM) && !c->has_bm) return fail(c, MVSV_ERR_STATE, "mvsv_set_bm_params not called");
    rc = check_consumers(c, slot, stages);
    if (rc) return rc;
    if (rectify && (!c->has_maps[0] || !c->has_maps[1]))
        return fail(c, MVSV_ERR_STATE, "rectify maps missing (mvsv_upload_rectify_maps)");
    if ((stages & MVSV_STAGE_BM) && c->bm_d12 >= 0 && c->W > bm_lrcheck_max_width())
        return fail(c, MVSV_ERR_UNSUPPORTED, "BM left-right check (disp12MaxDiff >= 0): image wider than 4096");
    const int iw = rectify ? c->fw : c->W, ih = rectify ? c->fh : c->H;
    if (lstride < (size_t)iw || rstride < (size_t)iw)
        return fail(c, MVSV_ERR_INVALID, rectify ? "stride smaller than frame width" : "stride smaller than image width");
    if (stages & MVSV_STAGE_SGBM) rc = ensure_sgbm_volumes(c);
    else if (stages & MVSV_STAGE_BM) rc = ensure_bm_volumes(c);
    if (rc) return rc;
    if ((stages & MVSV_STAGE_XYZ) && !slot.xyz) MVSV_CK(c, cudaMalloc(&slot.xyz, (size_t)c->maxB * c->H * c->W * 3 * sizeof(float)));

    // From here on the slot is taken: if a step fails it is left empty, so that a download reports the failure instead
    // of returning the frames of an older compute.
    c->cur = k;
    auto submit = [&]() -> int {
        // host inputs: the copies wait for the slot's previous compute (which may still read the input buffers), the
        // kernels wait for the copies
        if (!device_src) MVSV_CK(c, cudaStreamWaitEvent(c->copy_stream, slot.done, 0));
        uint8_t* const* dst = rectify ? slot.raw : slot.rect;
        const size_t dpitch = rectify ? c->raw_pitch : c->pitch;
        int r = upload_images(c, dst[0], dpitch, left, lstride, frame_stride, iw, ih, batch, device_src);
        if (!r) r = upload_images(c, dst[1], dpitch, right, rstride, frame_stride, iw, ih, batch, device_src);
        if (!r) r = inputs_uploaded(c, device_src);
        if (r) return r;
        if (rectify)
            for (int cam = 0; cam < 2; ++cam) {
                MVSV_CK(c, launch_remap(c, cam, batch));
                if (c->resize_factor > 0.0) MVSV_CK(c, launch_resize(c, cam, batch));
            }
        if (stages & MVSV_STAGE_SGBM) MVSV_CK(c, launch_sgbm(c, batch));
        else if (stages & MVSV_STAGE_BM) MVSV_CK(c, launch_bm(c, batch));
        if (stages & MVSV_STAGE_XYZ) MVSV_CK(c, launch_xyz(c, batch));
        if (stages & MVSV_STAGE_MEANS) MVSV_CK(c, launch_means(c, batch));
        MVSV_CK(c, cudaEventRecord(slot.done, c->stream));
        MVSV_CK(c, cudaEventRecord(c->ev_done, c->stream));
        return MVSV_OK;
    };
    rc = submit();
    slot.B = rc ? 0 : batch;
    slot.stages = rc ? 0 : stages;
    return rc;
}

// Copies the results a compute left in I/O slot `k` to the host on the download stream (so that it overlaps kernels
// submitted later) and waits for them.
int download_slot(mvsv_ctx* c, int k, int16_t* disp, size_t dstride, uint8_t* rectL, uint8_t* rectR, size_t rstride, float* xyz,
                  float* means)
{
    IoSlot& s = c->slot[k];
    const int B = s.B;
    if (B < 1) return fail(c, MVSV_ERR_STATE, "nothing computed yet");
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
    MVSV_CK(c, cudaStreamSynchronize(st));
    return MVSV_OK;
}

}  // namespace

extern "C" {

int mvsv_init(int device, int frame_width, int frame_height, int max_batch, mvsv_ctx** out)
{
    if (!out) return MVSV_ERR_INVALID;
    *out = nullptr;
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
    mvsv_ctx* c = new (std::nothrow) mvsv_ctx();
    if (!c) return MVSV_ERR_NOMEM;
    c->device = device; c->fw = frame_width; c->fh = frame_height; c->W = frame_width; c->H = frame_height; c->maxB = max_batch;
    c->raw_pitch = round_up((size_t)frame_width, 16);
    auto bail = [&](cudaError_t ee, const char* what) {
        g_init_error = std::string("mvsv_init: ") + what + ": " + cudaGetErrorString(ee);
        mvsv_destroy(c);
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
        mvsv_destroy(c);
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
    int rc = alloc_images(c);
    if (rc) { g_init_error = c->err; mvsv_destroy(c); return rc; }
    *out = c;
    return MVSV_OK;
}

void mvsv_destroy(mvsv_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->dl_stream) cudaStreamSynchronize(c->dl_stream);
    if (c->stream) cudaStreamSynchronize(c->stream);
    free_images(c);
    for (int k = 0; k < 2; ++k) {
        free_slot(c, k, SLOT_ALL);
        if (c->slot[k].done) cudaEventDestroy(c->slot[k].done);
    }
    free_sgbm_volumes(c);
    free_bm_volumes(c);
    for (int i = 0; i < 2; ++i) { dfree(c->map_xy[i]); dfree(c->crop[i]); }
    dfree(c->rois);
    for (auto& b : c->brackets) { cudaEventDestroy(b.a); cudaEventDestroy(b.b); }
    for (auto e : c->ev_free) cudaEventDestroy(e);
    if (c->timer_a) cudaEventDestroy(c->timer_a);
    if (c->timer_b) cudaEventDestroy(c->timer_b);
    for (cudaEvent_t ev : {c->ev_h2d, c->ev_done})
        if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : c->ev_chunk)
        if (ev) cudaEventDestroy(ev);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->dl_stream) cudaStreamDestroy(c->dl_stream);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

const char* mvsv_last_error(const mvsv_ctx* c) { return c ? c->err.c_str() : g_init_error.c_str(); }

int mvsv_set_sgbm_params(mvsv_ctx* c, const mvsv_sgbm_params* p)
{
    if (!c || !p) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    SgbmNorm n;
    rc = normalise_sgbm(c, p, &n);
    if (rc) return rc;
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    c->sg = n; c->sgbm_raw = *p; c->has_sgbm = true;
    c->td_nc = sgbm_choose_td_cluster(c);
    return ensure_sgbm_volumes(c);
}

int mvsv_set_bm_params(mvsv_ctx* c, const mvsv_bm_params* p)
{
    if (!c || !p) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    BmNorm n;
    rc = normalise_bm(c, p, &n);
    if (rc) return rc;
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    c->bm = n; c->bm_raw = *p; c->has_bm = true;
    return ensure_bm_volumes(c);
}

int mvsv_set_bm_filters(mvsv_ctx* c, int disp12MaxDiff, int speckleWindowSize, int speckleRange)
{
    if (!c) return MVSV_ERR_INVALID;
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
}

static int resize_rectified(mvsv_ctx* c, int W, int H)
{
    if (W == c->W && H == c->H) return MVSV_OK;
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    // the matcher parameters are re-normalised for the new geometry BEFORE anything is committed: a geometry the
    // contract rejects (e.g. a frame volume of 2^31 cells) leaves the engine exactly as it was
    const int oldW = c->W, oldH = c->H;
    SgbmNorm sg = c->sg;
    BmNorm bm = c->bm;
    c->W = W; c->H = H;
    int rc = MVSV_OK;
    if (c->has_sgbm) rc = normalise_sgbm(c, &c->sgbm_raw, &sg);
    if (!rc && c->has_bm) rc = normalise_bm(c, &c->bm_raw, &bm);
    if (rc) { c->W = oldW; c->H = oldH; return rc; }
    // mean-disparity ROIs are coordinates of the old map: drop them (run() asks for new ones)
    dfree(c->rois);
    c->nrois = 0;
    rc = alloc_images(c);
    if (rc) return rc;
    free_sgbm_volumes(c);
    free_bm_volumes(c);
    if (c->has_sgbm) {
        c->sg = sg;
        c->td_nc = sgbm_choose_td_cluster(c);
        rc = ensure_sgbm_volumes(c);
        if (rc) { c->has_sgbm = false; return rc; }
    }
    if (c->has_bm) {
        c->bm = bm;
        rc = ensure_bm_volumes(c);
        if (rc) { c->has_bm = false; return rc; }
    }
    return MVSV_OK;
}

// size of the images the matcher sees: the frame, the display ROI once maps are installed, the resized ROI when
// mvsv_set_resize is active; (re)allocates everything that depends on it
static int apply_geometry(mvsv_ctx* c)
{
    const bool maps = c->has_maps[0] || c->has_maps[1] || c->map_xy[0] || c->map_xy[1];
    int W = maps ? c->roi[2] : c->fw, H = maps ? c->roi[3] : c->fh;
    const bool resized = maps && c->resize_factor > 0.0;
    if (resized) {
        // cv::resize: dsize = Size(saturate_cast<int>(w*fx), saturate_cast<int>(h*fy)), round half to even
        W = (int)lrint((double)W * c->resize_factor);
        H = (int)lrint((double)H * c->resize_factor);
        if (W < 2 || H < 1 || W > 16384 || H > 16384) return fail(c, MVSV_ERR_INVALID, "resized image out of range");
    }
    int rc = resize_rectified(c, W, H);
    if (rc) return rc;
    for (int i = 0; i < 2; ++i) dfree(c->crop[i]);
    if (resized) {
        c->crop_pitch = round_up((size_t)c->roi[2], 16);
        for (int i = 0; i < 2; ++i) MVSV_CK(c, cudaMalloc(&c->crop[i], (size_t)c->maxB * c->roi[3] * c->crop_pitch));
    }
    return MVSV_OK;
}

// shared by the two ways of installing a camera's maps: checks the display ROI, sizes the rectified images and
// the raw-frame staging, allocates the fixed-point map
static int prepare_maps(mvsv_ctx* c, int cam, int roi_x, int roi_y, int roi_w, int roi_h)
{
    if (roi_x < 0 || roi_y < 0 || roi_w < 2 || roi_h < 1 || roi_x + roi_w > c->fw || roi_y + roi_h > c->fh)
        return fail(c, MVSV_ERR_INVALID, "display ROI outside the frame");
    const int other = 1 - cam;
    if (c->has_maps[other] && (c->roi[0] != roi_x || c->roi[1] != roi_y || c->roi[2] != roi_w || c->roi[3] != roi_h))
        return fail(c, MVSV_ERR_INVALID, "both cameras must share one display ROI (mDisplayROI)");
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    c->roi[0] = roi_x; c->roi[1] = roi_y; c->roi[2] = roi_w; c->roi[3] = roi_h;
    c->has_maps[cam] = false;
    dfree(c->map_xy[cam]);
    MVSV_CK(c, cudaMalloc(&c->map_xy[cam], (size_t)roi_w * roi_h * sizeof(int2)));
    int rc = apply_geometry(c);
    if (rc) return rc;
    return ensure_slots(c);
}

int mvsv_upload_rectify_maps(mvsv_ctx* c, int cam, const float* mapx, const float* mapy, size_t stride_bytes, int roi_x,
                             int roi_y, int roi_w, int roi_h)
{
    if (!c || !mapx || !mapy || cam < 0 || cam > 1) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    if (stride_bytes < (size_t)c->fw * sizeof(float) || stride_bytes % sizeof(float)) return fail(c, MVSV_ERR_INVALID, "bad map stride");
    rc = prepare_maps(c, cam, roi_x, roi_y, roi_w, roi_h);
    if (rc) return rc;
    float *dx = nullptr, *dy = nullptr;
    const size_t mbytes = (size_t)c->fw * c->fh * sizeof(float);
    MVSV_CK(c, cudaMalloc(&dx, mbytes));
    cudaError_t e = cudaMalloc(&dy, mbytes);
    if (e != cudaSuccess) { cudaFree(dx); c->err = "cudaMalloc(map)"; return MVSV_ERR_NOMEM; }
    const size_t w = (size_t)c->fw * sizeof(float);
    e = cudaMemcpy2DAsync(dx, w, mapx, stride_bytes, w, c->fh, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(dy, w, mapy, stride_bytes, w, c->fh, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = launch_convert_maps(c, cam, dx, dy, (size_t)c->fw);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(dx); cudaFree(dy);
    if (e != cudaSuccess) { c->err = std::string("map upload: ") + cudaGetErrorString(e); return MVSV_ERR_CUDA; }
    c->has_maps[cam] = true;
    return MVSV_OK;
}

int mvsv_set_rectification(mvsv_ctx* c, int cam, const double K[9], const double* dist, int n_dist, const double R[9],
                           const double P[12], int roi_x, int roi_y, int roi_w, int roi_h)
{
    if (!c || !K || !R || !P || cam < 0 || cam > 1 || n_dist < 0 || (n_dist > 0 && !dist)) return MVSV_ERR_INVALID;
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
    rc = prepare_maps(c, cam, roi_x, roi_y, roi_w, roi_h);
    if (rc) return rc;
    MVSV_CK(c, launch_rectify_maps(c, cam, q));
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    c->has_maps[cam] = true;
    return MVSV_OK;
}

int mvsv_reset_rectification(mvsv_ctx* c)
{
    if (!c) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    c->has_maps[0] = c->has_maps[1] = false;
    for (int i = 0; i < 2; ++i) dfree(c->map_xy[i]);
    return apply_geometry(c);
}

int mvsv_set_resize(mvsv_ctx* c, double factor)
{
    if (!c) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    if (!(factor == factor) || factor > 8.0) return fail(c, MVSV_ERR_INVALID, "resize factor must be in (0, 8]");
    if (factor <= 0.0 || factor == 1.0) factor = 0.0;       // off: cv::resize by 1 is the identity
    if (factor > 0.0 && factor < 1.0 / 64) return fail(c, MVSV_ERR_INVALID, "resize factor must be in (0, 8]");
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    const double old = c->resize_factor;
    c->resize_factor = factor;
    rc = apply_geometry(c);
    if (rc) { c->resize_factor = old; apply_geometry(c); }
    return rc;
}

int mvsv_tm(mvsv_ctx* c, const uint8_t* left, size_t lstride, const uint8_t* right, size_t rstride, size_t frame_stride,
            int batch, unsigned kernel_size, uint8_t* out, size_t ostride)
{
    if (!c || !left || !right || !out) return MVSV_ERR_INVALID;
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
    if (!c->tm_out) MVSV_CK(c, cudaMalloc(&c->tm_out, (size_t)c->maxB * H * c->pitch));
    MVSV_CK(c, cudaMemsetAsync(c->tm_out, 0, (size_t)batch * H * c->pitch, c->stream));   // cv::Scalar::all(0)
    // the reference's loops are `i < rows - kernelSize` in unsigned arithmetic: nothing to do unless k < rows, cols
    if ((int)kernel_size < H && (int)kernel_size < W) MVSV_CK(c, launch_tm(c, batch, (int)kernel_size, c->tm_out, c->pitch));
    MVSV_CK(c, cudaMemcpy2DAsync(out, ostride, c->tm_out, c->pitch, (size_t)W, (size_t)H * batch, cudaMemcpyDeviceToHost, c->stream));
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    return MVSV_OK;
}

int mvsv_set_Q(mvsv_ctx* c, const float q[16])
{
    if (!c || !q) return MVSV_ERR_INVALID;
    std::memcpy(c->Q, q, sizeof(float) * 16);
    c->has_Q = true;
    return MVSV_OK;
}

int mvsv_set_mean_rois(mvsv_ctx* c, const int* xywh, int n)
{
    if (!c || n < 0 || (n > 0 && !xywh)) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    for (int i = 0; i < n; ++i) {
        const int* r = xywh + 4 * i;
        if (r[0] < 0 || r[1] < 0 || r[2] < 1 || r[3] < 1 || r[0] + r[2] > c->W || r[1] + r[3] > c->H)
            return fail(c, MVSV_ERR_INVALID, "ROI outside the disparity map");
    }
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    dfree(c->rois);
    for (int k = 0; k < 2; ++k) free_slot(c, k, SLOT_MEANS);
    c->nrois = n;
    if (n == 0) return MVSV_OK;
    MVSV_CK(c, cudaMalloc(&c->rois, (size_t)n * 4 * sizeof(int)));
    rc = ensure_slots(c);
    if (rc) return rc;
    MVSV_CK(c, cudaMemcpy(c->rois, xywh, (size_t)n * 4 * sizeof(int), cudaMemcpyHostToDevice));
    return MVSV_OK;
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
    if (!c) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    if (age < 0 || age >= c->nslots) return fail(c, MVSV_ERR_INVALID, "age must be below the number of I/O slots");
    return download_slot(c, (c->cur + c->nslots - age) % c->nslots, disp, dstride, rectL, rectR, rstride, xyz, means);
}

int mvsv_set_io_slots(mvsv_ctx* c, int n)
{
    if (!c) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    if (n != 1 && n != 2) return fail(c, MVSV_ERR_INVALID, "1 or 2 I/O slots");
    if (n == c->nslots) return MVSV_OK;
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    MVSV_CK(c, cudaStreamSynchronize(c->copy_stream));
    if (n < c->nslots) free_slot(c, 1, SLOT_ALL);
    c->nslots = n;
    c->cur = 0;
    rc = ensure_slots(c);
    if (rc) { free_slot(c, 1, SLOT_ALL); c->nslots = 1; }
    return rc;
}

int mvsv_download_minmax(mvsv_ctx* c, int16_t* minmax)
{
    if (!c || !minmax) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    const int B = io(c).B;
    if (B < 1) return fail(c, MVSV_ERR_STATE, "nothing computed yet");
    if (!c->minmax) MVSV_CK(c, cudaMalloc(&c->minmax, (size_t)c->maxB * 2 * sizeof(int)));
    MVSV_CK(c, launch_minmax(c, B));
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

int mvsv_sync(mvsv_ctx* c)
{
    if (!c) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    MVSV_CK(c, cudaStreamSynchronize(c->stream));
    return MVSV_OK;
}

int mvsv_get_info(const mvsv_ctx* c, mvsv_info* info)
{
    if (!c || !info) return MVSV_ERR_INVALID;
    std::memset(info, 0, sizeof(*info));
    info->frame_width = c->fw; info->frame_height = c->fh; info->width = c->W; info->height = c->H; info->max_batch = c->maxB;
    if (c->has_sgbm) {
        info->sgbm_minX1 = c->sg.minX1; info->sgbm_W1 = c->sg.W1; info->sgbm_D = c->sg.D; info->sgbm_Dpad = c->sg.Dp;
        info->sgbm_npaths = c->sg.npaths;
    }
    info->num_rois = c->nrois; info->device = c->device; info->sgbm_td_cluster = c->has_sgbm ? c->td_nc : 0;
    info->last_batch = c->slot[c->cur].B;
    info->sgbm_s8 = c->last_s8 ? 1 : 0;
    info->bm_col8 = (c->has_bm && c->bm.col8 && !(c->debug_flags & 2u)) ? 1 : 0;
    return MVSV_OK;
}

void* mvsv_stream(mvsv_ctx* c) { return c ? (void*)c->stream : nullptr; }
unsigned long long mvsv_launch_count(const mvsv_ctx* c) { return c ? c->launches : 0ull; }

int mvsv_host_alloc(void** p, size_t bytes)
{
    if (!p) return MVSV_ERR_INVALID;
    return cudaHostAlloc(p, bytes, cudaHostAllocDefault) == cudaSuccess ? MVSV_OK : MVSV_ERR_NOMEM;
}
int mvsv_host_free(void* p) { return cudaFreeHost(p) == cudaSuccess ? MVSV_OK : MVSV_ERR_CUDA; }

int mvsv_timer_start(mvsv_ctx* c)
{
    if (!c) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    if (!c->timer_a) { MVSV_CK(c, cudaEventCreate(&c->timer_a)); MVSV_CK(c, cudaEventCreate(&c->timer_b)); }
    MVSV_CK(c, cudaEventRecord(c->timer_a, c->stream));
    return MVSV_OK;
}

int mvsv_timer_stop(mvsv_ctx* c, float* ms)
{
    if (!c || !ms || !c->timer_a) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    MVSV_CK(c, cudaEventRecord(c->timer_b, c->stream));
    MVSV_CK(c, cudaEventSynchronize(c->timer_b));
    MVSV_CK(c, cudaEventElapsedTime(ms, c->timer_a, c->timer_b));
    return MVSV_OK;
}

int mvsv_profile_enable(mvsv_ctx* c, int enable)
{
    if (!c) return MVSV_ERR_INVALID;
    c->prof = enable != 0;
    return MVSV_OK;
}

int mvsv_profile_read(mvsv_ctx* c, float* ms, int* counts, int n)
{
    if (!c || !ms || !counts || n < KID_COUNT) return MVSV_ERR_INVALID;
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
}

const char* mvsv_kernel_name(int kid) { return (kid >= 0 && kid < KID_COUNT) ? kKernelNames[kid] : ""; }

int mvsv_debug_set_flags(mvsv_ctx* c, unsigned flags)
{
    if (!c) return MVSV_ERR_INVALID;
    c->debug_flags = flags;
    if (c->has_sgbm) c->td_nc = sgbm_choose_td_cluster(c);
    return MVSV_OK;
}

int mvsv_debug_postfilter(mvsv_ctx* c, const int16_t* maps, size_t stride, int batch, int median, int newVal,
                          int maxSpeckleSize, int maxDiff, unsigned stages)
{
    if (!c) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    // the next I/O slot, taken as run() takes it
    const int k = (c->cur + 1) % c->nslots;
    IoSlot& slot = c->slot[k];
    if (!maps || batch < 1 || batch > c->maxB) return fail(c, MVSV_ERR_INVALID, "bad map pointer or batch size");
    if (stride < (size_t)c->W * sizeof(int16_t)) return fail(c, MVSV_ERR_INVALID, "stride smaller than the map width");
    if (stages & ~(unsigned)(MVSV_STAGE_XYZ | MVSV_STAGE_MEANS))
        return fail(c, MVSV_ERR_INVALID, "post-filter hook: only MVSV_STAGE_XYZ and MVSV_STAGE_MEANS");
    if (maxSpeckleSize > 0 && (newVal < -32768 || newVal > 32767)) return fail(c, MVSV_ERR_INVALID, "newVal does not fit CV_16S");
    rc = check_consumers(c, slot, stages);
    if (rc) return rc;
    if ((stages & MVSV_STAGE_XYZ) && !slot.xyz) MVSV_CK(c, cudaMalloc(&slot.xyz, (size_t)c->maxB * c->H * c->W * 3 * sizeof(float)));

    c->cur = k;                 // the slot is taken: a failing step leaves it empty
    auto submit = [&]() -> int {
        const size_t row = (size_t)c->W * sizeof(int16_t), npx = (size_t)batch * c->H * c->W;
        MVSV_CK(c, cudaMemcpy2DAsync(c->disp_raw, row, maps, stride, row, (size_t)c->H * batch, cudaMemcpyHostToDevice, c->stream));
        const bool speckle = maxSpeckleSize > 0;
        if (median) MVSV_CK(c, launch_median(c, c->disp_raw, speckle ? c->disp_med : slot.disp, batch));
        if (speckle)
            MVSV_CK(c, launch_speckle(c, median ? c->disp_med : c->disp_raw, slot.disp, batch, newVal, maxSpeckleSize, maxDiff));
        if (!median && !speckle)
            MVSV_CK(c, cudaMemcpyAsync(slot.disp, c->disp_raw, npx * sizeof(int16_t), cudaMemcpyDeviceToDevice, c->stream));
        if (stages & MVSV_STAGE_XYZ) MVSV_CK(c, launch_xyz(c, batch));
        if (stages & MVSV_STAGE_MEANS) MVSV_CK(c, launch_means(c, batch));
        MVSV_CK(c, cudaEventRecord(slot.done, c->stream));
        MVSV_CK(c, cudaEventRecord(c->ev_done, c->stream));
        return MVSV_OK;
    };
    rc = submit();
    slot.B = rc ? 0 : batch;
    slot.stages = rc ? 0 : stages;
    return rc;
}

long long mvsv_debug_read(mvsv_ctx* c, int which, void* host, size_t cap)
{
    if (!c || !host) return MVSV_ERR_INVALID;
    int rc = bind(c);
    if (rc) return rc;
    const void* src = nullptr;
    size_t bytes = 0;
    if (which == 7 || which == 8) {
        const int cam = which - 7;
        if (!c->has_maps[cam]) return fail(c, MVSV_ERR_STATE, "no rectification map for this camera");
        src = c->map_xy[cam];
        bytes = (size_t)c->roi[2] * c->roi[3] * sizeof(int2);
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
}

}  // extern "C"
