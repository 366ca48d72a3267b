// One ctx over several engines (mvsv_init_devices): every batch is cut into contiguous shares, one per part, and every
// setter is repeated on every part.  Host code only: the parts are ordinary single-device engines.
#include "mvsv_internal.h"

#include <algorithm>
#include <cstring>
#include <new>

struct Parts {
    std::vector<mvsv_ctx*> ctx;              // part k: an engine of maxB / n frames on device[k]
    std::vector<int> device;
    // the slice of the ctx's frame -> rig table each part holds (mvsv_set_frame_rigs of the part); {-1}: unknown
    std::vector<std::vector<int>> rigs;
    bool broken = false;                     // a setter failed in a way that can have left the parts different
};

namespace {

int fail(mvsv_ctx* c, int code, const std::string& msg)
{
    c->err = msg;
    return code;
}

int n_parts(const mvsv_ctx* c) { return (int)c->parts->ctx.size(); }

// frames [*first, *end) of a compute of `batch` frames go to part k
void share(int k, int n, int batch, int* first, int* end)
{
    *first = (int)((long long)k * batch / n);
    *end = (int)((long long)(k + 1) * batch / n);
}

// a failure of part k: its text, prefixed with the part, becomes the ctx's
int part_failed(mvsv_ctx* c, int k, int rc)
{
    return fail(c, rc, "part " + std::to_string(k) + " (device " + std::to_string(c->parts->device[k]) + "): " +
                           c->parts->ctx[k]->err);
}

// makes part k's device current (its calls that do not bind themselves)
int bind_part(mvsv_ctx* c, int k)
{
    mvsv_ctx* p = c->parts->ctx[k];
    const cudaError_t e = cudaSetDevice(p->device);
    if (e == cudaSuccess) return MVSV_OK;
    p->err = std::string("cudaSetDevice: ") + cudaGetErrorString(e);
    return part_failed(c, k, MVSV_ERR_CUDA);
}

int check_usable(mvsv_ctx* c)
{
    if (c->parts->broken)
        return fail(c, MVSV_ERR_STATE, "an earlier call failed on one part only, so the parts no longer hold the same state ("
                                       "only mvsv_destroy, mvsv_last_error and mvsv_get_info remain): " + c->err);
    return MVSV_OK;
}

// The parts keep their own I/O slots in lockstep with the ctx's.  A call that drops results (a geometry change, fewer
// I/O slots) drops them on every part; the last part holds frames of every compute, so it tells which slots lost theirs.
void follow_slots(mvsv_ctx* c)
{
    const mvsv_ctx* last = c->parts->ctx.back();
    c->nslots = last->nslots;
    c->cur = last->cur;
    for (int k = 0; k < 2; ++k)
        if (last->slot[k].B == 0) c->slot[k].B = 0;
}

// part k receives its slice of the frame -> rig table for frames [first, end) unless it holds it already
int send_rigs(mvsv_ctx* c, int k, int first, int end)
{
    const int n = (int)c->frame_rig.size();
    const int a = std::min(first, n), b = std::min(end, n);
    std::vector<int> slice(c->frame_rig.begin() + a, c->frame_rig.begin() + b);
    std::vector<int>& held = c->parts->rigs[k];
    if (slice == held) return MVSV_OK;
    mvsv_ctx* p = c->parts->ctx[k];
    const int rc = mvsv_set_frame_rigs(p, slice.data(), (int)slice.size());
    if (rc) {
        held.assign(1, -1);
        return part_failed(c, k, rc);
    }
    held.swap(slice);
    return MVSV_OK;
}

}  // namespace

int parts_each(mvsv_ctx* c, bool setter, int (*call)(mvsv_ctx* part, const void* arg), const void* arg)
{
    int rc = check_usable(c);
    if (rc) return rc;
    for (int k = 0; k < n_parts(c); ++k) {
        mvsv_ctx* p = c->parts->ctx[k];
        p->err.clear();
        rc = call(p, arg);
        if (rc < 0) {
            // every part holds the same state, so an argument or state rejection comes from part 0 before any part
            // changed; a CUDA or allocation error can leave part 0 half changed, and any failure past it leaves the
            // parts before it changed
            if (setter && (k > 0 || rc == MVSV_ERR_CUDA || rc == MVSV_ERR_NOMEM)) c->parts->broken = true;
            part_failed(c, k, rc);
            follow_slots(c);
            return rc;
        }
    }
    if (setter) follow_slots(c);
    return MVSV_OK;
}

int parts_unsupported(mvsv_ctx* c, const char* what)
{
    const int rc = check_usable(c);
    if (rc) return rc;
    return fail(c, MVSV_ERR_UNSUPPORTED, std::string(what) + " is not available on a multi-device ctx (mvsv_init_devices); "
                                                             "call it on a single-device engine");
}

int parts_set_frame_rigs(mvsv_ctx* c, const int* rig_of_frame, int n)
{
    int rc = check_usable(c);
    if (rc) return rc;
    if (n < 0 || (n > 0 && !rig_of_frame)) return MVSV_ERR_INVALID;
    if (n > c->maxB) return fail(c, MVSV_ERR_INVALID, "more frames than max_batch");
    for (int i = 0; i < n; ++i)
        if (rig_of_frame[i] < 0 || rig_of_frame[i] >= MVSV_MAX_RIGS)
            return fail(c, MVSV_ERR_INVALID, "rig of frame " + std::to_string(i) + " outside [0, MVSV_MAX_RIGS)");
    // the parts receive their slices when a compute needs them (send_rigs)
    c->frame_rig.assign(rig_of_frame, rig_of_frame + n);
    return MVSV_OK;
}

int parts_compute(mvsv_ctx* c, const uint8_t* left, size_t lstride, const uint8_t* right, size_t rstride, size_t frame_stride,
                  int batch, unsigned stages, bool device_src)
{
    int rc = check_usable(c);
    if (rc) return rc;
    if (!left || !right || batch < 1 || batch > c->maxB) return fail(c, MVSV_ERR_INVALID, "bad image pointers or batch size");
    const int n = n_parts(c);
    // phase 1: every part that gets frames checks them (and allocates what they need) before any part takes a slot,
    // so that a rejected compute leaves the results of earlier ones downloadable on every part
    for (int k = 0; k < n; ++k) {
        int first, end;
        share(k, n, batch, &first, &end);
        if (first == end) continue;
        rc = send_rigs(c, k, first, end);
        if (rc) return rc;
        mvsv_ctx* p = c->parts->ctx[k];
        rc = compute_check(p, left + first * frame_stride, lstride, right + first * frame_stride, rstride, end - first, stages);
        if (rc) return part_failed(c, k, rc);
    }
    // phase 2: every part takes its next slot (a part without frames leaves it empty) and submits its share
    c->cur = (c->cur + 1) % c->nslots;
    c->slot[c->cur].B = 0;
    for (int k = 0; k < n; ++k) {
        int first, end;
        share(k, n, batch, &first, &end);
        mvsv_ctx* p = c->parts->ctx[k];
        if (first == end) {
            compute_skip(p);
            continue;
        }
        rc = compute_submit(p, left + first * frame_stride, lstride, right + first * frame_stride, rstride, frame_stride,
                            end - first, stages, device_src);
        if (rc) {
            // the slot of this compute is left empty on every part: the parts before k drop what they submitted, the
            // parts after k take their slot empty
            for (int j = 0; j < k; ++j) { io(c->parts->ctx[j]).B = 0; io(c->parts->ctx[j]).stages = 0; }
            for (int j = k + 1; j < n; ++j) compute_skip(c->parts->ctx[j]);
            return part_failed(c, k, rc);
        }
    }
    c->slot[c->cur].B = batch;
    c->slot[c->cur].stages = stages;
    return MVSV_OK;
}

int parts_download(mvsv_ctx* c, int age, int16_t* disp, size_t dstride, uint8_t* rectL, uint8_t* rectR, size_t rstride,
                   float* xyz, float* means)
{
    int rc = check_usable(c);
    if (rc) return rc;
    if (age < 0 || age >= c->nslots) return fail(c, MVSV_ERR_INVALID, "age must be below the number of I/O slots");
    const int s = (c->cur + c->nslots - age) % c->nslots, batch = c->slot[s].B, n = n_parts(c);
    if (batch < 1) return fail(c, MVSV_ERR_STATE, "nothing computed yet");
    // every part's copies are queued before the first wait, so that the parts' downloads run side by side
    int queued = 0;
    for (; queued < n; ++queued) {
        int first, end;
        share(queued, n, batch, &first, &end);
        if (first == end) continue;
        mvsv_ctx* p = c->parts->ctx[queued];
        const size_t rows = (size_t)first * p->H;
        rc = bind_part(c, queued);
        if (rc) break;
        rc = download_enqueue(p, s, disp ? (int16_t*)((uint8_t*)disp + rows * dstride) : nullptr, dstride,
                              rectL ? rectL + rows * rstride : nullptr, rectR ? rectR + rows * rstride : nullptr, rstride,
                              xyz ? xyz + rows * p->W * 3 : nullptr, means ? means + (size_t)first * p->nrois : nullptr);
        if (rc) {
            part_failed(c, queued, rc);
            break;
        }
    }
    // wait also after a failure: the caller's buffers must not be written once the call has returned
    for (int k = 0; k <= std::min(queued, n - 1); ++k) {
        int first, end;
        share(k, n, batch, &first, &end);
        if (first == end) continue;
        int w = bind_part(c, k);
        if (!w) w = download_wait(c->parts->ctx[k]);
        if (w && !rc) rc = part_failed(c, k, w);
    }
    return rc;
}

int parts_download_minmax(mvsv_ctx* c, int16_t* minmax)
{
    int rc = check_usable(c);
    if (rc) return rc;
    const int batch = c->slot[c->cur].B, n = n_parts(c);
    if (batch < 1) return fail(c, MVSV_ERR_STATE, "nothing computed yet");
    // the reductions of all parts are launched before the first result is read back
    for (int pass = 0; pass < 2; ++pass)
        for (int k = 0; k < n; ++k) {
            int first, end;
            share(k, n, batch, &first, &end);
            if (first == end) continue;
            rc = bind_part(c, k);
            if (rc) return rc;
            mvsv_ctx* p = c->parts->ctx[k];
            rc = pass == 0 ? minmax_launch(p) : minmax_read(p, minmax + 2 * (size_t)first);
            if (rc) return part_failed(c, k, rc);
        }
    return MVSV_OK;
}

int parts_timer_stop(mvsv_ctx* c, float* ms)
{
    int rc = check_usable(c);
    if (rc) return rc;
    if (!ms) return MVSV_ERR_INVALID;
    float longest = 0.f;
    for (int k = 0; k < n_parts(c); ++k) {
        float t = 0.f;
        rc = mvsv_timer_stop(c->parts->ctx[k], &t);
        if (rc) return part_failed(c, k, rc);
        longest = std::max(longest, t);
    }
    *ms = longest;
    return MVSV_OK;
}

int parts_get_info(const mvsv_ctx* c, mvsv_info* info)
{
    const int rc = mvsv_get_info(c->parts->ctx[0], info);
    if (rc) return rc;
    info->max_batch = c->maxB;
    info->last_batch = c->slot[c->cur].B;
    info->device = c->device;
    return MVSV_OK;
}

unsigned long long parts_launch_count(const mvsv_ctx* c)
{
    unsigned long long n = 0;
    for (const mvsv_ctx* p : c->parts->ctx) n += mvsv_launch_count(p);
    return n;
}

void parts_destroy(mvsv_ctx* c)
{
    for (mvsv_ctx* p : c->parts->ctx) mvsv_destroy(p);
    delete c->parts;
    delete c;
}

extern "C" {

int mvsv_init_devices(const int* devices, int n, int frame_width, int frame_height, int max_batch, mvsv_ctx** out)
{
    if (!out) return MVSV_ERR_INVALID;
    *out = nullptr;
    if (!devices || n < 1 || n > max_batch) {
        init_error() = "mvsv_init_devices: the device list must name between 1 and max_batch devices";
        return MVSV_ERR_INVALID;
    }
    if (n == 1) return mvsv_init(devices[0], frame_width, frame_height, max_batch, out);
    mvsv_ctx* c = new (std::nothrow) mvsv_ctx();
    Parts* parts = c ? new (std::nothrow) Parts() : nullptr;
    if (!parts) { delete c; return MVSV_ERR_NOMEM; }
    c->parts = parts;
    const int cap = (max_batch + n - 1) / n;
    for (int k = 0; k < n; ++k) {
        mvsv_ctx* p = nullptr;
        const int rc = mvsv_init(devices[k], frame_width, frame_height, cap, &p);
        if (rc) {
            const std::string why = init_error();
            parts_destroy(c);
            init_error() = "mvsv_init_devices: part " + std::to_string(k) + " (device " + std::to_string(devices[k]) + "): " + why;
            return rc;
        }
        parts->ctx.push_back(p);
        parts->device.push_back(devices[k]);
    }
    parts->rigs.resize(n);
    c->device = devices[0];
    c->fw = c->W = frame_width; c->fh = c->H = frame_height;
    c->maxB = cap * n;
    *out = c;
    return MVSV_OK;
}

int mvsv_get_devices(const mvsv_ctx* c, int* devices, int n)
{
    if (!c || n < 0 || (n > 0 && !devices)) return MVSV_ERR_INVALID;
    if (!is_multi(c)) {
        if (n > 0) devices[0] = c->device;
        return 1;
    }
    const std::vector<int>& d = c->parts->device;
    std::copy(d.begin(), d.begin() + std::min(n, (int)d.size()), devices);
    return (int)d.size();
}

}  // extern "C"
