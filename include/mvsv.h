/*
 * mvsv.h -- C ABI of the B200-native stereo disparity engine (libmvsv.so).
 *
 * This is the drop-in boundary for mvStereoVision3's hot path.  Every entry point names the
 * reference interface it replaces (paths relative to the reference repository root).  Plain
 * pointers and sizes only; no C++/torch/OpenCV types cross this line.  All functions return
 * MVSV_OK (0) or a negative error code and never throw; mvsv_last_error() gives the text.
 * There is no CPU fallback: without a CUDA device mvsv_init fails with MVSV_ERR_CUDA.
 *
 * Threading contract (reference: one worker std::thread calls Disparity::sgbm,
 * trgt/demo.cpp:68-77,195): a ctx is thread-compatible -- any thread may call, one at a time.
 * Several ctxs (one per GPU or stream) may run concurrently.
 *
 * Multi-device ctx (mvsv_init_devices): one ctx over several engines, each on one of the listed devices.  Every entry
 * point accepts it; the comments below say where its behaviour differs from that of an mvsv_init ctx.
 */
#ifndef MVSV_H_
#define MVSV_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mvsv_ctx mvsv_ctx;

enum {
    MVSV_OK = 0,
    MVSV_ERR_INVALID = -1,     /* bad argument / parameter outside the bit-exact contract */
    MVSV_ERR_CUDA = -2,        /* CUDA runtime error (text in mvsv_last_error)            */
    MVSV_ERR_NOMEM = -3,
    MVSV_ERR_STATE = -4,       /* call order (e.g. compute before set_*_params)           */
    MVSV_ERR_UNSUPPORTED = -5
};

/* stage bit-mask for mvsv_compute* */
enum {
    MVSV_STAGE_RECTIFY = 1,    /* cv::remap x2 + crop      src/Stereosystem.cpp:252-256 */
    MVSV_STAGE_SGBM = 2,       /* Disparity::sgbm          src/disparity.cpp:6-10       */
    MVSV_STAGE_BM = 4,         /* Disparity::bm            src/disparity.cpp:18-22      */
    MVSV_STAGE_XYZ = 8,        /* Utility::dmap2pcl loop   src/utility.cpp:242-262      */
    MVSV_STAGE_MEANS = 16,     /* Utility::calcMeanDisparity per ROI  src/utility.cpp:265-285 */
    /* Utility::dmap2pcl  src/utility.cpp:242-262: the point list.  Over the whole batch, in (frame, row, column) order,
     * every pixel of the final map with disparity > 0 gives the three floats MVSV_STAGE_XYZ writes for it (same
     * arithmetic, same Z = 0 where Z/1000 is infinite), packed one after the other; fetched with mvsv_download_points.
     * With or without MVSV_STAGE_XYZ, after either matcher; like XYZ it needs the Q of every frame's rig. */
    MVSV_STAGE_POINTS = 32,
    /* MeanDisparityDetection::detectObstacles and SamplepointDetection::detectObstacles  src/MeanDisparityDetection.cpp:
     * 71-266, src/SamplePointDetection.cpp:29-178 (as mirrored by include/mvsv_detection.hpp): the range test and
     * Utility::calcCoordinate of every ROI mean, on the device.  Needs MVSV_STAGE_MEANS in the same compute and a table
     * from mvsv_set_detection; the found-obstacle lists are fetched with mvsv_download_obstacles. */
    MVSV_STAGE_DETECT = 64
};

/* Field order of the first nine ints == struct Disparity::sgbmParameters (inc/disparity.h:17-27).
 * P1/P2 are never set by the reference (src/disparity.cpp:83-90): leave 0 to get OpenCV's 2 / 5. */
typedef struct mvsv_sgbm_params {
    int minDisp, numDisp, blockSize, disp12MaxDiff, preFilterCap, uniquenessRatio;
    int speckleWindowSize, speckleRange, disparityMode; /* 1 = MODE_HH (8 paths), else MODE_SGBM (5 paths) */
    int P1, P2;
} mvsv_sgbm_params;

/* cv::StereoBM state as driven by configs/bm.yml (PREFILTER_XSOBEL, minDisparity 0). */
typedef struct mvsv_bm_params {
    int numDisp, blockSize, preFilterCap, textureThreshold, uniquenessRatio;
} mvsv_bm_params;

typedef struct mvsv_info {
    int frame_width, frame_height;   /* raw camera frame                                        */
    int width, height;               /* rectified + cropped pair == disparity map size          */
    int max_batch;
    int sgbm_minX1, sgbm_W1, sgbm_D, sgbm_Dpad, sgbm_npaths;   /* evaluated cost domain          */
    int num_rois;
    int device;
    int sgbm_td_cluster;             /* column strips (CTAs) per frame of the fused previous-row sweep at max_batch
                                        (0: independent passes)                                */
    int last_batch;                  /* stereo pairs of the last compute == frames mvsv_download copies      */
    int sgbm_s8;                     /* the last SGBM compute kept the aggregated volume as one byte per cell
                                        (npaths * P2 <= 255: every path cost is C + e, 0 <= e <= P2)              */
    int bm_col8;                     /* the StereoBM parameters keep the column-sum volume as one byte per cell
                                        (blockSize * 2 * preFilterCap <= 255, e.g. configs/bm.yml: 21 * 4 = 84)   */
} mvsv_info;

/* Create an engine on CUDA device `device` for raw frames of frame_width x frame_height, holding up to
 * max_batch stereo pairs in flight per compute call.  Replaces the cv::Ptr<cv::StereoSGBM>/StereoBM
 * objects the drivers create (trgt/demo.cpp:190-194) and Stereosystem's rectification state. */
int mvsv_init(int device, int frame_width, int frame_height, int max_batch, mvsv_ctx** out);
void mvsv_destroy(mvsv_ctx* ctx);
const char* mvsv_last_error(const mvsv_ctx* ctx); /* ctx may be NULL: error of the last failed mvsv_init(_devices) */

/* One ctx over the devices devices[0 .. n-1] (one engine per GPU of a box, behind one handle).  Part k is an engine of
 * mvsv_init(devices[k], frame_width, frame_height, ceil(max_batch / n)); the ctx holds n * ceil(max_batch / n) frames.
 * A device may be listed more than once: its parts are separate engines, each with its own volumes.  n == 1 is exactly
 * mvsv_init(devices[0], ...).  Rejected with MVSV_ERR_INVALID: devices == NULL, n < 1, n > max_batch, and whatever
 * mvsv_init rejects for one of the parts (also with its code, e.g. MVSV_ERR_CUDA without a device); a failure frees the
 * parts already created, leaves *out == NULL and puts the text, prefixed with the part, in mvsv_last_error(NULL).
 *   Compute: a batch of b frames gives part k the contiguous frames [floor(k*b/n), floor((k+1)*b/n)), read at
 *     base + first*frame_stride (host or device memory; device inputs on another device are copied peer to peer).  When
 *     b < n some parts get no frames.  Every part is checked (arguments, state, rigs, consumers, allocations) before any
 *     part submits: a rejected compute leaves the results of earlier ones downloadable, as on one engine; a failure while
 *     submitting leaves the compute's I/O slot empty on every part.  Every compute advances the I/O slot of every part,
 *     so the slots of all parts always hold the same compute.
 *   Setters (parameters, filters, maps, rectification, resize, Q, ROIs, I/O slots) are repeated on every part in order.
 *     The parts hold the same state, so an argument or state rejection comes from part 0 before any part changed.  A
 *     CUDA or allocation error of such a call (e.g. a device with less free memory than the others) can leave the parts
 *     different and marks the ctx broken: every later call except mvsv_destroy, mvsv_last_error and mvsv_get_info then
 *     returns MVSV_ERR_STATE.  A part's error text is prefixed with its index and device.
 *   mvsv_set_frame_rigs keeps the whole table; a compute hands each part the table from the part's first frame on (as
 *     far as the part's capacity reaches) when it differs from the one the part holds, which waits for that part's
 *     stream.  While the batch size stays the same nothing is re-sent; a batch size that moves a part's first frame
 *     costs that wait with a rig table installed.
 *   Downloads queue the copies of every part (at out + first*height*stride, XYZ and means likewise) before they wait, so
 *     that the parts' copies run side by side; mvsv_download_minmax launches on every part, then gathers;
 *     mvsv_download_points fetches every part's frame offsets, then queues every part's points after the points of the
 *     parts before it.
 *   mvsv_get_info: part 0's fields, except max_batch (all parts), last_batch (all frames of the last compute) and device
 *     (devices[0]).  mvsv_sync: every part.  mvsv_launch_count: the sum.  mvsv_timer_start / stop: events on every part;
 *     stop returns the longest part's interval.  mvsv_stream: NULL.
 *   Not available (MVSV_ERR_UNSUPPORTED; use a single-device engine): mvsv_tm, mvsv_profile_enable / read and the test
 *     hooks mvsv_debug_set_flags, mvsv_debug_read, mvsv_debug_postfilter.
 * No reference counterpart (the reference runs one pair at a time on the CPU). */
int mvsv_init_devices(const int* devices, int n, int frame_width, int frame_height, int max_batch, mvsv_ctx** out);
/* The devices of a ctx: returns the number of parts (1 for an mvsv_init ctx) and writes up to n of their ids. */
int mvsv_get_devices(const mvsv_ctx* ctx, int* devices, int n);

/* Replaces the eight StereoSGBM setters + setMode of Disparity::loadSGBMParameters
 * (src/disparity.cpp:83-95).  Parameters outside the bit-exact contract are rejected:
 * numDisp in [8,512] and a multiple of 8; blockSize^2*(2*ftzero+63)+P2 <= 32767 (SURVEY.md section 7).
 * numDisp > 256 also needs a non-empty cost domain, W + min(minDisp, 0) > max(minDisp + numDisp, 0) (MVSV_ERR_INVALID
 * otherwise, also for a later geometry change that would empty it); a cost volume of one frame above 2^31 cells
 * (H * W1 * padded numDisp, e.g. 3840x2160 at numDisp > 256) is MVSV_ERR_UNSUPPORTED. */
int mvsv_set_sgbm_params(mvsv_ctx* ctx, const mvsv_sgbm_params* p);
/* cv::StereoBM::create(numDisp, blockSize) + setters (trgt/disparityTest.cpp:268, configs/bm.yml). */
int mvsv_set_bm_params(mvsv_ctx* ctx, const mvsv_bm_params* p);
/* The post-filters of cv::StereoBM, in cv2's own units (cv::StereoBM::setDisp12MaxDiff / setSpeckleWindowSize /
 * setSpeckleRange):
 *   disp12MaxDiff     >= 0: left-right check, a pixel is FILTERED (-16) when the disparities seen from the right
 *                     image at both of its integer neighbours differ from it by more than disp12MaxDiff pixels;
 *                     0 is the strictest check, < 0 switches it off.  Needs width <= 4096.
 *   speckleWindowSize > 0: cv::filterSpeckles(disp, -16, speckleWindowSize, speckleRange) after the check;
 *                     speckleRange is compared with the x16 fixed-point values as given (StereoSGBM multiplies it
 *                     by 16, StereoBM does not).  0 switches it off.
 * Defaults -1 / 0 / 0 (cv::StereoBM's): the engine computes what it computes without this call.  The setting is kept
 * across mvsv_set_bm_params and geometry changes.  Rejected: speckleWindowSize < 0, speckleRange < 0 with a window. */
int mvsv_set_bm_filters(mvsv_ctx* ctx, int disp12MaxDiff, int speckleWindowSize, int speckleRange);

/* Replaces Stereosystem::initRectification's map state (src/Stereosystem.cpp:214-220): float CV_32FC1
 * maps of one camera (cam 0 = left, 1 = right), frame-sized, plus mDisplayROI.  The maps are converted once
 * to OpenCV's fixed-point (CV_16SC2 + 5-bit fractions) form on the device.  stride is in bytes. */
int mvsv_upload_rectify_maps(mvsv_ctx* ctx, int cam, const float* mapx, const float* mapy, size_t stride_bytes,
                             int roi_x, int roi_y, int roi_w, int roi_h);
/* The same state built on the device from the calibration itself: replaces the call
 * cv::initUndistortRectifyMap(K, D, R, P, size, CV_32FC1, map1, map2) of Stereosystem::initRectification
 * (src/Stereosystem.cpp:214-217) together with the upload above.  K: 3x3 camera matrix (intrinsic.yml, halved for
 * binning as src/Stereosystem.cpp:203-208 does), dist: n_dist = 0, 4 or 5 coefficients k1 k2 p1 p2 [k3]
 * (mDistCoeffs), R: 3x3 rectifying rotation and P: 3x4 projection from cv::stereoRectify (mR0/mR1, mP0/mP1),
 * all row-major doubles as the cv::Mat's hold them.  The fixed-point maps equal the ones OpenCV derives from its
 * float maps (cv2 4.13: identical for the reference's three calibrations, tests/test_rectify_maps.py). */
int mvsv_set_rectification(mvsv_ctx* ctx, int cam, const double K[9], const double* dist, int n_dist,
                           const double R[9], const double P[12], int roi_x, int roi_y, int roi_w, int roi_h);
/* Stereosystem::getRectifiedImagepair(sip, factor) (src/Stereosystem.cpp:279-315): after remap + crop the pair is
 * scaled with cv::resize(roi, dst, cv::Size(0,0), factor, factor) (INTER_LINEAR, which OpenCV replaces by its 2x2
 * area average at factor 0.5 -- the value trgt/test.cpp:213 passes).  Applies to MVSV_STAGE_RECTIFY computes; width
 * and height of mvsv_get_info become cvRound(roi * factor).  factor <= 0 or == 1 switches it off. */
int mvsv_set_resize(mvsv_ctx* ctx, double factor);
/* Stereosystem::resetRectification (src/Stereosystem.cpp:317-320): inputs are taken as already rectified.  Drops the
 * maps of every rig. */
int mvsv_reset_rectification(mvsv_ctx* ctx);

/* Q as the CV_32F copy the drivers hold (trgt/demo.cpp:179-180), row-major 4x4. */
int mvsv_set_Q(mvsv_ctx* ctx, const float q[16]);

/* Several stereo rigs in one batch.  The reference holds one Stereosystem (one calibration) per rig; an application with
 * N rigs holds N of them and the Q of each.  Here one engine holds up to MVSV_MAX_RIGS calibrations and every frame of a
 * compute names the rig it comes from, so that the frames of all rigs share one batch and one set of cost volumes.
 * Rig 0 is the state the calls above set: mvsv_upload_rectify_maps, mvsv_set_rectification and mvsv_set_Q are the
 * rig == 0 cases of the three calls below, which take the same arguments plus `rig` in [0, MVSV_MAX_RIGS).
 * Geometry: all rigs share the frame size, the display-ROI width and height, and the resize factor; roi_x / roi_y may
 * differ per rig (both cameras of one rig share one ROI).  Installing maps whose ROI size differs from that of maps
 * another rig holds is MVSV_ERR_INVALID. */
#define MVSV_MAX_RIGS 64
/* Stereosystem::initRectification's map state of rig `rig` (src/Stereosystem.cpp:214-220), see mvsv_upload_rectify_maps. */
int mvsv_upload_rectify_maps_rig(mvsv_ctx* ctx, int rig, int cam, const float* mapx, const float* mapy, size_t stride_bytes,
                                 int roi_x, int roi_y, int roi_w, int roi_h);
/* cv::initUndistortRectifyMap of rig `rig` (src/Stereosystem.cpp:214-217), see mvsv_set_rectification. */
int mvsv_set_rectification_rig(mvsv_ctx* ctx, int rig, int cam, const double K[9], const double* dist, int n_dist,
                               const double R[9], const double P[12], int roi_x, int roi_y, int roi_w, int roi_h);
/* The Q of rig `rig` (trgt/demo.cpp:179-180), see mvsv_set_Q. */
int mvsv_set_Q_rig(mvsv_ctx* ctx, int rig, const float q[16]);
/* Frame i of every later compute (mvsv_compute, mvsv_compute_device, and the XYZ / points of mvsv_debug_postfilter) comes from
 * rig rig_of_frame[i], i < n <= max_batch; frames past n, or all frames when n == 0, come from rig 0.  Waits for the
 * engine's stream before it replaces the table: computes already submitted keep the assignment they were submitted
 * with.  A compute whose frames name a rig without both maps (MVSV_STAGE_RECTIFY) or without Q (MVSV_STAGE_XYZ) fails
 * with MVSV_ERR_STATE before it takes an I/O slot: the results of earlier computes stay downloadable (MVSV_STAGE_POINTS
 * needs Q as MVSV_STAGE_XYZ does).  Nothing in the
 * matchers, post-filters, ROI means or min/max depends on the rig.  No reference counterpart (one Stereosystem per rig,
 * src/Stereosystem.cpp:244-277, each rectifying its own pairs on the CPU). */
int mvsv_set_frame_rigs(mvsv_ctx* ctx, const int* rig_of_frame, int n);
/* ROIs (x, y, w, h quadruples in disparity-map coordinates) whose mean disparity is wanted:
 * the 81 Subimages (src/MeanDisparityDetection.cpp:80-93) and/or the 5x5 Samplepoint windows
 * (src/SamplePointDetection.cpp:38-47), already shifted by the dMapROI offset (trgt/demo.cpp:87-113). */
/* The ROIs are coordinates of the current disparity-map geometry: a call that changes width/height
 * (mvsv_upload_rectify_maps, mvsv_set_rectification, mvsv_set_resize, mvsv_reset_rectification) drops them, and
 * MVSV_STAGE_MEANS then fails with MVSV_ERR_STATE until they are set again. */
int mvsv_set_mean_rois(mvsv_ctx* ctx, const int* xywh, int n);

/* Obstacle detection on the device (MVSV_STAGE_DETECT).  The host mirror include/mvsv_detection.hpp defines the result:
 * for every frame f of a compute and every ROI i with a detector d = detector_of_roi[i] >= 0, with rig = the frame's rig
 * (mvsv_set_frame_rigs), Q its Q and value = the ROI mean of MVSV_STAGE_MEANS,
 *   first  = Utility::calcDMapValues({0, 0, min_distance[d] * 1000}, Q).dValue,
 *   second = Utility::calcDMapValues({0, 0, max_distance[d] * 1000}, Q).dValue   (float arithmetic, as in the header),
 * ROI i is a hit iff value < first && value > second (the reference's test, kept as is), and a
 * hit gives the record {roi = i, value, xyzw = Utility::calcCoordinate({value, cx_i, cy_i}, Q)}: the Vec4 the detectors
 * push to getFoundPoints(), bit for bit (products accumulated in double in the order k = 0..3, each component rounded
 * to float, then multiplied by the double reciprocal of the fourth; z := 0 where z / 1000 is infinite).  A frame's
 * records come in ascending ROI order, the detectors interleaved by ROI index as their two host loops visit them. */
typedef struct mvsv_obstacle {
    int32_t roi;
    float value;
    float xyzw[4];
} mvsv_obstacle;   /* 24 bytes */
#define MVSV_MAX_DETECTORS 8
/* The detection table for the ROIs of mvsv_set_mean_rois.  n must equal their count (MVSV_ERR_STATE otherwise: set the
 * ROIs first).  detector_of_roi[i] in [-1, ndet): the detector ROI i belongs to, -1 for a ROI that is not tested.
 * centers_xy[2i], centers_xy[2i+1]: the image_x, image_y calcCoordinate takes for ROI i, in dMapWork coordinates (the
 * map without the dMapROI x offset): Subimage::roi_center, Samplepoint::center.  min_max_distance[2d], [2d+1]: the
 * min_distance / max_distance of detector d in metres (the init() arguments), ndet in [1, MVSV_MAX_DETECTORS].  The
 * disparity range of every (rig, detector) is computed on the host, again whenever a Q or the table changes.
 * mvsv_set_mean_rois and every geometry change (which drops the ROIs) drop the table, and with it the obstacle lists
 * the I/O slots hold.  A compute with MVSV_STAGE_DETECT fails before it takes an I/O slot, with the results of earlier
 * computes still downloadable: MVSV_ERR_INVALID without MVSV_STAGE_MEANS; MVSV_ERR_STATE without a table, with a
 * table whose length no longer matches the ROIs, or when a frame names a rig without Q.
 * Multi-device ctx: repeated on every part, like the other setters.  No reference counterpart (the reference runs the
 * detectors on the CPU, trgt/demo.cpp:271-276). */
int mvsv_set_detection(mvsv_ctx* ctx, const int* detector_of_roi, const float* centers_xy, int n,
                       const float* min_max_distance, int ndet);

/* One pass of the hot path over `batch` stereo pairs held in HOST memory (pair i at base + i*frame_stride).
 * Asynchronous when the host buffers are pinned (mvsv_host_alloc): the copies run on the ctx's copy stream and the
 * call returns at once.  Pageable buffers are accepted too, but the CUDA driver then stages them itself and the call
 * returns only when the input copies have been staged (the ctx keeps no staging buffer of its own).  With
 * MVSV_STAGE_RECTIFY the inputs are raw frames (frame size),
 * otherwise rectified pairs (width x height of mvsv_get_info).  Strides in bytes.  A call that fails before it submits
 * work (arguments, engine state, allocation) leaves the results of earlier calls as they were; one that fails while
 * submitting leaves no results (mvsv_download then returns MVSV_ERR_STATE).  Multi-device ctx: the batch is split
 * across the parts (mvsv_init_devices). */
int mvsv_compute(mvsv_ctx* ctx, const uint8_t* left, size_t lstride, const uint8_t* right, size_t rstride,
                 size_t frame_stride, int batch, unsigned stages);
/* Same, inputs already resident in device memory (used for the HBM-resident bench figure and pipelines
 * that produce frames on the GPU). */
int mvsv_compute_device(mvsv_ctx* ctx, const uint8_t* dleft, size_t lstride, const uint8_t* dright, size_t rstride,
                        size_t frame_stride, int batch, unsigned stages);

/* GPU producers and consumers: ordering against the caller's CUDA stream.
 * `stream` of the three calls below is a cudaStream_t on any device; cudaStreamLegacy and cudaStreamPerThread name the
 * stream of the device current on the calling thread when the call is entered.  NULL means no ordering with the caller.
 * The ctx keeps one event per device of the streams it is given (created on first use, freed by mvsv_destroy).
 *
 * mvsv_compute_device with `stream`: the engine reads the inputs only after the work queued on `stream` before the
 * call, and work queued on `stream` after the call starts once the engine has copied the inputs into its I/O slot (not
 * after the whole compute): the caller may then overwrite or free the inputs on that stream.  The call does not wait on
 * the host.  stream == NULL is exactly mvsv_compute_device, which is this call with NULL.  Multi-device ctx: every part
 * waits for the caller's stream, and the stream waits for the input copies of every part. */
int mvsv_compute_device_stream(mvsv_ctx* ctx, const uint8_t* dleft, size_t lstride, const uint8_t* dright, size_t rstride,
                               size_t frame_stride, int batch, unsigned stages, void* stream);
/* Disparity::tm(Stereopair const&, cv::Mat& output, unsigned kernelSize) (src/disparity.cpp:25-58): for every pixel
 * (i, j), i < rows-kernelSize, j < cols-kernelSize, the kernelSize x kernelSize block of the left image is matched
 * by normalised cross-correlation (cv::matchTemplate TM_CCORR_NORMED) against the right image's blocks at
 * (j + x, i), x in [0, cols-j-kernelSize); out(i, j) = (uint8) x of the first maximum (cv::minMaxLoc), 0 elsewhere.
 * Synchronous: host images in (rectified size of mvsv_get_info, pair b at base + b*frame_stride), `batch` CV_8U
 * maps out (map b at out + b*height*ostride).  The ranking is evaluated in exact integer arithmetic; OpenCV's
 * floating-point scores can order exact ties and last-bit near-ties differently (tests/test_tm.py).
 * Limits: kernelSize in [1, 31], width <= 4096. */
int mvsv_tm(mvsv_ctx* ctx, const uint8_t* left, size_t lstride, const uint8_t* right, size_t rstride,
            size_t frame_stride, int batch, unsigned kernel_size, uint8_t* out, size_t ostride);
/* Copy results of the last compute back to host memory and synchronise.  Any pointer may be NULL.  The number
 * of frames copied is that of the last compute (mvsv_info.last_batch): size the buffers for it.
 *   disp  : batch x height x (dstride bytes per row) int16, CV_16S x16 fixed point, INVALID=(minD-1)*16
 *   rectL/R: batch x height x (rstride bytes) uint8
 *   xyz   : batch x height x width x 3 float (0,0,0 where disparity <= 0)
 *   means : batch x num_rois float */
int mvsv_download(mvsv_ctx* ctx, int16_t* disp, size_t dstride, uint8_t* rectL, uint8_t* rectR, size_t rstride,
                  float* xyz, float* means);
/* Pipelining inside one engine.  With two I/O slots (default: one) consecutive compute calls alternate between two
 * sets of input / result buffers while sharing one set of cost volumes: the host->device copy of call k+1 runs on
 * the copy stream while the kernels of call k execute, and mvsv_download_age(ctx, 1, ...) fetches the results of
 * call k (age 1 = the call before the last one) on a download stream while the kernels of call k+1 execute.  The
 * kernels themselves run in submission order on the ctx stream.  A slot's results must be downloaded before the
 * call after next overwrites them.  No reference counterpart (the reference computes one pair per call on the
 * CPU, src/disparity.cpp:6-10); mvsv_download == age 0. */
int mvsv_set_io_slots(mvsv_ctx* ctx, int n);
int mvsv_download_age(mvsv_ctx* ctx, int age, int16_t* disp, size_t dstride, uint8_t* rectL, uint8_t* rectR, size_t rstride,
                      float* xyz, float* means);
/* The point list of MVSV_STAGE_POINTS (Utility::dmap2pcl, src/utility.cpp:242-262) of the compute in I/O slot `age`
 * (ages as in mvsv_download_age), copied to host memory; synchronous.  Writes offsets[0 .. batch] (batch: frames of
 * that compute): frame f's points are points[3*offsets[f] .. 3*offsets[f+1]), offsets[batch] is the total.  Then
 * copies exactly offsets[batch] points (x, y, z floats each) into `points`, which holds capacity_points points.
 *   points == NULL: only the offsets (the size query).
 *   capacity_points < offsets[batch]: MVSV_ERR_INVALID, with the offsets written and `points` untouched.
 *   the compute did not run MVSV_STAGE_POINTS: MVSV_ERR_STATE.
 * Multi-device ctx: the offsets of every part are fetched first; part k's points then go right after those of the parts
 * before it, with its frame offsets rebased onto them, and the parts' copies run side by side. */
int mvsv_download_points(mvsv_ctx* ctx, int age, int64_t* offsets, float* points, size_t capacity_points);
/* mvsv_download_age into DEVICE memory, for consumers on the GPU.  Same buffers, strides, frames and offsets as
 * mvsv_download_age (disp at disp + first*height*dstride for the frames of each part, XYZ and means likewise; the frames
 * of that slot's compute), on any device: the copies use cudaMemcpyDefault, so that unified addressing finds both ends
 * and copies peer to peer where the devices differ.  No kernel runs: the copy engines move the results.
 *   stream != NULL: the copies start after the work queued on `stream` before the call, work queued on `stream` after
 *     the call sees the results, and the call returns without a host wait.
 *   stream == NULL: the call waits for the copies before it returns, as mvsv_download_age does.
 * Rejected, with the results left downloadable: MVSV_ERR_INVALID for a non-NULL destination that
 * cudaPointerGetAttributes does not report as device or managed memory (host memory: mvsv_download_age); everything
 * mvsv_download_age rejects, with its code (strides below the row, an age outside the slots, nothing computed, a stage
 * the compute did not run).  A failure while the copies of several parts are queued waits for the copies queued before
 * it: no copy into the caller's memory is in flight after an error.
 * Slot lifetime: copies still in flight hold their I/O slot.  A compute (or mvsv_debug_postfilter) that takes the slot
 * writes it only after them, and mvsv_set_io_slots, mvsv_set_mean_rois, a geometry change (maps, rectification, resize)
 * and mvsv_destroy wait for them before they free slot buffers. */
int mvsv_download_device(mvsv_ctx* ctx, int age, int16_t* disp, size_t dstride, uint8_t* rectL, uint8_t* rectR,
                         size_t rstride, float* xyz, float* means, void* stream);
/* mvsv_download_points with the points into DEVICE memory (offsets still to host memory).  The list's size depends on the
 * data, so the frame offsets are fetched to `offsets` first, exactly as mvsv_download_points does (multi-device rebase
 * included): this phase WAITS ON THE HOST until the compute has finished.  The point copies then run as in
 * mvsv_download_device, ordered on `stream`.  points == NULL (the size query), capacity_points too small
 * (MVSV_ERR_INVALID, offsets written, `points` untouched) and MVSV_ERR_STATE are those of mvsv_download_points; a
 * non-NULL `points` that is not device or managed memory is MVSV_ERR_INVALID. */
int mvsv_download_points_device(mvsv_ctx* ctx, int age, int64_t* offsets, float* points, size_t capacity_points,
                                void* stream);
/* The point list of I/O slot `age` entirely in DEVICE memory, with no host wait: a kernel on the engine's download
 * stream writes both the offsets and the points, so the host never needs the list's size.
 *   offsets: device or managed memory, not NULL.  Receives batch + 1 values (batch: frames of that slot's compute),
 *     exactly those mvsv_download_points writes, multi-device rebase included.
 *   points: device or managed memory, or NULL (the offsets only).  Receives points[0 .. min(total, capacity_points)):
 *     the list cut off at the capacity, in list order; nothing past it is written.  The host does not know the total
 *     here, so a short buffer truncates instead of failing.  A consumer detects truncation on the device by
 *     offsets[batch] > capacity_points; every frame f with offsets[f+1] <= capacity_points is complete.
 *   stream != NULL: the writes start after the work queued on `stream` before the call, work queued on `stream` after
 *     the call sees them, and the call never waits on the host (no stream or event synchronisation, no copy to pageable
 *     memory).  stream == NULL: the call waits for its writes before it returns.  cudaStreamLegacy and
 *     cudaStreamPerThread as in mvsv_download_device.
 *   Multi-device ctx: part k's base (the points of the parts before it) is summed on the device from their totals,
 *     which part k's download stream copies from them once their computes are done (cudaMemcpyPeerAsync).  Where a
 *     destination is on another device than a part, the part writes it through peer access, which the call enables
 *     for this process (cudaDeviceEnablePeerAccess) where cudaDeviceCanAccessPeer allows it.
 * Rejected before anything is queued, with earlier results still downloadable: MVSV_ERR_INVALID for a NULL `offsets`,
 * `offsets` or `points` that cudaPointerGetAttributes does not report as device or managed memory, or an age outside
 * the slots; MVSV_ERR_STATE when nothing was computed or the compute did not run MVSV_STAGE_POINTS;
 * MVSV_ERR_UNSUPPORTED for a destination on a device that some part cannot reach by peer access.
 * Slot lifetime as in mvsv_download_device: the writes finish before the slot's pending downloads are, so a compute that
 * takes the slot next, and the setters that free slot buffers, wait for them. */
int mvsv_download_points_stream(mvsv_ctx* ctx, int age, int64_t* offsets, float* points, size_t capacity_points,
                                void* stream);
/* The found obstacles of MVSV_STAGE_DETECT of the compute in I/O slot `age`, copied to host memory; synchronous.  As
 * mvsv_download_points with records for points: offsets[0 .. batch] (frame f's records are out[offsets[f] ..
 * offsets[f+1]), offsets[batch] the total), then exactly offsets[batch] records into `out`, which holds `capacity`.
 *   out == NULL: only the offsets (the size query).
 *   capacity < offsets[batch]: MVSV_ERR_INVALID, with the offsets written and `out` untouched.
 *   the compute did not run MVSV_STAGE_DETECT: MVSV_ERR_STATE.  Ages, the rebase of a multi-device ctx and the other
 *   rejections are those of mvsv_download_points. */
int mvsv_download_obstacles(mvsv_ctx* ctx, int age, int64_t* offsets, mvsv_obstacle* out, size_t capacity);
/* The found obstacles in DEVICE memory with no host wait, as mvsv_download_points_stream gives the point list: offsets
 * (device or managed memory, not NULL) receive the batch + 1 values of mvsv_download_obstacles; out (device or managed
 * memory, or NULL for the offsets only) receives out[0 .. min(total, capacity)), cut off at the capacity, nothing past it;
 * offsets[batch] > capacity tells a consumer on the device that the list was cut.  Ordering on `stream`,
 * stream == NULL, peer access on a multi-device ctx (the parts' totals summed on the device), the slot lifetime and the
 * rejections are those of mvsv_download_points_stream, with MVSV_STAGE_DETECT in place of MVSV_STAGE_POINTS. */
int mvsv_download_obstacles_stream(mvsv_ctx* ctx, int age, int64_t* offsets, mvsv_obstacle* out, size_t capacity,
                                   void* stream);
/* Utility::calcMinMaxDisparity (src/utility.cpp:287-304) of the last computed maps as a GPU reduction: for every
 * frame the smallest and largest disparity value > 0, minmax[2*i], minmax[2*i+1]; (0, 0) when a map has none (the
 * reference dereferences an end iterator there).  Consumed by the PLY writer's grey ramp (src/ply.cpp:62-95). */
int mvsv_download_minmax(mvsv_ctx* ctx, int16_t* minmax);
/* mvsv_download_minmax of I/O slot `age` (ages as in mvsv_download_age) into DEVICE memory: 2 * batch int16 values,
 * minmax[2*i], minmax[2*i+1], (0, 0) for a frame without a value > 0; on a multi-device ctx part k's frames at
 * minmax + 2 * (its first frame).  The reduction runs on the engine's download stream into buffers of the slot, so it
 * never races with mvsv_download_minmax.  Ordering on `stream`, stream == NULL and the slot lifetime are those of
 * mvsv_download_points_stream.  Rejected, with earlier results still downloadable: MVSV_ERR_INVALID for a NULL
 * `minmax` or one that is not device or managed memory, or an age outside the slots; MVSV_ERR_STATE when nothing was
 * computed. */
int mvsv_download_minmax_device(mvsv_ctx* ctx, int age, int16_t* minmax, void* stream);
int mvsv_sync(mvsv_ctx* ctx);

int mvsv_get_info(const mvsv_ctx* ctx, mvsv_info* info);
/* The CUDA stream (cudaStream_t) all work of this ctx is issued on -- for CUDA-event timing by the caller.  NULL for a
 * multi-device ctx, whose parts each have their own (time it with mvsv_timer_start / stop). */
void* mvsv_stream(mvsv_ctx* ctx);
/* Number of kernel launches issued by this ctx since creation (bench.py's gpu_launches). */
unsigned long long mvsv_launch_count(const mvsv_ctx* ctx);

/* CUDA-event timing on the ctx stream (the stream the kernels are launched on).  timer_start/stop bracket a
 * region; profile_enable(1) additionally brackets every kernel launch with events, and profile_read returns the
 * accumulated milliseconds and launch counts per kernel id since the last read (n >= number of kernel ids;
 * returns that number).  mvsv_kernel_name(id) names an id ("" past the end).  While per-kernel timing is enabled the
 * engine launches its kernels one after the other; without it the SGBM cost kernel and the first row scan of
 * different chunks of a batch run side by side on two streams (a little faster, but a kernel's duration then
 * includes its neighbour's). */
int mvsv_timer_start(mvsv_ctx* ctx);
int mvsv_timer_stop(mvsv_ctx* ctx, float* ms);
int mvsv_profile_enable(mvsv_ctx* ctx, int enable);
int mvsv_profile_read(mvsv_ctx* ctx, float* ms, int* counts, int n);
const char* mvsv_kernel_name(int kid);

/* Pinned host memory for zero-staging async copies.  With unified addressing (every 64-bit platform CUDA supports) it
 * counts as pinned on every device, so one buffer serves all parts of a multi-device ctx. */
int mvsv_host_alloc(void** p, size_t bytes);
int mvsv_host_free(void* p);

/* Test hooks: read an internal device buffer of the last compute into host memory.
 * which: 0 = cost volume C, 1 = aggregated S (before the final right-to-left pass), 2 = raw disparity
 * (after LR check, before median; StereoBM with a speckle window: after the LR check, before speckle), 3 = vertical-sum volume, 4 = disparity after median (before speckle),
 * 5 = BM prefiltered left, 6 = BM prefiltered right, 7 / 8 = fixed-point rectification map of camera 0 / 1
 * (roi_h x roi_w int32 pairs: x*32, y*32 rounded).  Returns bytes written or a negative error. */
/* bit 0: keep the complete aggregated S volume (all paths) readable through mvsv_debug_read(which=1).
 * bit 1: never keep a volume as bytes (mvsv_info.sgbm_s8, mvsv_info.bm_col8).
 * bit 2: run the 3x3 median with its one-column-per-lane kernel also where the four-columns-per-lane kernel qualifies
 * (width % 4 == 0).
 * bits 8..15: force the number of column strips per frame of the fused sweep (0xff = force the independent passes,
 * 0xfe = force the sweep with the usual choice of strips: small batches otherwise take the independent passes).
 * bits 16..23: force the number of frames per chunk of the overlapped cost kernel / first row scan (0 = chosen by the
 * engine: about seven chunks per batch, one chunk for small batches). */
/* Environment variables read by the library (diagnostics only): MVSV_SERIAL=1 launches every kernel of a compute
 * one after the other (as per-kernel timing does) -- for profilers, which serialise kernels anyway; MVSV_NO_DSM=1
 * sends the sweep's border records through global memory also where a thread-block cluster would be used. */
int mvsv_debug_set_flags(mvsv_ctx* ctx, unsigned flags);
long long mvsv_debug_read(mvsv_ctx* ctx, int which, void* host, size_t capacity_bytes);
/* Test hook: the post-filters and consumers of a compute, run on caller-supplied disparity maps instead of a matcher's
 * output.  `batch` int16 maps of width x height of mvsv_get_info in HOST memory (row stride `stride` bytes, map b at
 * maps + b*height*stride) become the raw disparity (mvsv_debug_read which=2); then, in the order cv::StereoSGBM applies
 * them, medianBlur(3) when median != 0 and filterSpeckles(newVal, maxSpeckleSize, maxDiff) when maxSpeckleSize > 0
 * (maxDiff in x16 units, as filterSpeckles takes it; neither: a plain copy) leave the final map in the next I/O slot,
 * and `stages` (MVSV_STAGE_XYZ, MVSV_STAGE_POINTS, MVSV_STAGE_MEANS and / or MVSV_STAGE_DETECT with MVSV_STAGE_MEANS
 * only) run on it.  The slot is then read like that of a compute (mvsv_download, mvsv_download_age,
 * mvsv_download_points, mvsv_download_obstacles, mvsv_download_minmax, mvsv_debug_read 2 and 4).  Argument and state
 * checks, and the handling of a failure, are those of mvsv_compute. */
int mvsv_debug_postfilter(mvsv_ctx* ctx, const int16_t* maps, size_t stride, int batch, int median, int newVal,
                          int maxSpeckleSize, int maxDiff, unsigned stages);

#ifdef __cplusplus
}
#endif
#endif /* MVSV_H_ */
