"""ctypes binding of libmvsv.so (C ABI: include/mvsv.h) plus a host-side mirror of the reference's
disparity interface (reference inc/disparity.h:17-35, src/disparity.cpp:6-22,60-108).

No CPU fallback: if the CUDA library is missing or there is no GPU, construction raises.
"""
import contextlib
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmvsv.so")

STAGE_RECTIFY, STAGE_SGBM, STAGE_BM, STAGE_XYZ, STAGE_MEANS, STAGE_POINTS, STAGE_DETECT = 1, 2, 4, 8, 16, 32, 64
MAX_DETECTORS = 8   # MVSV_MAX_DETECTORS
# struct mvsv_obstacle: one found obstacle of STAGE_DETECT (24 bytes)
OBSTACLE_DTYPE = np.dtype([("roi", "<i4"), ("value", "<f4"), ("xyzw", "<f4", (4,))])
CUDA_STREAM_LEGACY = 1      # cudaStreamLegacy: the legacy default stream of the current device


def _torch():
    # imported on first use: the module, its host calls and the CPU tests work without torch
    import torch
    return torch

# every symbol include/mvsv.h declares (tests check the library exports all of them)
ABI_SYMBOLS = (
    "mvsv_init", "mvsv_destroy", "mvsv_last_error", "mvsv_set_sgbm_params", "mvsv_set_bm_params",
    "mvsv_upload_rectify_maps", "mvsv_set_rectification", "mvsv_set_resize", "mvsv_reset_rectification", "mvsv_set_Q", "mvsv_set_mean_rois", "mvsv_compute",
    "mvsv_compute_device", "mvsv_tm", "mvsv_download", "mvsv_sync", "mvsv_get_info", "mvsv_stream", "mvsv_launch_count",
    "mvsv_host_alloc", "mvsv_host_free", "mvsv_debug_set_flags", "mvsv_debug_read",
    "mvsv_download_minmax", "mvsv_download_age", "mvsv_set_io_slots", "mvsv_timer_start", "mvsv_timer_stop", "mvsv_profile_enable", "mvsv_profile_read", "mvsv_kernel_name",
    "mvsv_set_bm_filters", "mvsv_debug_postfilter",
    "mvsv_upload_rectify_maps_rig", "mvsv_set_rectification_rig", "mvsv_set_Q_rig", "mvsv_set_frame_rigs",
    "mvsv_init_devices", "mvsv_get_devices", "mvsv_download_points",
    "mvsv_compute_device_stream", "mvsv_download_device", "mvsv_download_points_device",
    "mvsv_download_points_stream", "mvsv_download_minmax_device",
    "mvsv_set_detection", "mvsv_download_obstacles", "mvsv_download_obstacles_stream",
)
MAX_RIGS = 64       # MVSV_MAX_RIGS


class MvsvError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("mvsv error %d: %s" % (code, msg))
        self.code = code


class SgbmParams(C.Structure):
    """== struct Disparity::sgbmParameters (reference inc/disparity.h:17-27) + P1, P2."""
    _fields_ = [(n, C.c_int) for n in (
        "minDisp", "numDisp", "blockSize", "disp12MaxDiff", "preFilterCap", "uniquenessRatio",
        "speckleWindowSize", "speckleRange", "disparityMode", "P1", "P2")]


class BmParams(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("numDisp", "blockSize", "preFilterCap", "textureThreshold", "uniquenessRatio")]


class Info(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "frame_width", "frame_height", "width", "height", "max_batch", "sgbm_minX1", "sgbm_W1", "sgbm_D",
        "sgbm_Dpad", "sgbm_npaths", "num_rois", "device", "sgbm_td_cluster", "last_batch", "sgbm_s8", "bm_col8")]


_lib = None


def load_library():
    """Load libmvsv.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libmvsv.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "or `make -C mvstereovision3_b200/csrc`); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    vp, sz, ci = C.c_void_p, C.c_size_t, C.c_int
    lib.mvsv_init.argtypes = [ci, ci, ci, ci, C.POINTER(vp)]
    lib.mvsv_init_devices.argtypes = [vp, ci, ci, ci, ci, C.POINTER(vp)]
    lib.mvsv_get_devices.argtypes = [vp, vp, ci]
    lib.mvsv_destroy.argtypes = [vp]
    lib.mvsv_destroy.restype = None
    lib.mvsv_last_error.argtypes = [vp]
    lib.mvsv_last_error.restype = C.c_char_p
    lib.mvsv_set_sgbm_params.argtypes = [vp, C.POINTER(SgbmParams)]
    lib.mvsv_set_bm_params.argtypes = [vp, C.POINTER(BmParams)]
    lib.mvsv_set_bm_filters.argtypes = [vp, ci, ci, ci]
    lib.mvsv_upload_rectify_maps.argtypes = [vp, ci, vp, vp, sz, ci, ci, ci, ci]
    lib.mvsv_set_rectification.argtypes = [vp, ci, vp, vp, ci, vp, vp, ci, ci, ci, ci]
    lib.mvsv_set_resize.argtypes = [vp, C.c_double]
    lib.mvsv_reset_rectification.argtypes = [vp]
    lib.mvsv_set_Q.argtypes = [vp, vp]
    lib.mvsv_upload_rectify_maps_rig.argtypes = [vp, ci, ci, vp, vp, sz, ci, ci, ci, ci]
    lib.mvsv_set_rectification_rig.argtypes = [vp, ci, ci, vp, vp, ci, vp, vp, ci, ci, ci, ci]
    lib.mvsv_set_Q_rig.argtypes = [vp, ci, vp]
    lib.mvsv_set_frame_rigs.argtypes = [vp, vp, ci]
    lib.mvsv_set_mean_rois.argtypes = [vp, vp, ci]
    lib.mvsv_compute.argtypes = [vp, vp, sz, vp, sz, sz, ci, C.c_uint]
    lib.mvsv_compute_device.argtypes = [vp, vp, sz, vp, sz, sz, ci, C.c_uint]
    lib.mvsv_compute_device_stream.argtypes = [vp, vp, sz, vp, sz, sz, ci, C.c_uint, vp]
    lib.mvsv_tm.argtypes = [vp, vp, sz, vp, sz, sz, ci, C.c_uint, vp, sz]
    lib.mvsv_download.argtypes = [vp, vp, sz, vp, vp, sz, vp, vp]
    lib.mvsv_download_age.argtypes = [vp, ci, vp, sz, vp, vp, sz, vp, vp]
    lib.mvsv_download_points.argtypes = [vp, ci, vp, vp, sz]
    lib.mvsv_download_device.argtypes = [vp, ci, vp, sz, vp, vp, sz, vp, vp, vp]
    lib.mvsv_download_points_device.argtypes = [vp, ci, vp, vp, sz, vp]
    lib.mvsv_download_points_stream.argtypes = [vp, ci, vp, vp, sz, vp]
    lib.mvsv_download_minmax_device.argtypes = [vp, ci, vp, vp]
    lib.mvsv_set_detection.argtypes = [vp, vp, vp, ci, vp, ci]
    lib.mvsv_download_obstacles.argtypes = [vp, ci, vp, vp, sz]
    lib.mvsv_download_obstacles_stream.argtypes = [vp, ci, vp, vp, sz, vp]
    lib.mvsv_set_io_slots.argtypes = [vp, ci]
    lib.mvsv_sync.argtypes = [vp]
    lib.mvsv_download_minmax.argtypes = [vp, vp]
    lib.mvsv_get_info.argtypes = [vp, C.POINTER(Info)]
    lib.mvsv_stream.argtypes = [vp]
    lib.mvsv_stream.restype = vp
    lib.mvsv_launch_count.argtypes = [vp]
    lib.mvsv_launch_count.restype = C.c_ulonglong
    lib.mvsv_host_alloc.argtypes = [C.POINTER(vp), sz]
    lib.mvsv_host_free.argtypes = [vp]
    lib.mvsv_debug_set_flags.argtypes = [vp, C.c_uint]
    lib.mvsv_debug_read.argtypes = [vp, ci, vp, sz]
    lib.mvsv_debug_read.restype = C.c_longlong
    lib.mvsv_debug_postfilter.argtypes = [vp, vp, sz, ci, ci, ci, ci, ci, C.c_uint]
    lib.mvsv_timer_start.argtypes = [vp]
    lib.mvsv_timer_stop.argtypes = [vp, C.POINTER(C.c_float)]
    lib.mvsv_profile_enable.argtypes = [vp, ci]
    lib.mvsv_profile_read.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(ci), ci]
    lib.mvsv_kernel_name.argtypes = [ci]
    lib.mvsv_kernel_name.restype = C.c_char_p
    _lib = lib
    return lib


class _Pinned:
    """Page-locked host buffer (mvsv_host_alloc) exposed as a numpy array via .array."""

    def __init__(self, shape, dtype):
        self._lib = load_library()
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        rc = self._lib.mvsv_host_alloc(C.byref(p), max(self.nbytes, 1))
        if rc != 0:
            raise MvsvError(rc, "mvsv_host_alloc failed")
        self.ptr = p.value
        buf = (C.c_uint8 * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def close(self):
        if self.ptr:
            self.array = None
            self._lib.mvsv_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def pinned(shape, dtype):
    return _Pinned(shape, dtype)


class Engine:
    """One mvsv_ctx: one GPU, one stream.  Mirrors the objects a reference driver holds: the
    cv::Ptr<cv::StereoSGBM>/StereoBM matcher (trgt/demo.cpp:190-194) and Stereosystem's rectification state.
    With `devices` (a list of device ids, repeats allowed) the ctx spans several engines (mvsv_init_devices): every batch
    is split into contiguous shares, one per listed device, and `device` is ignored."""

    def __init__(self, frame_width, frame_height, max_batch=1, device=0, devices=None):
        self._lib = load_library()
        self._ctx = C.c_void_p()
        if devices is None:
            rc = self._lib.mvsv_init(device, frame_width, frame_height, max_batch, C.byref(self._ctx))
        else:
            ids = np.ascontiguousarray(devices, np.int32).ravel()
            rc = self._lib.mvsv_init_devices(ids.ctypes.data if ids.size else None, int(ids.size), frame_width, frame_height,
                                             max_batch, C.byref(self._ctx))
        if rc != 0:
            raise MvsvError(rc, self._lib.mvsv_last_error(None).decode())
        self.max_batch = max_batch

    # -- plumbing -------------------------------------------------------------------------------
    def _ck(self, rc):
        if rc < 0:
            raise MvsvError(rc, self._lib.mvsv_last_error(self._ctx).decode())
        return rc

    def close(self):
        if self._ctx:
            self._lib.mvsv_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def info(self):
        i = Info()
        self._ck(self._lib.mvsv_get_info(self._ctx, C.byref(i)))
        return i

    @property
    def devices(self):
        """the device of every part (one entry for an engine of one device)"""
        n = self._ck(self._lib.mvsv_get_devices(self._ctx, None, 0))
        ids = np.zeros(n, np.int32)
        self._ck(self._lib.mvsv_get_devices(self._ctx, ids.ctypes.data, n))
        return [int(v) for v in ids]

    @property
    def stream(self):
        return self._lib.mvsv_stream(self._ctx)

    @property
    def launch_count(self):
        return int(self._lib.mvsv_launch_count(self._ctx))

    # -- parameters -----------------------------------------------------------------------------
    def set_sgbm_params(self, **kw):
        p = SgbmParams(**{k: int(v) for k, v in kw.items()})
        self._ck(self._lib.mvsv_set_sgbm_params(self._ctx, C.byref(p)))

    def set_bm_params(self, **kw):
        p = BmParams(**{k: int(v) for k, v in kw.items()})
        self._ck(self._lib.mvsv_set_bm_params(self._ctx, C.byref(p)))

    def set_bm_filters(self, disp12MaxDiff=-1, speckleWindowSize=0, speckleRange=0):
        """cv::StereoBM::setDisp12MaxDiff / setSpeckleWindowSize / setSpeckleRange, in cv2's units (include/mvsv.h)."""
        self._ck(self._lib.mvsv_set_bm_filters(self._ctx, int(disp12MaxDiff), int(speckleWindowSize), int(speckleRange)))

    def upload_rectify_maps(self, cam, mapx, mapy, roi, rig=0):
        mapx = np.ascontiguousarray(mapx, np.float32)
        mapy = np.ascontiguousarray(mapy, np.float32)
        self._ck(self._lib.mvsv_upload_rectify_maps_rig(self._ctx, int(rig), cam, mapx.ctypes.data, mapy.ctypes.data,
                                                        mapx.strides[0], *[int(v) for v in roi]))

    def set_rectification(self, cam, K, dist, R, P, roi, rig=0):
        """cv::initUndistortRectifyMap on the device (reference src/Stereosystem.cpp:214-217) + mDisplayROI, of rig `rig`."""
        K = np.ascontiguousarray(K, np.float64).reshape(9)
        d = np.ascontiguousarray(np.asarray(dist, np.float64).ravel()) if dist is not None else np.zeros(0)
        R = np.ascontiguousarray(R, np.float64).reshape(9)
        P = np.ascontiguousarray(P, np.float64).reshape(12)
        self._ck(self._lib.mvsv_set_rectification_rig(self._ctx, int(rig), cam, K.ctypes.data, d.ctypes.data if d.size else None,
                                                      int(d.size), R.ctypes.data, P.ctypes.data, *[int(v) for v in roi]))

    def set_frame_rigs(self, rigs):
        """Frame i of every later compute comes from rig rigs[i] (frames past the end: rig 0); len(rigs) <= max_batch."""
        r = np.ascontiguousarray(rigs, np.int32).ravel()
        self._ck(self._lib.mvsv_set_frame_rigs(self._ctx, r.ctypes.data if r.size else None, int(r.size)))

    def read_rectify_map(self, cam, roi):
        """Fixed-point map of one camera as the device holds it: int32 [roi_h, roi_w, 2] = rint(map * 32)."""
        a = np.empty((int(roi[3]), int(roi[2]), 2), np.int32)
        n = self._ck(self._lib.mvsv_debug_read(self._ctx, 7 + cam, a.ctypes.data, a.nbytes))
        assert n == a.nbytes, (n, a.nbytes)
        return a

    def set_resize(self, factor):
        """cv::resize(.., factor, factor) after remap + crop (reference src/Stereosystem.cpp:279-315); 0 = off."""
        self._ck(self._lib.mvsv_set_resize(self._ctx, float(factor)))

    def reset_rectification(self):
        self._ck(self._lib.mvsv_reset_rectification(self._ctx))

    def set_Q(self, Q, rig=0):
        Q = np.ascontiguousarray(Q, np.float32).reshape(16)
        self._ck(self._lib.mvsv_set_Q_rig(self._ctx, int(rig), Q.ctypes.data))

    def set_mean_rois(self, rois):
        r = np.ascontiguousarray(rois, np.int32).reshape(-1, 4)
        self._ck(self._lib.mvsv_set_mean_rois(self._ctx, r.ctypes.data, len(r)))

    def set_detection(self, detector_of_roi, centers, ranges):
        """The detection table of STAGE_DETECT (mvsv_set_detection) for the ROIs of set_mean_rois: detector_of_roi [n]
        (-1: not tested), centers [n, 2] (calcCoordinate's image_x, image_y of each ROI, without the dMapROI x offset),
        ranges [ndet, 2] (each detector's min_distance, max_distance in metres)."""
        d = np.ascontiguousarray(detector_of_roi, np.int32).ravel()
        xy = np.ascontiguousarray(centers, np.float32).reshape(-1, 2)
        rg = np.ascontiguousarray(ranges, np.float32).reshape(-1, 2)
        if len(xy) != len(d):
            raise ValueError("detector_of_roi and centers must have one entry per ROI")
        self._ck(self._lib.mvsv_set_detection(self._ctx, d.ctypes.data if d.size else None, xy.ctypes.data if xy.size else None,
                                              int(d.size), rg.ctypes.data if rg.size else None, len(rg)))

    # -- compute --------------------------------------------------------------------------------
    @staticmethod
    def _batchify(img):
        img = np.asarray(img)
        if img.ndim == 2:
            img = img[None]
        if img.dtype != np.uint8 or img.ndim != 3 or img.strides[2] != 1:
            raise ValueError("images must be uint8 [B,]H,W with unit column stride")
        return img

    def compute(self, left, right, stages):
        """Host images (numpy uint8, [B,]H,W; row stride may exceed W, as for cv::Mat ROI views)."""
        left, right = self._batchify(left), self._batchify(right)
        if left.shape != right.shape:
            raise ValueError("left/right shapes differ")
        if left.strides[0] != right.strides[0] and left.shape[0] > 1:
            raise ValueError("left/right frame strides differ")
        self._ck(self._lib.mvsv_compute(self._ctx, left.ctypes.data, left.strides[1], right.ctypes.data, right.strides[1],
                                        left.strides[0], left.shape[0], stages))
        self._keep = (left, right)

    def compute_device(self, dleft_ptr, lstride, dright_ptr, rstride, frame_stride, batch, stages, stream=None):
        """Inputs in device memory.  `stream` (a torch.cuda.Stream): the inputs are read after the work queued on it, and
        work queued on it afterwards waits only for the input copies (mvsv_compute_device_stream); None: no ordering."""
        self._on_stream(stream, lambda h: self._ck(self._lib.mvsv_compute_device_stream(
            self._ctx, dleft_ptr, lstride, dright_ptr, rstride, frame_stride, batch, stages, h)))

    def compute_tensors(self, left, right, stages, stream=None):
        """uint8 CUDA tensors [B,]H,W with unit column stride; the row and frame strides are the tensors' own."""
        torch = _torch()

        def batchify(t):
            if t.dim() == 2:
                t = t.unsqueeze(0)
            if t.dtype != torch.uint8 or t.dim() != 3 or not t.is_cuda or t.stride(2) != 1:
                raise ValueError("images must be uint8 CUDA tensors [B,]H,W with unit column stride")
            return t
        left, right = batchify(left), batchify(right)
        if left.shape != right.shape:
            raise ValueError("left/right shapes differ")
        if left.stride(0) != right.stride(0) and left.shape[0] > 1:
            raise ValueError("left/right frame strides differ")
        self.compute_device(left.data_ptr(), left.stride(1), right.data_ptr(), right.stride(1), left.stride(0),
                            left.shape[0], stages, stream)

    def _on_stream(self, stream, call):
        """call(handle) with the ABI's `stream` argument for a torch.cuda.Stream or None.  Torch reports its default stream
        as handle 0, which the ABI reads as "no ordering": it goes as cudaStreamLegacy, with the stream's device current."""
        if stream is None:
            return call(None)
        with _torch().cuda.device(stream.device):
            return call(stream.cuda_stream or CUDA_STREAM_LEGACY)

    def _device_out(self, stream, device):
        """the device results are allocated on (default: the first part's), and the context that allocates them on
        `stream`, so that their memory follows that stream's order"""
        torch = _torch()
        dev = torch.device("cuda", self.devices[0]) if device is None else torch.device(device)   # an int is a CUDA ordinal
        return dev, (torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext())

    def tm(self, left, right, kernel_size):
        """Disparity::tm (reference src/disparity.cpp:25-58) on host images [B,]H,W -> uint8 [B,H,W]."""
        left, right = self._batchify(left), self._batchify(right)
        if left.shape != right.shape:
            raise ValueError("left/right shapes differ")
        if left.strides[0] != right.strides[0] and left.shape[0] > 1:
            raise ValueError("left/right frame strides differ")
        out = np.empty(left.shape, np.uint8)
        self._ck(self._lib.mvsv_tm(self._ctx, left.ctypes.data, left.strides[1], right.ctypes.data, right.strides[1],
                                   left.strides[0], left.shape[0], int(kernel_size), out.ctypes.data, out.strides[1]))
        return out

    def sync(self):
        self._ck(self._lib.mvsv_sync(self._ctx))

    def _check_batch(self, batch, i):
        # mvsv_download copies the frames of the last compute, whatever the caller's buffers hold
        if batch != i.last_batch:
            raise ValueError("download(%d): the last compute held %d stereo pairs" % (batch, i.last_batch))

    def set_io_slots(self, n):
        """1 (default) or 2 sets of input/result buffers: with 2, compute k+1 may be submitted before the results of
        compute k are fetched with download(..., age=1); copies and kernels then overlap inside this one engine."""
        self._ck(self._lib.mvsv_set_io_slots(self._ctx, n))

    def download(self, batch, disp=True, rect=False, xyz=False, means=False, out=None, age=0):
        i = self.info
        if age == 0:
            self._check_batch(batch, i)
        H, W = i.height, i.width
        res = {}
        d = (out["disp"] if out and "disp" in out else np.empty((batch, H, W), np.int16)) if disp else None
        rl = np.empty((batch, H, W), np.uint8) if rect else None
        rr = np.empty((batch, H, W), np.uint8) if rect else None
        xz = np.empty((batch, H, W, 3), np.float32) if xyz else None
        mn = np.empty((batch, i.num_rois), np.float32) if means else None
        self._ck(self._lib.mvsv_download_age(self._ctx, age, d.ctypes.data if disp else None, W * 2,
                                         rl.ctypes.data if rect else None, rr.ctypes.data if rect else None, W,
                                         xz.ctypes.data if xyz else None, mn.ctypes.data if means else None))
        if disp:
            res["disp"] = d
        if rect:
            res["rectL"], res["rectR"] = rl, rr
        if xyz:
            res["xyz"] = xz
        if means:
            res["means"] = mn
        return res

    def download_points(self, batch, age=0, out=None):
        """The point list of STAGE_POINTS (Utility::dmap2pcl, reference src/utility.cpp:242-262) of the compute `age`
        calls back: (offsets int64 [batch + 1], points float32 [n, 3]); frame f's points are
        points[offsets[f]:offsets[f + 1]].  `out`: a float32 array (e.g. api.pinned((cap, 3), np.float32).array) the
        points are copied into, so that a pipelined loop allocates nothing per step; the points returned are a view of it.
        Without `out` the list is sized by a first call that fetches only the offsets."""
        i = self.info
        if age == 0:
            self._check_batch(batch, i)
        offs = np.empty(i.max_batch + 1, np.int64)         # the C call writes the compute's frames + 1 entries
        if out is None:
            self._ck(self._lib.mvsv_download_points(self._ctx, age, offs.ctypes.data, None, 0))
            out = np.empty((int(offs[batch]), 3), np.float32)
        elif out.dtype != np.float32 or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous float32 array")
        self._ck(self._lib.mvsv_download_points(self._ctx, age, offs.ctypes.data, out.ctypes.data, out.size // 3))
        return offs[:batch + 1], out.reshape(-1)[:3 * int(offs[batch])].reshape(-1, 3)

    def download_device(self, batch, disp=True, rect=False, xyz=False, means=False, out=None, age=0, stream=None,
                        device=None):
        """The results of download() as torch tensors in device memory (mvsv_download_device): disp int16 [batch, H, W],
        rectL / rectR uint8 [batch, H, W], xyz float32 [batch, H, W, 3], means float32 [batch, num_rois].  They are
        allocated on `device` (default: the engine's first device), or taken from `out` (a dict with those keys): disp and
        rect may be pitched views (unit column stride, frame stride = H * row stride), xyz and means are contiguous.
        `stream` (a torch.cuda.Stream): the copies are ordered on it and the call returns without waiting; None: the call
        returns with the copies done."""
        torch = _torch()
        i = self.info
        if age == 0:
            self._check_batch(batch, i)
        H, W = i.height, i.width
        dev, on_stream = self._device_out(stream, device)
        out = out or {}
        spec = (("disp", disp, (batch, H, W), torch.int16, True), ("rectL", rect, (batch, H, W), torch.uint8, True),
                ("rectR", rect, (batch, H, W), torch.uint8, True), ("xyz", xyz, (batch, H, W, 3), torch.float32, False),
                ("means", means, (batch, i.num_rois), torch.float32, False))
        res = {}
        with on_stream:
            for key, on, shape, dtype, pitched in spec:
                if not on:
                    continue
                t = out.get(key)
                if t is None:
                    t = torch.empty(shape, dtype=dtype, device=dev)
                elif t.dtype != dtype or tuple(t.shape) != shape or not t.is_cuda:
                    raise ValueError("out[%r] must be a %s CUDA tensor of shape %s" % (key, dtype, shape))
                elif (t.stride(-1) != 1 or t.stride(0) != H * t.stride(1)) if pitched else not t.is_contiguous():
                    raise ValueError("out[%r]: %s" % (key, "unit column stride and frame stride = H * row stride" if pitched
                                                      else "must be contiguous"))
                res[key] = t
        if rect and res["rectL"].stride(1) != res["rectR"].stride(1):
            raise ValueError("rectL and rectR must share one row stride")

        def ptr(key):
            return res[key].data_ptr() if key in res else None
        dstride = res["disp"].stride(1) * 2 if disp else 0
        rstride = res["rectL"].stride(1) if rect else 0
        self._on_stream(stream, lambda h: self._ck(self._lib.mvsv_download_device(
            self._ctx, age, ptr("disp"), dstride, ptr("rectL"), ptr("rectR"), rstride, ptr("xyz"), ptr("means"), h)))
        return res

    def download_points_device(self, batch, age=0, out=None, stream=None, device=None):
        """The point list of download_points() with the points in device memory (mvsv_download_points_device):
        (offsets int64 numpy [batch + 1], points float32 tensor [n, 3]).  Fetching the offsets waits on the host for the
        compute; the point copy is then ordered on `stream` as in download_device.  `out`: a contiguous float32 CUDA
        tensor the points are copied into (the points returned are a view of it); without it the list is allocated on
        `device` (default: the engine's first device), sized by a first call that fetches only the offsets."""
        torch = _torch()
        i = self.info
        if age == 0:
            self._check_batch(batch, i)
        offs = np.empty(i.max_batch + 1, np.int64)         # the C call writes the compute's frames + 1 entries
        if out is None:
            self._ck(self._lib.mvsv_download_points_device(self._ctx, age, offs.ctypes.data, None, 0, None))
            dev, on_stream = self._device_out(stream, device)
            with on_stream:
                out = torch.empty((int(offs[batch]), 3), dtype=torch.float32, device=dev)
        elif out.dtype != torch.float32 or not out.is_cuda or not out.is_contiguous():
            raise ValueError("out must be a contiguous float32 CUDA tensor")
        self._on_stream(stream, lambda h: self._ck(self._lib.mvsv_download_points_device(
            self._ctx, age, offs.ctypes.data, out.data_ptr() or None, out.numel() // 3, h)))
        return offs[:batch + 1], out.view(-1)[:3 * int(offs[batch])].view(-1, 3)

    def download_points_stream(self, batch, age=0, out=None, stream=None, device=None):
        """The point list of download_points() entirely in device memory, with no host wait (mvsv_download_points_stream):
        (offsets int64 tensor [batch + 1], points float32 tensor [capacity, 3]); frame f's points are
        points[offsets[f]:offsets[f + 1]].  Without `out` both are allocated on `device` (default: the engine's first
        device) with capacity batch * H * W, every pixel, so the list is never cut off.  `out`: (offsets, points)
        contiguous CUDA tensors; points past its capacity are not written, and offsets[batch] > capacity tells so.
        `stream` (a torch.cuda.Stream): the writes are ordered on it; None: the call returns with them done."""
        torch = _torch()
        i = self.info
        if age == 0:
            self._check_batch(batch, i)
        if out is None:
            dev, on_stream = self._device_out(stream, device)
            with on_stream:
                offs = torch.empty(batch + 1, dtype=torch.int64, device=dev)
                pts = torch.empty((batch * i.height * i.width, 3), dtype=torch.float32, device=dev)
        else:
            offs, pts = out
            if offs.dtype != torch.int64 or tuple(offs.shape) != (batch + 1,) or not offs.is_cuda or not offs.is_contiguous():
                raise ValueError("out[0] must be a contiguous int64 CUDA tensor of shape (%d,)" % (batch + 1))
            if pts.dtype != torch.float32 or pts.dim() != 2 or pts.shape[1] != 3 or not pts.is_cuda or not pts.is_contiguous():
                raise ValueError("out[1] must be a contiguous float32 CUDA tensor [capacity, 3]")
        self._on_stream(stream, lambda h: self._ck(self._lib.mvsv_download_points_stream(
            self._ctx, age, offs.data_ptr(), pts.data_ptr() if pts.numel() else None, pts.shape[0], h)))
        return offs, pts

    def download_obstacles(self, batch, age=0):
        """The found obstacles of STAGE_DETECT of the compute `age` calls back (mvsv_download_obstacles): (offsets int64
        [batch + 1], records [n] of OBSTACLE_DTYPE: roi, value, xyzw); frame f's records are records[offsets[f]:offsets[f + 1]],
        in ascending ROI order."""
        i = self.info
        if age == 0:
            self._check_batch(batch, i)
        offs = np.empty(i.max_batch + 1, np.int64)         # the C call writes the compute's frames + 1 entries
        self._ck(self._lib.mvsv_download_obstacles(self._ctx, age, offs.ctypes.data, None, 0))
        out = np.empty(int(offs[batch]), OBSTACLE_DTYPE)
        self._ck(self._lib.mvsv_download_obstacles(self._ctx, age, offs.ctypes.data, out.ctypes.data if out.size else None,
                                                   out.size))
        return offs[:batch + 1], out

    def download_obstacles_stream(self, batch, age=0, out=None, stream=None, device=None):
        """The found obstacles of download_obstacles() entirely in device memory, with no host wait
        (mvsv_download_obstacles_stream): (offsets int64 tensor [batch + 1], records float32 tensor [capacity, 6]), a
        record being roi (int32 bits: records.view(torch.int32)[:, 0]), value, x, y, z, w.  Without `out` both are
        allocated on `device` (default: the engine's first device) with capacity batch * num_rois, so the list is never cut
        off.  `out`: (offsets, records) contiguous CUDA tensors; records past its capacity are not written, and
        offsets[batch] > capacity tells so.  `stream` as in download_points_stream."""
        torch = _torch()
        i = self.info
        if age == 0:
            self._check_batch(batch, i)
        if out is None:
            dev, on_stream = self._device_out(stream, device)
            with on_stream:
                offs = torch.empty(batch + 1, dtype=torch.int64, device=dev)
                rec = torch.empty((batch * i.num_rois, 6), dtype=torch.float32, device=dev)
        else:
            offs, rec = out
            if offs.dtype != torch.int64 or tuple(offs.shape) != (batch + 1,) or not offs.is_cuda or not offs.is_contiguous():
                raise ValueError("out[0] must be a contiguous int64 CUDA tensor of shape (%d,)" % (batch + 1))
            if rec.dtype != torch.float32 or rec.dim() != 2 or rec.shape[1] != 6 or not rec.is_cuda or not rec.is_contiguous():
                raise ValueError("out[1] must be a contiguous float32 CUDA tensor [capacity, 6]")
        self._on_stream(stream, lambda h: self._ck(self._lib.mvsv_download_obstacles_stream(
            self._ctx, age, offs.data_ptr(), rec.data_ptr() if rec.numel() else None, rec.shape[0], h)))
        return offs, rec

    def download_minmax_device(self, batch, age=0, out=None, stream=None, device=None):
        """download_minmax() of the compute `age` calls back as an int16 CUDA tensor [batch, 2]
        (mvsv_download_minmax_device), allocated on `device` (default: the engine's first device) or taken from `out`
        (contiguous); ordered on `stream` as in download_points_stream."""
        torch = _torch()
        i = self.info
        if age == 0:
            self._check_batch(batch, i)
        if out is None:
            dev, on_stream = self._device_out(stream, device)
            with on_stream:
                out = torch.empty((batch, 2), dtype=torch.int16, device=dev)
        elif out.dtype != torch.int16 or tuple(out.shape) != (batch, 2) or not out.is_cuda or not out.is_contiguous():
            raise ValueError("out must be a contiguous int16 CUDA tensor of shape (%d, 2)" % batch)
        self._on_stream(stream, lambda h: self._ck(self._lib.mvsv_download_minmax_device(self._ctx, age, out.data_ptr(), h)))
        return out

    def download_minmax(self, batch):
        """Utility::calcMinMaxDisparity (reference src/utility.cpp:287-304) per frame, reduced on the GPU."""
        self._check_batch(batch, self.info)
        mm = np.empty((batch, 2), np.int16)
        self._ck(self._lib.mvsv_download_minmax(self._ctx, mm.ctypes.data))
        return mm

    # -- timing ---------------------------------------------------------------------------------
    def timer_start(self):
        self._ck(self._lib.mvsv_timer_start(self._ctx))

    def timer_stop(self):
        ms = C.c_float()
        self._ck(self._lib.mvsv_timer_stop(self._ctx, C.byref(ms)))
        return ms.value

    def profile_enable(self, on=True):
        self._ck(self._lib.mvsv_profile_enable(self._ctx, 1 if on else 0))

    def profile_read(self):
        """{kernel name: (total ms, launches)} since the last read (CUDA events on the ctx stream)."""
        n = 64
        ms = (C.c_float * n)()
        cnt = (C.c_int * n)()
        k = self._ck(self._lib.mvsv_profile_read(self._ctx, ms, cnt, n))
        return {self._lib.mvsv_kernel_name(i).decode(): (ms[i], cnt[i]) for i in range(k) if cnt[i]}

    # -- test hooks -----------------------------------------------------------------------------
    def debug_set_flags(self, flags):
        self._ck(self._lib.mvsv_debug_set_flags(self._ctx, flags))

    def debug_postfilter(self, maps, median=True, new_val=0, speckle_size=0, speckle_diff=0, stages=0):
        """mvsv_debug_postfilter: int16 maps [B,]H,W (row stride may exceed W) through medianBlur(3) when `median`, then
        filterSpeckles(new_val, speckle_size, speckle_diff) when speckle_size > 0, then `stages` (STAGE_XYZ |
        STAGE_POINTS | STAGE_MEANS | STAGE_DETECT); the results are fetched with download / download_minmax / debug_read like those of a compute."""
        m = np.asarray(maps)
        if m.ndim == 2:
            m = m[None]
        if m.dtype != np.int16 or m.ndim != 3:
            raise ValueError("maps must be int16 [B,]H,W")
        if m.strides[2] != 2 or m.strides[0] != m.shape[1] * m.strides[1]:
            m = np.ascontiguousarray(m)
        self._ck(self._lib.mvsv_debug_postfilter(self._ctx, m.ctypes.data, m.strides[1], m.shape[0], 1 if median else 0,
                                                 int(new_val), int(speckle_size), int(speckle_diff), stages))

    def debug_read(self, which, batch):
        i = self.info
        H, W = i.height, i.width
        if which in (0, 1, 3):
            a = np.empty((batch, H, i.sgbm_W1, i.sgbm_Dpad), np.int16)
        elif which in (2, 4):
            a = np.empty((batch, H, W), np.int16)
        else:
            pitch = (W + 15) // 16 * 16
            a = np.empty((batch, H, pitch), np.uint8)
        n = self._ck(self._lib.mvsv_debug_read(self._ctx, which, a.ctypes.data, a.nbytes))
        assert n == a.nbytes, (n, a.nbytes)
        if which in (0, 1, 3):
            return a[..., :i.sgbm_D]
        if which in (5, 6):
            return a[..., :W]
        return a


# ---------------------------------------------------------------------------------------------------
# Host-side mirror of the reference's disparity.h interface (same names, argument meaning, error behaviour)
# ---------------------------------------------------------------------------------------------------
class Stereopair:
    """reference inc/utility.h:31-41: carrier of the (rectified) pair, CV_8UC1."""

    def __init__(self, left=None, right=None):
        self.mLeft, self.mRight = left, right


SGBM_YAML_KEYS = ("minDisp", "numDisp", "blockSize", "disp12MaxDiff", "preFilterCap", "uniquenessRatio",
                  "speckleWindowSize", "speckleWindowRange", "mode")


def _read_flat_yaml(filename):
    """OpenCV FileStorage '%YAML:1.0' file holding flat `key: int` pairs (reference configs/*.yml)."""
    out = {}
    with open(filename, "r") as f:
        for line in f:
            line = line.split("#", 1)[0].strip()
            if not line or line.startswith("%") or line == "---" or ":" not in line:
                continue
            k, v = line.split(":", 1)
            v = v.strip()
            try:
                out[k.strip()] = int(float(v))
            except ValueError:
                out[k.strip()] = v
    return out


def loadSGBMParameters(filename, engine, para):
    """Mirror of Disparity::loadSGBMParameters (reference src/disparity.cpp:60-108).

    Fills the dict `para` (the sgbmParameters struct) and drives the engine's setters; P1/P2 are never set
    (they stay 0 -> OpenCV's 2/5).  Returns False (and leaves the engine untouched) when the file cannot be
    opened or one of numDisp/blockSize/speckleWindowSize/speckleWindowRange is missing, like the reference.
    """
    try:
        fs = _read_flat_yaml(filename)
    except OSError:
        return False
    for need in ("numDisp", "blockSize", "speckleWindowSize", "speckleWindowRange"):
        if need not in fs:
            return False
    # cv::FileNode >> int of a missing node yields 0
    para["minDisp"] = fs.get("minDisp", 0)
    para["numDisp"] = fs["numDisp"]
    para["blockSize"] = fs["blockSize"]
    para["disp12MaxDiff"] = fs.get("disp12MaxDiff", 0)
    para["preFilterCap"] = fs.get("preFilterCap", 0)
    para["uniquenessRatio"] = fs.get("uniquenessRatio", 0)
    para["speckleWindowSize"] = fs["speckleWindowSize"]
    para["speckleRange"] = fs["speckleWindowRange"]
    para["disparityMode"] = fs.get("mode", 0)
    engine.set_sgbm_params(**para)
    return True


def loadBMParameters(filename, engine, para):
    """configs/bm.yml has no loader in the reference (SURVEY.md section 2 row 4); this one reads its keys the
    way trgt/disparityTest.cpp drives cv::StereoBM (numDisp, blockSize + setters); preFilterSize is ignored by
    PREFILTER_XSOBEL.  The optional keys disp12MaxDiff, speckleWindowSize and speckleRange, when present, set the
    post-filters (cv::StereoBM's defaults -1 / 0 / 0 for the ones left out)."""
    try:
        fs = _read_flat_yaml(filename)
    except OSError:
        return False
    if "numDisp" not in fs or "blockSize" not in fs:
        return False
    para.update(numDisp=fs["numDisp"], blockSize=fs["blockSize"], preFilterCap=fs.get("preFilterCap", 31),
                textureThreshold=fs.get("textureThreshold", 10), uniquenessRatio=fs.get("uniquenessRatio", 15))
    engine.set_bm_params(**para)
    if any(k in fs for k in ("disp12MaxDiff", "speckleWindowSize", "speckleRange")):
        engine.set_bm_filters(fs.get("disp12MaxDiff", -1), fs.get("speckleWindowSize", 0), fs.get("speckleRange", 0))
    return True


def sgbm(inputImages, engine):
    """Mirror of Disparity::sgbm (reference src/disparity.cpp:6-10): returns the CV_16S map (x16 fixed point)."""
    engine.compute(inputImages.mLeft, inputImages.mRight, STAGE_SGBM)
    return engine.download(1)["disp"][0]


def bm(inputImages, engine):
    """Mirror of Disparity::bm (reference src/disparity.cpp:18-22)."""
    engine.compute(inputImages.mLeft, inputImages.mRight, STAGE_BM)
    return engine.download(1)["disp"][0]


def tm(inputImages, engine, kernelSize):
    """Mirror of Disparity::tm (reference src/disparity.cpp:25-58): CV_8U map, same size as the inputs."""
    return engine.tm(inputImages.mLeft, inputImages.mRight, kernelSize)[0]


def subimage_rois(cols, rows, x_offset=0):
    """The 81 Subimage rectangles of MeanDisparityDetection::init (reference src/MeanDisparityDetection.cpp:80-93),
    for a dMapWork view of cols x rows that starts x_offset columns into the raw map (trgt/demo.cpp:87-113)."""
    dx, dy = cols // 9, rows // 9
    return [(x_offset + c * dx, r * dy, dx, dy) for r in range(9) for c in range(9)]


def samplepoint_rois(cols, rows, x_offset=0, radius=2):
    """5x5 Samplepoint windows of SamplepointDetection::init (reference src/SamplePointDetection.cpp:38-47;
    column-major order c then r, window = [c-radius, c+radius] x [r-radius, r+radius], inc/Samplepoint.h:24-28)."""
    nx, ny = cols // 8, rows // 8
    out = []
    for c in range(1, nx):
        for r in range(1, ny):
            cx, cy = c * (cols // nx), r * (rows // ny)
            out.append((x_offset + cx - radius, cy - radius, 2 * radius + 1, 2 * radius + 1))
    return out


def dmap_roi_offset(num_disp, cols):
    """pixelShift of createDMapROIS (reference trgt/demo.cpp:87-101), including its odd-value adjustment."""
    shift = num_disp // 2
    if shift % 2 == 1:
        shift += 1
        if (cols - shift) % 8 != 0:
            shift = shift + (cols - shift % 8)
    return shift
