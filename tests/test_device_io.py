"""Results in device memory, ordered on the caller's CUDA stream: mvsv_compute_device_stream, mvsv_download_device and
mvsv_download_points_device (Engine.compute_tensors / compute_device(stream=), download_device, download_points_device).

The device downloads must give what the host downloads give, bit for bit (XYZ included: it is the same buffer), into
pitched destinations too.  The ordering tests delay the caller's stream (torch.cuda._sleep) or the engine's, so that a
missing wait shows up every time instead of sometimes."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import test_devices as td
from mvstereovision3_b200 import api

ERR_INVALID, ERR_STATE = -1, -4
FW, FH = td.FW, td.FH
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SLEEP = 40_000_000            # torch.cuda._sleep cycles: about 20 ms, far longer than a compute of these sizes
SENT16, SENT8 = 0x5A5A, 0xA5  # sentinels of the pitched destinations' padding


# ---- CPU side --------------------------------------------------------------------------------------------------------
def test_api_imports_without_torch():
    code = ("import sys; sys.modules['torch'] = None\n"          # `import torch` now raises ImportError
            "from mvstereovision3_b200 import api\n"
            "assert {'mvsv_compute_device_stream', 'mvsv_download_device', 'mvsv_download_points_device'} <= "
            "set(api.ABI_SYMBOLS)\n"
            "assert api.CUDA_STREAM_LEGACY == 1\n")
    subprocess.check_call([sys.executable, "-c", code], cwd=ROOT)


def test_new_prototypes_declared():
    lib = api.load_library()
    vp, sz, ci = C.c_void_p, C.c_size_t, C.c_int
    assert lib.mvsv_compute_device_stream.argtypes == [vp, vp, sz, vp, sz, sz, ci, C.c_uint, vp]
    assert lib.mvsv_download_device.argtypes == [vp, ci, vp, sz, vp, vp, sz, vp, vp, vp]
    assert lib.mvsv_download_points_device.argtypes == [vp, ci, vp, vp, sz, vp]
    with open(os.path.join(ROOT, "include", "mvsv.h")) as f:
        header = f.read()
    for name in ("mvsv_compute_device_stream", "mvsv_download_device", "mvsv_download_points_device"):
        assert "int %s(" % name in header


# ---- helpers ---------------------------------------------------------------------------------------------------------
def _torch():
    return pytest.importorskip("torch")


def workload(e, name, B):
    """the test_devices.py workloads; "points": its three-rig pipeline plus MVSV_STAGE_POINTS"""
    stages, want = td.setup(e, "pipeline" if name == "points" else name, B)
    if name == "points":
        stages |= api.STAGE_POINTS
    return stages, want


def to_dev(a, dev=0):
    return _torch().from_numpy(np.ascontiguousarray(a)).cuda(dev)


def host(res):
    return {k: v.cpu().numpy() for k, v in res.items()}


def same(got, ref, what):
    td.assert_same(host(got) if any(hasattr(v, "cpu") for v in got.values()) else got, ref, what)


def pitched(B, H, W, rect):
    """pitched destinations filled with sentinels: disp row stride 2W + 64 bytes, rect row stride W + 32"""
    torch = _torch()
    d = torch.full((B, H, W + 32), SENT16, dtype=torch.int16, device="cuda:0")
    out = {"disp": d[:, :, :W]}
    bufs = [d]
    if rect:
        for k in ("rectL", "rectR"):
            r = torch.full((B, H, W + 32), SENT8, dtype=torch.uint8, device="cuda:0")
            out[k] = r[:, :, :W]
            bufs.append(r)
    return out, bufs


def padding_intact(bufs, W):
    for b in bufs:
        pad = b[:, :, W:].cpu().numpy()
        assert (pad == (SENT16 if b.element_size() == 2 else SENT8)).all(), "padding written"


def streams(kind):
    torch = _torch()
    return torch.cuda.default_stream() if kind == "default" else torch.cuda.Stream()


# ---- 1. equality with the host download ------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sgbm", "bm", "points"])
@pytest.mark.parametrize("kind", ["none", "side", "default"])
def test_equals_host_download(name, kind):
    torch = _torch()
    B = 10
    L, R = td.frames(B, seed=3)
    with api.Engine(FW, FH, max_batch=B) as e:
        stages, want = workload(e, name, B)
        e.compute(L, R, stages)
        ref = e.download(B, **want)
        s = None if kind == "none" else streams(kind)
        got = e.download_device(B, stream=s, **want)
        out, bufs = pitched(B, e.info.height, e.info.width, want.get("rect", False))
        got_p = e.download_device(B, out=out, stream=s, **want)
        if s is not None:
            s.synchronize()
        assert got["disp"].dtype == torch.int16 and got["disp"].device == torch.device("cuda", 0)
        assert tuple(got["disp"].shape) == (B, e.info.height, e.info.width)
        same(got, ref, name)
        same(got_p, {k: ref[k] for k in got_p}, name + " pitched")
        assert got_p["disp"].data_ptr() == out["disp"].data_ptr()
        padding_intact(bufs, e.info.width)
        if name == "points":
            offs, pts = e.download_points(B)
            offs_d, pts_d = e.download_points_device(B, stream=s)
            if s is not None:
                s.synchronize()
            assert np.array_equal(offs, offs_d) and pts_d.dtype == torch.float32 and tuple(pts_d.shape) == pts.shape
            assert np.array_equal(pts_d.cpu().numpy().view(np.uint8), pts.view(np.uint8))
            # into a preallocated tensor with room to spare: the rest keeps its sentinel
            buf = torch.full((len(pts) + 5, 3), -7.0, device="cuda:0")
            offs_o, pts_o = e.download_points_device(B, out=buf, stream=s)
            if s is not None:
                s.synchronize()
            assert pts_o.data_ptr() == buf.data_ptr() and np.array_equal(offs_o, offs)
            assert np.array_equal(pts_o.cpu().numpy().view(np.uint8), pts.view(np.uint8))
            assert (buf[len(pts):] == -7.0).all()


# ---- 2. pipelined loop -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sgbm", "points"])
def test_pipelined_loop(name):
    """two I/O slots, device inputs, compute k+1 and the age-1 download of k on one stream, no host wait in the loop"""
    torch = _torch()
    B, N = 6, 7
    inputs = [td.frames(B, seed=100 + 10 * k) for k in range(N)]
    with api.Engine(FW, FH, max_batch=B) as e, api.Engine(FW, FH, max_batch=B) as ref:
        stages, want = workload(e, name, B)
        workload(ref, name, B)
        want_ref = []
        for L, R in inputs:
            ref.compute(L, R, stages)
            want_ref.append(ref.download(B, **want))
        dev_in = [(to_dev(L), to_dev(R)) for L, R in inputs]
        torch.cuda.synchronize()
        e.set_io_slots(2)
        s = torch.cuda.Stream()
        got = []
        with torch.cuda.stream(s):
            e.compute_tensors(*dev_in[0], stages, stream=s)
            for k in range(1, N):
                e.compute_tensors(*dev_in[k], stages, stream=s)
                got.append(e.download_device(B, age=1, stream=s, **want))
            got.append(e.download_device(B, age=0, stream=s, **want))
        s.synchronize()
        for k in range(N):
            same(got[k], want_ref[k], "%s step %d" % (name, k))


# ---- 3. ordering, made deterministic ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["side", "default"])
def test_compute_reads_inputs_after_the_producer(kind):
    torch = _torch()
    B = 8
    L0, R0 = td.frames(B, seed=200)
    L1, R1 = td.frames(B, seed=300)
    with api.Engine(FW, FH, max_batch=B) as e, api.Engine(FW, FH, max_batch=B) as ref:
        stages, want = workload(e, "sgbm", B)
        workload(ref, "sgbm", B)
        ref.compute(L1, R1, stages)
        want1 = ref.download(B)
        dl, dr = to_dev(L0), to_dev(R0)
        new_l, new_r = to_dev(L1), to_dev(R1)
        torch.cuda.synchronize()
        s = streams(kind)
        with torch.cuda.stream(s):
            torch.cuda._sleep(SLEEP)
            dl.copy_(new_l)
            dr.copy_(new_r)
            e.compute_tensors(dl, dr, stages, stream=s)
        same(e.download(B), want1, "inputs written by the producer after a delay")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["side", "default"])
def test_caller_may_overwrite_inputs_after_compute(kind):
    """the engine is held back (a compute behind a delayed stream): the caller's overwrite must wait for the input copy"""
    torch = _torch()
    B = 8
    L0, R0 = td.frames(B, seed=210)
    L1, R1 = td.frames(B, seed=310)
    with api.Engine(FW, FH, max_batch=B) as e, api.Engine(FW, FH, max_batch=B) as ref:
        stages, want = workload(e, "sgbm", B)
        workload(ref, "sgbm", B)
        ref.compute(L0, R0, stages)
        want0 = ref.download(B)
        dl, dr = to_dev(L0), to_dev(R0)
        hold_l, hold_r = to_dev(L1), to_dev(R1)
        torch.cuda.synchronize()
        slow = torch.cuda.Stream()
        with torch.cuda.stream(slow):
            torch.cuda._sleep(SLEEP)
        e.compute_tensors(hold_l, hold_r, stages, stream=slow)         # the engine's stream now waits for `slow`
        s = streams(kind)
        with torch.cuda.stream(s):
            e.compute_tensors(dl, dr, stages, stream=s)
            dl.fill_(0)
            dr.fill_(255)
        s.synchronize()
        same(e.download(B), want0, "inputs overwritten on the caller's stream after the call")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["side", "default"])
def test_delayed_download_holds_the_slot(kind):
    """one I/O slot: a compute submitted at once after a delayed device download writes the slot only after the copy"""
    torch = _torch()
    B = 8
    L0, R0 = td.frames(B, seed=220)
    L1, R1 = td.frames(B, seed=320)
    with api.Engine(FW, FH, max_batch=B) as e, api.Engine(FW, FH, max_batch=B) as ref:
        stages, want = workload(e, "points", B)
        workload(ref, "points", B)
        refs = []
        for L, R in ((L0, R0), (L1, R1)):
            ref.compute(L, R, stages)
            refs.append((ref.download(B, **want), ref.download_points(B)))
        e.compute(L0, R0, stages)
        e.sync()
        s = streams(kind)
        with torch.cuda.stream(s):
            torch.cuda._sleep(SLEEP)
            got = e.download_device(B, stream=s, **want)
        e.compute(L1, R1, stages)                                        # the same (only) slot
        s.synchronize()
        same(got, refs[0][0], "delayed download")
        same(e.download(B, **want), refs[1][0], "the compute after it")
        # the points: offsets on the host first, then the copy behind the delay
        e.compute(L0, R0, stages)
        with torch.cuda.stream(s):
            torch.cuda._sleep(SLEEP)
            offs, pts = e.download_points_device(B, stream=s)
        e.compute(L1, R1, stages)
        s.synchronize()
        assert np.array_equal(offs, refs[0][1][0])
        assert np.array_equal(pts.cpu().numpy().view(np.uint8), refs[0][1][1].view(np.uint8))
        offs1, pts1 = e.download_points(B)
        assert np.array_equal(offs1, refs[1][1][0]) and np.array_equal(pts1.view(np.uint8), refs[1][1][1].view(np.uint8))


@pytest.mark.gpu
@pytest.mark.parametrize("setter", ["io_slots", "mean_rois", "resize"])
def test_setters_wait_for_pending_downloads(setter):
    """set_io_slots, set_mean_rois and set_resize free slot buffers: they wait for a device download still in flight"""
    torch = _torch()
    B = 8
    L, R = td.frames(B, seed=230)
    with api.Engine(FW, FH, max_batch=B) as e, api.Engine(FW, FH, max_batch=B) as ref:
        stages, want = workload(e, "pipeline", B)
        workload(ref, "pipeline", B)
        ref.compute(L, R, stages)
        want0 = ref.download(B, **want)
        e.compute(L, R, stages)
        e.sync()
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            torch.cuda._sleep(SLEEP)
            got = e.download_device(B, stream=s, **want)

        def change(eng):
            if setter == "io_slots":
                eng.set_io_slots(2)
            elif setter == "mean_rois":
                eng.set_mean_rois(api.subimage_rois(eng.info.width, eng.info.height))
            else:
                eng.set_resize(0.5)
                eng.set_mean_rois(api.subimage_rois(eng.info.width, eng.info.height))
        change(e)
        s.synchronize()
        same(got, want0, "download pending across set_%s" % setter)
        change(ref)
        for k in range(2):
            ref.compute(L, R, stages)
            e.compute(L, R, stages)
            same(e.download_device(B, **want), ref.download(B, **want), "compute %d after set_%s" % (k, setter))


# ---- 4. stream=None --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_no_stream_returns_with_the_copies_done():
    """the compute is held back behind a delayed stream; a download without a stream returns only once its copies are
    done, so a read on an unrelated stream without any wait already sees the results"""
    torch = _torch()
    B = 8
    L, R = td.frames(B, seed=240)
    with api.Engine(FW, FH, max_batch=B) as e, api.Engine(FW, FH, max_batch=B) as ref:
        stages, want = workload(e, "points", B)
        workload(ref, "points", B)
        ref.compute(L, R, stages)
        want0, (offs0, pts0) = ref.download(B, **want), ref.download_points(B)
        dl, dr = to_dev(L), to_dev(R)
        out, _ = pitched(B, e.info.height, e.info.width, False)
        pts_buf = torch.full((len(pts0) + 1, 3), -7.0, device="cuda:0")
        torch.cuda.synchronize()
        slow, reader = torch.cuda.Stream(), torch.cuda.Stream()
        for what in ("disp", "points"):
            with torch.cuda.stream(slow):
                torch.cuda._sleep(SLEEP)
            e.compute_tensors(dl, dr, stages, stream=slow)
            with torch.cuda.stream(reader):
                if what == "disp":
                    e.download_device(B, out={"disp": out["disp"]})
                    snap = out["disp"].clone()
                else:
                    e.download_points_device(B, out=pts_buf)
                    snap = pts_buf.clone()
            reader.synchronize()
            if what == "disp":
                assert np.array_equal(snap.cpu().numpy(), want0["disp"])
            else:
                assert np.array_equal(snap[:len(pts0)].cpu().numpy().view(np.uint8), pts0.view(np.uint8))
            torch.cuda.synchronize()


# ---- 5. multi-device -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("devs", td.DEVICE_LISTS, ids=td.LIST_IDS)
def test_multi_device(devs):
    torch = _torch()
    mb = td.max_batch(devs)
    with api.Engine(FW, FH, max_batch=mb, devices=devs) as e:
        B = e.info.max_batch
        L, R = td.frames(B, seed=250)
        stages, want = workload(e, "points", B)
        with api.Engine(FW, FH, max_batch=B) as one:
            workload(one, "points", B)
            targets = [0] + ([1] if td.NDEV >= 2 else [])          # destination and caller stream on another device too
            for b in sorted({1, len(devs), B}):
                one.compute(L[:b], R[:b], stages)
                ref, (offs, pts) = one.download(b, **want), one.download_points(b)
                for dev in targets:
                    with torch.cuda.device(dev):
                        s = torch.cuda.Stream()
                    dl, dr = to_dev(L[:b], dev), to_dev(R[:b], dev)
                    torch.cuda.synchronize(dev)
                    e.compute_tensors(dl, dr, stages, stream=s)
                    got = e.download_device(b, stream=s, device=dev, **want)
                    offs_d, pts_d = e.download_points_device(b, stream=s, device=dev)
                    s.synchronize()
                    assert got["disp"].device == torch.device("cuda", dev) and pts_d.device == torch.device("cuda", dev)
                    same(got, ref, "devices %s, batch %d, destination on device %d" % (devs, b, dev))
                    assert np.array_equal(offs_d, offs), (devs, b, dev)
                    assert np.array_equal(pts_d.cpu().numpy().view(np.uint8), pts.view(np.uint8)), (devs, b, dev)


# ---- 6. rejections ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_rejections_leave_results_downloadable():
    torch = _torch()
    B = 6
    L, R = td.frames(B, seed=260)
    with api.Engine(FW, FH, max_batch=B) as e:
        lib, ctx = e._lib, e._ctx
        stages, want = workload(e, "points", B)
        H, W = e.info.height, e.info.width
        dev = torch.empty((B, H, W), dtype=torch.int16, device="cuda:0")
        # nothing computed yet
        assert lib.mvsv_download_device(ctx, 0, dev.data_ptr(), 2 * W, None, None, 0, None, None, None) == ERR_STATE
        offs = np.full(B + 1, -1, np.int64)
        assert lib.mvsv_download_points_device(ctx, 0, offs.ctypes.data, None, 0, None) == ERR_STATE
        e.compute(L, R, stages & ~api.STAGE_XYZ)
        before = e.download(B, rect=True, means=True)
        offs0, pts0 = e.download_points(B)

        hostbuf = np.zeros((B, H, W), np.int16)
        pin = api.pinned((B, H, W), np.int16)
        pin_pts = api.pinned((len(pts0) + 1, 3), np.float32)
        try:
            for p in (hostbuf.ctypes.data, pin.ptr):
                rc = lib.mvsv_download_device(ctx, 0, p, 2 * W, None, None, 0, None, None, None)
                assert rc == ERR_INVALID and "mvsv_download_age" in lib.mvsv_last_error(ctx).decode()
            for p in (np.zeros((len(pts0) + 1, 3), np.float32).ctypes.data, pin_pts.ptr):
                rc = lib.mvsv_download_points_device(ctx, 0, offs.ctypes.data, p, len(pts0) + 1, None)
                assert rc == ERR_INVALID and "mvsv_download_points" in lib.mvsv_last_error(ctx).decode()
        finally:
            pin.close()
            pin_pts.close()
        assert pin.ptr is None
        xyz = torch.empty((B, H, W, 3), dtype=torch.float32, device="cuda:0")
        calls = [
            (ERR_INVALID, lambda: lib.mvsv_download_device(ctx, 0, dev.data_ptr(), 2 * W - 2, None, None, 0, None, None, None)),
            (ERR_INVALID, lambda: lib.mvsv_download_device(ctx, 0, None, 0, dev.data_ptr(), None, W - 1, None, None, None)),
            (ERR_INVALID, lambda: lib.mvsv_download_device(ctx, 1, dev.data_ptr(), 2 * W, None, None, 0, None, None, None)),
            (ERR_INVALID, lambda: lib.mvsv_download_device(ctx, -1, dev.data_ptr(), 2 * W, None, None, 0, None, None, None)),
            (ERR_INVALID, lambda: lib.mvsv_download_points_device(ctx, 1, offs.ctypes.data, None, 0, None)),
            (ERR_STATE, lambda: lib.mvsv_download_device(ctx, 0, None, 0, None, None, 0, xyz.data_ptr(), None, None)),
        ]
        for code, call in calls:
            assert call() == code
            torch.cuda.synchronize()
            td.assert_same(e.download(B, rect=True, means=True), before, "after a rejection")
        # a points buffer too small: offsets written, the destination untouched
        if len(pts0) > 0:
            small = torch.full((len(pts0) - 1, 3), -7.0, device="cuda:0")
            offs[:] = -1
            s = torch.cuda.Stream()
            rc = lib.mvsv_download_points_device(ctx, 0, offs.ctypes.data, small.data_ptr(), len(pts0) - 1, s.cuda_stream)
            assert rc == ERR_INVALID
            assert np.array_equal(offs, offs0)
            torch.cuda.synchronize()
            assert (small == -7.0).all()
        o2, p2 = e.download_points_device(B)
        assert np.array_equal(o2, offs0) and np.array_equal(p2.cpu().numpy().view(np.uint8), pts0.view(np.uint8))


# ---- 7. Python -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_python_binding_types_and_out():
    torch = _torch()
    B = 5
    L, R = td.frames(B, seed=270)
    with api.Engine(FW, FH, max_batch=B) as e:
        stages, want = workload(e, "pipeline", B)
        e.compute(L, R, stages)
        ref = e.download(B, **want)
        H, W = e.info.height, e.info.width
        got = e.download_device(B, **want)
        shapes = {"disp": ((B, H, W), torch.int16), "rectL": ((B, H, W), torch.uint8), "rectR": ((B, H, W), torch.uint8),
                  "xyz": ((B, H, W, 3), torch.float32), "means": ((B, e.info.num_rois), torch.float32)}
        assert set(got) == set(shapes)
        for k, (shape, dtype) in shapes.items():
            assert tuple(got[k].shape) == shape and got[k].dtype == dtype and got[k].is_cuda, k
        same(got, ref, "defaults")
        out = {k: torch.empty(shape, dtype=dtype, device="cuda:0") for k, (shape, dtype) in shapes.items()}
        got = e.download_device(B, out=out, **want)
        assert all(got[k].data_ptr() == out[k].data_ptr() for k in shapes)
        same(got, ref, "out=")
        with pytest.raises(ValueError):
            e.download_device(B, out={"disp": torch.empty((B, H, W), dtype=torch.int32, device="cuda:0")})
        with pytest.raises(ValueError):
            e.download_device(B, xyz=True, out={"xyz": torch.empty((B, H, W, 4), device="cuda:0")[..., :3]})
        with pytest.raises(ValueError):
            e.download_device(B - 1)
        # device inputs with pitched rows: compute_tensors reads the tensors' strides
        mb = e.info.max_batch
        with api.Engine(FW, FH, max_batch=mb) as ref2, api.Engine(FW, FH, max_batch=mb) as e2:
            stages2, _ = workload(ref2, "sgbm", mb)
            workload(e2, "sgbm", mb)
            Lp = torch.zeros((B, FH, FW + 48), dtype=torch.uint8, device="cuda:0")
            Rp = torch.zeros((B, FH, FW + 16), dtype=torch.uint8, device="cuda:0")
            Lp[:, :, :FW] = to_dev(L)
            Rp[:, :, :FW] = to_dev(R)
            with pytest.raises(ValueError):                      # different frame strides
                e2.compute_tensors(Lp[:, :, :FW], Rp[:, :, :FW], stages2)
            Rq = torch.zeros((B, FH, FW + 48), dtype=torch.uint8, device="cuda:0")
            Rq[:, :, :FW] = to_dev(R)
            torch.cuda.synchronize()
            e2.compute_tensors(Lp[:, :, :FW], Rq[:, :, :FW], stages2)
            ref2.compute(L, R, stages2)
            td.assert_same(e2.download(B), ref2.download(B), "pitched device inputs")
            e2.compute_tensors(Lp[0, :, :FW], Rq[0, :, :FW], stages2)      # one frame, 2-D
            ref2.compute(L[0], R[0], stages2)
            td.assert_same(e2.download(1), ref2.download(1), "one 2-D frame")
            with pytest.raises(ValueError):
                e2.compute_tensors(Lp.float(), Rq.float(), stages2)
