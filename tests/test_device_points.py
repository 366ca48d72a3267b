"""Point lists and per-frame min/max into device memory with no host wait: mvsv_download_points_stream and
mvsv_download_minmax_device (Engine.download_points_stream, download_minmax_device).

Both must give what the host calls of the same compute give, bit for bit: mvsv_download_points (offsets and points) and
mvsv_download_minmax.  The points are written by a kernel on the engine's download stream, cut off at the caller's
capacity; the tests check the cut, the sentinels past it, and that the offsets are always complete.  The ordering tests
delay the caller's stream (torch.cuda._sleep), so that a host wait or a missing device wait shows every time."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import cases
import test_devices as td
from mvstereovision3_b200 import api
from test_device_io import SLEEP, streams, to_dev, workload
import test_points as tp
from test_points import frame_kinds, runs_map, same_bits

ERR_INVALID, ERR_STATE = -1, -4
FW, FH = td.FW, td.FH
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENT = -7.0                     # sentinel of the points past the capacity


# ---- CPU side --------------------------------------------------------------------------------------------------------
def test_api_imports_without_torch():
    code = ("import sys; sys.modules['torch'] = None\n"          # `import torch` now raises ImportError
            "from mvstereovision3_b200 import api\n"
            "assert {'mvsv_download_points_stream', 'mvsv_download_minmax_device'} <= set(api.ABI_SYMBOLS)\n")
    subprocess.check_call([sys.executable, "-c", code], cwd=ROOT)


def test_prototypes_declared():
    lib = api.load_library()
    vp, sz, ci = C.c_void_p, C.c_size_t, C.c_int
    assert lib.mvsv_download_points_stream.argtypes == [vp, ci, vp, vp, sz, vp]
    assert lib.mvsv_download_minmax_device.argtypes == [vp, ci, vp, vp]
    assert {"mvsv_download_points_stream", "mvsv_download_minmax_device"} <= set(api.ABI_SYMBOLS)
    with open(os.path.join(ROOT, "include", "mvsv.h")) as f:
        header = f.read()
    assert "int mvsv_download_points_stream(mvsv_ctx* ctx, int age, int64_t* offsets, float* points, size_t capacity_points," \
           in header
    assert "int mvsv_download_minmax_device(mvsv_ctx* ctx, int age, int16_t* minmax, void* stream);" in header


# ---- helpers ---------------------------------------------------------------------------------------------------------
def _torch():
    return pytest.importorskip("torch")


def host_of(e, B, age=0):
    """the host calls' results: offsets, points and (age 0 only) min/max"""
    offs, pts = e.download_points(B, age=age)
    return offs, pts, (e.download_minmax(B) if age == 0 else None)


def check_points(offs_d, pts_d, offs, pts, what, cap=None):
    """device results against the host list: offsets complete, points[:min(total, cap)] equal"""
    assert offs_d.dtype == _torch().int64 and np.array_equal(offs_d.cpu().numpy(), offs), what
    n = len(pts) if cap is None else min(len(pts), cap)
    same_bits(pts_d[:n].cpu().numpy(), pts[:n], what)


def size(name):
    """frame size of a workload: test_devices.py's frames, or test_points.py's StereoBM pairs"""
    return (FW, FH) if name == "points" else (260, 90)


def inputs(name, B, seed):
    return td.frames(B, seed=seed) if name == "points" else tp.pairs(B, 90, 260, seed=seed)


def setup(e, name, B):
    """"points": the three-rig rectify + SGBM + XYZ + POINTS pipeline; "bm": configs/bm.yml StereoBM with the left-right
    check and the speckle filter, XYZ and POINTS"""
    if name == "points":
        return workload(e, "points", B)[0]
    e.set_bm_params(**tp.BM)
    e.set_bm_filters(0, 40, 16)
    e.set_Q(cases.Q_REFERENCE)
    return api.STAGE_BM | api.STAGE_XYZ | api.STAGE_POINTS


# ---- 1. equality with the host calls ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["points", "bm"])
@pytest.mark.parametrize("kind", ["none", "side", "default"])
def test_equals_host_calls(name, kind):
    torch = _torch()
    B = 10
    L, R = inputs(name, B, 5)
    with api.Engine(*size(name), max_batch=B) as e:
        stages = setup(e, name, B)
        e.compute(L, R, stages)
        offs, pts, mm = host_of(e, B)
        assert 0 < offs[-1] < B * e.info.height * e.info.width
        s = None if kind == "none" else streams(kind)
        n0 = e.launch_count
        offs_d, pts_d = e.download_points_stream(B, stream=s)
        mm_d = e.download_minmax_device(B, stream=s)
        assert e.launch_count - n0 == 4                 # k_points_out; k_minmax_init, k_minmax, k_minmax_fold
        if s is not None:
            s.synchronize()
        assert tuple(offs_d.shape) == (B + 1,) and tuple(pts_d.shape) == (B * e.info.height * e.info.width, 3)
        assert pts_d.dtype == torch.float32 and mm_d.dtype == torch.int16 and tuple(mm_d.shape) == (B, 2)
        check_points(offs_d, pts_d, offs, pts, "%s %s" % (name, kind))
        assert np.array_equal(mm_d.cpu().numpy(), mm)


CRAFTED = ((2049, 1, 3), (64, 32, 3), (40, 103, 3), (752, 479, 2))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", CRAFTED, ids=["%dx%dx%d" % s for s in CRAFTED])
def test_crafted_maps(shape):
    """runs of valid pixels across tile, warp and frame boundaries with the int16 limits; empty and full frames"""
    W, H, B = shape
    maps = [runs_map(W, H, B, seed=W * H), frame_kinds(W, H)]
    with api.Engine(W, H, max_batch=len(maps[1])) as e:
        e.set_Q(cases.Q_REFERENCE)
        for m in maps:
            b = len(m)
            e.debug_postfilter(m, median=False, stages=api.STAGE_POINTS)
            offs, pts, mm = host_of(e, b)
            s = _torch().cuda.Stream()
            offs_d, pts_d = e.download_points_stream(b, stream=s)
            mm_d = e.download_minmax_device(b, stream=s)
            s.synchronize()
            check_points(offs_d, pts_d, offs, pts, "%dx%d batch %d" % (W, H, b))
            assert np.array_equal(mm_d.cpu().numpy(), mm)
        assert (mm == 0).all(axis=1).any()                              # frame_kinds has frames without a value > 0


# ---- 2. NULL points and truncation -----------------------------------------------------------------------------------
@pytest.mark.gpu
def test_offsets_only_and_truncation():
    torch = _torch()
    B = 8
    L, R = td.frames(B, seed=11)
    with api.Engine(FW, FH, max_batch=B) as e:
        lib, ctx = e._lib, e._ctx
        stages = setup(e, "points", B)
        e.compute(L, R, stages)
        offs, pts, _ = host_of(e, B)
        total = int(offs[-1])
        assert total > 2 and offs[3] > offs[2]
        od = torch.full((B + 1,), -1, dtype=torch.int64, device="cuda:0")
        torch.cuda.synchronize()
        assert lib.mvsv_download_points_stream(ctx, 0, od.data_ptr(), None, 0, None) == 0
        assert np.array_equal(od.cpu().numpy(), offs)
        mid = int(offs[2] + (offs[3] - offs[2]) // 2)                  # ends inside frame 2
        for cap in (0, total - 1, total, mid):
            buf = torch.full((total + 9, 3), SENT, device="cuda:0")
            od.fill_(-1)
            torch.cuda.synchronize()
            s = torch.cuda.Stream()
            assert lib.mvsv_download_points_stream(ctx, 0, od.data_ptr(), buf.data_ptr(), cap, s.cuda_stream) == 0
            s.synchronize()
            o = od.cpu().numpy()
            assert np.array_equal(o, offs), cap                          # always complete
            assert (o[-1] > cap) == (cap < total)                         # truncation shows on the device
            check_points(od, buf, offs, pts, "capacity %d" % cap, cap=cap)
            assert (buf[min(cap, total):] == SENT).all(), cap            # nothing past the capacity
            complete = [f for f in range(B) if o[f + 1] <= cap]
            assert complete == list(range(len(complete)))
        # the binding: a preallocated pair, shorter than the list
        bo = torch.empty(B + 1, dtype=torch.int64, device="cuda:0")
        bp = torch.full((mid, 3), SENT, device="cuda:0")
        offs_d, pts_d = e.download_points_stream(B, out=(bo, bp))
        assert offs_d.data_ptr() == bo.data_ptr() and pts_d.data_ptr() == bp.data_ptr()
        check_points(offs_d, pts_d, offs, pts, "out=", cap=mid)
        with pytest.raises(ValueError):
            e.download_points_stream(B, out=(bo[:B], bp))
        with pytest.raises(ValueError):
            e.download_points_stream(B, out=(bo, bp.view(-1)))


# ---- 3. two slots: age 1 -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_two_slot_loop_and_minmax_age():
    """compute k+1, then the age-1 point list and min/max of compute k, all on one stream without a host wait; min/max at
    age 1 equals the host call made right after the earlier compute, frames without a value > 0 included"""
    torch = _torch()
    W, H = 64, 32
    N, B = 5, 7
    maps = [frame_kinds(W, H)] + [runs_map(W, H, B, seed=k) for k in range(1, N)]
    with api.Engine(W, H, max_batch=B) as e, api.Engine(W, H, max_batch=B) as ref:
        refs = []
        for m in maps:
            ref.set_Q(cases.Q_REFERENCE)
            ref.debug_postfilter(m, median=False, stages=api.STAGE_POINTS)
            refs.append(host_of(ref, B))
        assert (refs[0][2] == 0).all(axis=1).any()
        e.set_Q(cases.Q_REFERENCE)
        e.set_io_slots(2)
        s = torch.cuda.Stream()
        got = []
        e.debug_postfilter(maps[0], median=False, stages=api.STAGE_POINTS)
        for k in range(1, N):
            e.debug_postfilter(maps[k], median=False, stages=api.STAGE_POINTS)
            got.append((e.download_points_stream(B, age=1, stream=s), e.download_minmax_device(B, age=1, stream=s)))
        got.append((e.download_points_stream(B, age=0, stream=s), e.download_minmax_device(B, age=0, stream=s)))
        s.synchronize()
        for k, ((od, pd), mmd) in enumerate(got):
            check_points(od, pd, refs[k][0], refs[k][1], "step %d" % k)
            assert np.array_equal(mmd.cpu().numpy(), refs[k][2]), k


@pytest.mark.gpu
def test_pipelined_compute_loop():
    """device inputs, two I/O slots, the age-1 results of the previous compute on the caller's stream"""
    torch = _torch()
    B, N = 6, 5
    inputs = [td.frames(B, seed=400 + 10 * k) for k in range(N)]
    with api.Engine(FW, FH, max_batch=B) as e, api.Engine(FW, FH, max_batch=B) as ref:
        stages = setup(e, "points", B)
        setup(ref, "points", B)
        want = []
        for L, R in inputs:
            ref.compute(L, R, stages)
            want.append(host_of(ref, B))
        dev_in = [(to_dev(L), to_dev(R)) for L, R in inputs]
        torch.cuda.synchronize()
        e.set_io_slots(2)
        s = torch.cuda.Stream()
        got = []
        e.compute_tensors(*dev_in[0], stages, stream=s)
        for k in range(1, N):
            e.compute_tensors(*dev_in[k], stages, stream=s)
            got.append((e.download_points_stream(B, age=1, stream=s), e.download_minmax_device(B, age=1, stream=s)))
        got.append((e.download_points_stream(B, stream=s), e.download_minmax_device(B, stream=s)))
        s.synchronize()
        for k, ((od, pd), mmd) in enumerate(got):
            check_points(od, pd, want[k][0], want[k][1], "step %d" % k)
            assert np.array_equal(mmd.cpu().numpy(), want[k][2]), k


# ---- 4. no host wait, ordering ---------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["side", "default"])
def test_no_host_wait(kind):
    """the compute waits for a delayed caller's stream: the download calls return while the stream is still busy"""
    torch = _torch()
    B = 8
    L, R = td.frames(B, seed=500)
    with api.Engine(FW, FH, max_batch=B) as e, api.Engine(FW, FH, max_batch=B) as ref:
        stages = setup(e, "points", B)
        setup(ref, "points", B)
        ref.compute(L, R, stages)
        offs, pts, mm = host_of(ref, B)
        dl, dr = to_dev(L), to_dev(R)
        # the outputs exist before the delay: the calls themselves allocate nothing
        od = torch.empty(B + 1, dtype=torch.int64, device="cuda:0")
        pd = torch.empty((B * e.info.height * e.info.width, 3), dtype=torch.float32, device="cuda:0")
        mmd = torch.empty((B, 2), dtype=torch.int16, device="cuda:0")
        e.compute_tensors(dl, dr, stages)                 # the engine's own allocations happen before the delay too
        e.download_points_stream(B, out=(od, pd))
        e.download_minmax_device(B, out=mmd)
        torch.cuda.synchronize()
        s = streams(kind)
        with torch.cuda.stream(s):
            torch.cuda._sleep(SLEEP)
            e.compute_tensors(dl, dr, stages, stream=s)
            e.download_points_stream(B, out=(od, pd), stream=s)
            e.download_minmax_device(B, out=mmd, stream=s)
            busy = not s.query()
        assert busy, "a download call waited on the host"
        s.synchronize()
        check_points(od, pd, offs, pts, "behind a delay")
        assert np.array_equal(mmd.cpu().numpy(), mm)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["side", "default"])
def test_pending_points_out_holds_the_slot(kind):
    """one I/O slot: a compute submitted at once after a delayed download writes the slot only after k_points_out and the
    min/max reduction have read it"""
    torch = _torch()
    B = 8
    L0, R0 = td.frames(B, seed=520)
    L1, R1 = td.frames(B, seed=620)
    with api.Engine(FW, FH, max_batch=B) as e, api.Engine(FW, FH, max_batch=B) as ref:
        stages = setup(e, "points", B)
        setup(ref, "points", B)
        refs = []
        for L, R in ((L0, R0), (L1, R1)):
            ref.compute(L, R, stages)
            refs.append(host_of(ref, B))
        e.compute(L0, R0, stages)
        e.sync()
        s = streams(kind)
        with torch.cuda.stream(s):
            torch.cuda._sleep(SLEEP)
            od, pd = e.download_points_stream(B, stream=s)
            mmd = e.download_minmax_device(B, stream=s)
        e.compute(L1, R1, stages)                                        # the same (only) slot
        s.synchronize()
        check_points(od, pd, refs[0][0], refs[0][1], "delayed download")
        assert np.array_equal(mmd.cpu().numpy(), refs[0][2])
        offs1, pts1, mm1 = host_of(e, B)
        assert np.array_equal(offs1, refs[1][0]) and np.array_equal(mm1, refs[1][2])
        same_bits(pts1, refs[1][1], "the compute after it")


@pytest.mark.gpu
def test_no_stream_returns_with_the_writes_done():
    """the compute is held back behind a delayed stream; without a stream the calls return with their writes done, so a
    read on an unrelated stream sees the results without any wait"""
    torch = _torch()
    B = 8
    L, R = td.frames(B, seed=540)
    with api.Engine(FW, FH, max_batch=B) as e, api.Engine(FW, FH, max_batch=B) as ref:
        stages = setup(e, "points", B)
        setup(ref, "points", B)
        ref.compute(L, R, stages)
        offs, pts, mm = host_of(ref, B)
        dl, dr = to_dev(L), to_dev(R)
        torch.cuda.synchronize()
        slow, reader = torch.cuda.Stream(), torch.cuda.Stream()
        with torch.cuda.stream(slow):
            torch.cuda._sleep(SLEEP)
        e.compute_tensors(dl, dr, stages, stream=slow)
        with torch.cuda.stream(reader):
            od, pd = e.download_points_stream(B)
            mmd = e.download_minmax_device(B)
            snap = (od.clone(), pd.clone(), mmd.clone())
        reader.synchronize()
        check_points(snap[0], snap[1], offs, pts, "stream=None")
        assert np.array_equal(snap[2].cpu().numpy(), mm)


# ---- 5. multi-device -------------------------------------------------------------------------------------------------
def _multi_device_case(devs, dev):
    """the single engine's host calls against a ctx of the parts `devs`, the destinations and the caller's stream on
    device `dev`: batches with parts without frames, a part without points, a capacity inside the second part's share"""
    torch = _torch()
    mb, n = td.max_batch(devs), len(devs)
    for name in ("points", "bm"):
        with api.Engine(*size(name), max_batch=mb, devices=devs) as e:
            B = e.info.max_batch
            one = api.Engine(*size(name), max_batch=B)
            L, R = inputs(name, B, 560)
            L[:B // n], R[:B // n] = 0, 0         # textureless: under StereoBM's texture check part 0 has no point
            stages = setup(e, name, B)
            setup(one, name, B)
            with torch.cuda.device(dev):
                s = torch.cuda.Stream()
            for b in sorted({1, n - 1, n, B} - {0}):
                one.compute(L[:b], R[:b], stages)
                offs, pts, mm = host_of(one, b)
                e.compute(L[:b], R[:b], stages)
                od, pd = e.download_points_stream(b, stream=s, device=dev)
                mmd = e.download_minmax_device(b, stream=s, device=dev)
                s.synchronize()
                what = "devices %s %s batch %d on device %d" % (devs, name, b, dev)
                assert od.device == torch.device("cuda", dev) and mmd.device == od.device
                check_points(od, pd, offs, pts, what)
                assert np.array_equal(mmd.cpu().numpy(), mm), what
                first = [k * b // n for k in range(n + 1)]
                if name == "bm" and b == B:
                    assert offs[first[1]] == 0 < offs[-1], what
                a, z = int(offs[first[1]]), int(offs[first[2]])
                if z - a >= 2:
                    cap = (a + z) // 2
                    buf = torch.full((z + 5, 3), SENT, device=od.device)
                    torch.cuda.synchronize(dev)
                    od2, pd2 = e.download_points_stream(b, out=(torch.empty_like(od), buf[:cap]), stream=s)
                    s.synchronize()
                    check_points(od2, buf, offs, pts, what + ", capacity %d" % cap, cap=cap)
                    assert (buf[cap:] == SENT).all(), what
            one.close()


@pytest.mark.gpu
@pytest.mark.parametrize("devs", td.DEVICE_LISTS, ids=td.LIST_IDS)
def test_multi_device(devs):
    _multi_device_case(devs, 0)


@pytest.mark.gpu
@pytest.mark.skipif(td.NDEV < 2, reason="needs a second GPU for a destination on another device")
@pytest.mark.parametrize("devs", [[0, 0], [0, 1]], ids=["0x0", "0x1"])
def test_multi_device_destination_on_another_gpu(devs):
    _multi_device_case(devs, 1)


# ---- 6. rejections ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_rejections_leave_results_downloadable():
    torch = _torch()
    B = 6
    L, R = td.frames(B, seed=580)
    with api.Engine(FW, FH, max_batch=B) as e:
        lib, ctx = e._lib, e._ctx
        stages = setup(e, "points", B)
        od = torch.full((B + 1,), -1, dtype=torch.int64, device="cuda:0")
        pd = torch.full((B * e.info.height * e.info.width, 3), SENT, device="cuda:0")
        mmd = torch.full((B, 2), -3, dtype=torch.int16, device="cuda:0")
        torch.cuda.synchronize()
        cap = pd.shape[0]
        # nothing computed yet
        assert lib.mvsv_download_points_stream(ctx, 0, od.data_ptr(), pd.data_ptr(), cap, None) == ERR_STATE
        assert lib.mvsv_download_minmax_device(ctx, 0, mmd.data_ptr(), None) == ERR_STATE
        e.compute(L, R, stages)
        offs, pts, mm = host_of(e, B)
        e.compute(L, R, stages & ~api.STAGE_POINTS)
        assert lib.mvsv_download_points_stream(ctx, 0, od.data_ptr(), pd.data_ptr(), cap, None) == ERR_STATE
        assert "POINTS" in lib.mvsv_last_error(ctx).decode()
        e.compute(L, R, stages)

        host_offs = np.zeros(B + 1, np.int64)
        host_pts = np.zeros((cap, 3), np.float32)
        pin = api.pinned((cap, 3), np.float32)
        try:
            calls = [
                (ERR_INVALID, lambda: lib.mvsv_download_points_stream(ctx, 0, None, pd.data_ptr(), cap, None)),
                (ERR_INVALID, lambda: lib.mvsv_download_points_stream(ctx, 0, host_offs.ctypes.data, pd.data_ptr(), cap, None)),
                (ERR_INVALID, lambda: lib.mvsv_download_points_stream(ctx, 0, od.data_ptr(), host_pts.ctypes.data, cap, None)),
                (ERR_INVALID, lambda: lib.mvsv_download_points_stream(ctx, 0, od.data_ptr(), pin.ptr, cap, None)),
                (ERR_INVALID, lambda: lib.mvsv_download_points_stream(ctx, 1, od.data_ptr(), pd.data_ptr(), cap, None)),
                (ERR_INVALID, lambda: lib.mvsv_download_points_stream(ctx, -1, od.data_ptr(), pd.data_ptr(), cap, None)),
                (ERR_INVALID, lambda: lib.mvsv_download_minmax_device(ctx, 0, None, None)),
                (ERR_INVALID, lambda: lib.mvsv_download_minmax_device(ctx, 0, host_offs.ctypes.data, None)),
                (ERR_INVALID, lambda: lib.mvsv_download_minmax_device(ctx, 0, pin.ptr, None)),
                (ERR_INVALID, lambda: lib.mvsv_download_minmax_device(ctx, 1, mmd.data_ptr(), None)),
                (ERR_INVALID, lambda: lib.mvsv_download_minmax_device(ctx, -1, mmd.data_ptr(), None)),
            ]
            for code, call in calls:
                assert call() == code
                torch.cuda.synchronize()
                assert (od == -1).all() and (pd == SENT).all() and (mmd == -3).all(), "a rejected call wrote"
                o, p, m = host_of(e, B)
                assert np.array_equal(o, offs) and np.array_equal(m, mm)
                same_bits(p, pts, "after a rejection")
        finally:
            pin.close()
        got_o, got_p = e.download_points_stream(B)
        check_points(got_o, got_p, offs, pts, "after the rejections")
        assert np.array_equal(e.download_minmax_device(B).cpu().numpy(), mm)
        with pytest.raises(ValueError):
            e.download_minmax_device(B, out=torch.empty((B, 2), dtype=torch.int32, device="cuda:0"))
