"""One engine over several devices (mvsv_init_devices): every batch is split into contiguous shares across the parts, and
the outputs are those of one single-device engine given the whole batch, bit for bit (XYZ included).

The device lists are [0, 0] and [0, 0, 0] (several engines on one GPU, which exercises the splitting on any box) and,
on a box with two or more GPUs, every device."""
import numpy as np
import pytest

import cases
from mvstereovision3_b200 import api, synth

ERR_INVALID, ERR_CUDA, ERR_STATE, ERR_UNSUPPORTED = -1, -2, -4, -5


def _device_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


NDEV = _device_count()
DEVICE_LISTS = [[0, 0], [0, 0, 0]] + ([list(range(NDEV))] if NDEV >= 2 else [])
LIST_IDS = ["x".join(map(str, d)) for d in DEVICE_LISTS]

# cv::StereoSGBM with configs/sgbm.yml at numDisp 64 (cfg 2), StereoBM with the filters of mvsv_set_bm_filters
SGBM = dict(minDisp=1, numDisp=64, blockSize=13, disp12MaxDiff=0, preFilterCap=0, uniquenessRatio=0,
            speckleWindowSize=150, speckleRange=2, disparityMode=0)
BM = dict(numDisp=64, blockSize=21, preFilterCap=31, textureThreshold=10, uniquenessRatio=15)
FW, FH = 256, 72                      # raw frames
ROI_W, ROI_H = 224, 60                # rectified ROI of every rig
RIGS = (0, 7, 63)                     # three rigs: warp maps of different seeds at different ROI offsets


def max_batch(devs):
    return max(10, 2 * len(devs) + 1)


def batches(devs):
    n, mb = len(devs), max_batch(devs)
    return sorted({1, n - 1, n, n + 1, 2 * n + 1, mb} - {0})


def frames(B, seed=0):
    pairs = [synth.stereogram(FH, FW, 1, 64, seed=seed + i)[:2] for i in range(B)]
    return np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs])


def rig_table(B):
    """unsorted: every rig, in a shuffled order"""
    return [int(v) for v in np.random.default_rng(5).choice(RIGS, B)]


def setup(e, workload, B):
    """the state of one workload; returns its stages and what to download"""
    if workload == "sgbm":
        e.set_sgbm_params(**SGBM)
        return api.STAGE_SGBM, {}
    if workload == "bm":
        e.set_bm_params(**BM)
        e.set_bm_filters(1, 100, 32)
        return api.STAGE_BM, {}
    # rectify + SGBM + XYZ + MEANS with three rigs, resized by 0.5 in "pipeline_resize"
    for k, rig in enumerate(RIGS):
        for cam in range(2):
            mx, my = cases.warp_maps(FH, FW, seed=10 * k + cam)
            e.upload_rectify_maps(cam, mx, my, (4 + 9 * k, 2 + 3 * k, ROI_W, ROI_H), rig=rig)
        q = cases.Q_REFERENCE.copy()
        q[0, 3] -= 3 * k
        q[3, 2] *= 1 + 0.1 * k
        e.set_Q(q, rig=rig)
    if workload == "pipeline_resize":
        e.set_resize(0.5)
    e.set_sgbm_params(**SGBM)
    W, H = e.info.width, e.info.height
    e.set_mean_rois(api.subimage_rois(W, H) + api.samplepoint_rois(W, H))
    e.set_frame_rigs(rig_table(B))
    return api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_XYZ | api.STAGE_MEANS, dict(rect=True, xyz=True, means=True)


def results(e, batch, want, age=0):
    out = e.download(batch, age=age, **want)
    if age == 0:
        out["minmax"] = e.download_minmax(batch)
    return out


def assert_same(got, ref, what):
    assert got.keys() == ref.keys(), what
    for key in ref:
        # bit for bit, NaN payloads of XYZ included
        assert np.array_equal(got[key].view(np.uint8), ref[key].view(np.uint8)), "%s: %s differs" % (what, key)


def compute(e, L, R, stages, device_inputs):
    if device_inputs is None:
        e.compute(L, R, stages)
    else:
        dl, dr = device_inputs
        B, H, W = L.shape
        e.compute_device(dl.data_ptr(), W, dr.data_ptr(), W, H * W, B, stages)


WORKLOADS = [("sgbm", False), ("bm", False), ("pipeline", False), ("pipeline_resize", True)]


@pytest.mark.gpu
@pytest.mark.parametrize("devs", DEVICE_LISTS, ids=LIST_IDS)
@pytest.mark.parametrize("workload,device_inputs", WORKLOADS, ids=[w + ("_device" if d else "") for w, d in WORKLOADS])
def test_split_equals_one_engine(devs, workload, device_inputs):
    """every batch size from one frame (parts without frames) to the whole capacity"""
    mb = max_batch(devs)
    with api.Engine(FW, FH, max_batch=mb, devices=devs) as e:
        B = e.info.max_batch
        L, R = frames(B)
        dev_in = None
        if device_inputs:
            torch = pytest.importorskip("torch")
            dev_in = (torch.from_numpy(L).cuda(0), torch.from_numpy(R).cuda(0))
            torch.cuda.synchronize()
        stages, want = setup(e, workload, B)
        with api.Engine(FW, FH, max_batch=B) as ref:
            setup(ref, workload, B)
            for b in sorted(set(batches(devs) + [B])):
                d = (dev_in[0][:b], dev_in[1][:b]) if dev_in else None
                compute(e, L[:b], R[:b], stages, d)
                compute(ref, L[:b], R[:b], stages, d)
                assert e.info.last_batch == b
                assert_same(results(e, b, want), results(ref, b, want), "%s, batch %d" % (workload, b))


@pytest.mark.gpu
@pytest.mark.parametrize("devs", DEVICE_LISTS, ids=LIST_IDS)
def test_two_io_slots_across_batch_sizes(devs):
    """age 1 is the same compute on every part, also when consecutive computes split differently (re-cut rig slices)"""
    mb = max_batch(devs)
    n = len(devs)
    sizes = [mb, 1, n + 1, 2 * n + 1, n - 1, mb]
    L, R = frames(mb, seed=20)
    with api.Engine(FW, FH, max_batch=mb, devices=devs) as e, api.Engine(FW, FH, max_batch=mb) as ref:
        stages, want = setup(e, "pipeline", mb)
        setup(ref, "pipeline", mb)
        e.set_io_slots(2)
        want_prev = None
        for i, b in enumerate(sizes):
            first = (3 * i) % (mb - b + 1)                 # a different window of frames each time
            e.compute(L[first:first + b], R[first:first + b], stages)
            if want_prev is not None:
                assert_same(e.download(want_prev[0], age=1, **want), want_prev[1], "age 1 before compute %d" % i)
            ref.compute(L[first:first + b], R[first:first + b], stages)
            want_prev = (b, ref.download(b, **want))
        assert_same(e.download(want_prev[0], **want), want_prev[1], "last compute")


def _rejections(e):
    """each setter rejection include/mvsv.h lists, as (what, code)"""
    x, y, w, h = 4, 2, ROI_W, ROI_H
    mx, my = cases.warp_maps(FH, FW, seed=0)
    K = np.array([[300.0, 0, 120], [0, 300, 36], [0, 0, 1]])
    Rm = np.eye(3)
    P = np.hstack([K, np.zeros((3, 1))])
    calls = [
        ("sgbm numDisp", lambda: e.set_sgbm_params(**dict(SGBM, numDisp=12))),
        ("sgbm contract", lambda: e.set_sgbm_params(**dict(SGBM, blockSize=31, preFilterCap=63))),
        ("sgbm uniqueness", lambda: e.set_sgbm_params(**dict(SGBM, uniquenessRatio=101))),
        ("bm numDisp", lambda: e.set_bm_params(**dict(BM, numDisp=24))),
        ("bm blockSize", lambda: e.set_bm_params(**dict(BM, blockSize=20))),
        ("bm speckle window", lambda: e.set_bm_filters(1, -1, 0)),
        ("bm speckle range", lambda: e.set_bm_filters(1, 100, -1)),
        ("resize", lambda: e.set_resize(9.0)),
        ("maps roi", lambda: e.upload_rectify_maps(0, mx, my, (x, y, FW, h))),
        ("maps rig", lambda: e.upload_rectify_maps(0, mx, my, (x, y, w, h), rig=api.MAX_RIGS)),
        ("rectification model", lambda: e.set_rectification(0, K, np.zeros(3), Rm, P, (x, y, w, h))),
        ("rectification singular", lambda: e.set_rectification(0, K, None, Rm, np.zeros((3, 4)), (x, y, w, h))),
        ("rig roi size", lambda: e.upload_rectify_maps(0, mx, my, (x, y, w - 2, h), rig=5)),
        ("camera roi", lambda: e.upload_rectify_maps(1, mx, my, (x + 1, y, w, h))),
        ("Q rig", lambda: e.set_Q(cases.Q_REFERENCE, rig=-1)),
        ("frame rigs length", lambda: e.set_frame_rigs([0] * (e.info.max_batch + 1))),
        ("frame rigs rig", lambda: e.set_frame_rigs([0, api.MAX_RIGS])),
        ("roi outside", lambda: e.set_mean_rois([(0, 0, e.info.width + 1, 1)])),
        ("io slots", lambda: e.set_io_slots(3)),
    ]
    out = []
    for what, call in calls:
        with pytest.raises(api.MvsvError) as ei:
            call()
        out.append((what, ei.value.code))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("devs", DEVICE_LISTS[:2], ids=LIST_IDS[:2])
def test_rejections(devs):
    mb = max_batch(devs)
    L, R = frames(mb, seed=30)
    with api.Engine(FW, FH, max_batch=mb, devices=devs) as e, api.Engine(FW, FH, max_batch=e.info.max_batch) as one:
        stages, want = setup(e, "pipeline", mb)
        setup(one, "pipeline", mb)
        e.compute(L, R, stages)
        before = e.download(mb, **want)
        # the same codes as on one engine, and the engine keeps computing what it computed
        assert _rejections(e) == _rejections(one)
        e.compute(L, R, stages)
        assert_same(e.download(mb, **want), before, "after the setter rejections")

        # computes rejected in phase 1, also when only the last part's frames are at fault: the slot stays as it was
        def rejected(table, code):
            e.set_frame_rigs(table)
            with pytest.raises(api.MvsvError) as ei:
                e.compute(L, R, stages)
            assert ei.value.code == code
            assert e.info.last_batch == mb
            assert_same(e.download(mb, **want), before, "after a rejected compute")

        rejected([0] * (mb - 1) + [9], ERR_STATE)                    # rig 9: no maps
        for cam in range(2):
            e.upload_rectify_maps(cam, *cases.warp_maps(FH, FW, seed=cam), (4, 2, ROI_W, ROI_H), rig=9)
        rejected([0] * (mb - 1) + [9], ERR_STATE)                    # rig 9: maps, no Q
        e.set_frame_rigs(rig_table(mb))
        e.set_resize(1.0)                                            # no geometry change: ROIs and results stay
        assert_same(e.download(mb, **want), before, "after set_resize(1)")
        with pytest.raises(api.MvsvError) as ei:
            e.compute(L, R, api.STAGE_SGBM | 4)                       # SGBM and BM
        assert ei.value.code == ERR_INVALID
        assert e._lib.mvsv_compute(e._ctx, L.ctypes.data, FW, R.ctypes.data, FW, FH * FW, e.info.max_batch + 1,
                                   stages) == ERR_INVALID
        assert_same(e.download(mb, **want), before, "after rejected arguments")
        e.set_resize(0.5)                                            # a geometry change drops the ROIs and the results
        assert e.info.last_batch == 0
        d = np.zeros((mb, e.info.height, e.info.width), np.int16)
        assert e._lib.mvsv_download(e._ctx, d.ctypes.data, e.info.width * 2, None, None, 0, None, None) == ERR_STATE
        with pytest.raises(api.MvsvError) as ei:
            e.compute(L, R, stages)
        assert ei.value.code == ERR_STATE and "ROIs" in str(ei.value)
        e.compute(L, R, stages & ~api.STAGE_MEANS)
        with pytest.raises(api.MvsvError) as ei:
            e.download(mb, means=True)
        assert ei.value.code == ERR_STATE


@pytest.mark.gpu
def test_unsupported_calls():
    import ctypes as C
    with api.Engine(FW, FH, max_batch=4, devices=[0, 0]) as e:
        lib, ctx = e._lib, e._ctx
        buf = np.zeros(1 << 16, np.uint8)
        ms, counts = (C.c_float * 64)(), (C.c_int * 64)()
        for rc in (lib.mvsv_tm(ctx, buf.ctypes.data, FW, buf.ctypes.data, FW, 0, 1, 3, buf.ctypes.data, FW),
                   lib.mvsv_debug_read(ctx, 2, buf.ctypes.data, buf.nbytes),
                   lib.mvsv_debug_set_flags(ctx, 1),
                   lib.mvsv_debug_postfilter(ctx, buf.ctypes.data, FW * 2, 1, 1, 0, 0, 0, 0),
                   lib.mvsv_profile_enable(ctx, 1),
                   lib.mvsv_profile_read(ctx, ms, counts, 64)):
            assert rc == ERR_UNSUPPORTED
        assert "multi-device" in lib.mvsv_last_error(ctx).decode()
        assert e.stream is None


@pytest.mark.gpu
@pytest.mark.parametrize("devs", DEVICE_LISTS, ids=LIST_IDS)
def test_info_devices_and_aggregates(devs):
    n, mb = len(devs), max_batch(devs)
    cap = -(-mb // n)
    L, R = frames(mb, seed=40)
    with api.Engine(FW, FH, max_batch=mb, devices=devs) as e, api.Engine(FW, FH, max_batch=mb) as one:
        assert e.devices == devs
        assert one.devices == [0]
        first = np.zeros(1, np.int32)
        assert e._lib.mvsv_get_devices(e._ctx, first.ctypes.data, 1) == n and first[0] == devs[0]
        i = e.info
        assert (i.max_batch, i.device, i.last_batch, i.frame_width, i.width) == (n * cap, devs[0], 0, FW, FW)
        for eng in (e, one):
            eng.set_sgbm_params(**SGBM)
        fields = ("width", "height", "sgbm_minX1", "sgbm_W1", "sgbm_D", "sgbm_Dpad", "sgbm_npaths", "num_rois")
        assert [getattr(e.info, f) for f in fields] == [getattr(one.info, f) for f in fields]
        e.timer_start()
        e.compute(L, R, api.STAGE_SGBM)
        assert e.timer_stop() > 0
        e.sync()
        assert e.info.last_batch == mb
        one.compute(L, R, api.STAGE_SGBM)
        assert_same(e.download(mb), one.download(mb), "sgbm")
        # the launch count is the sum of the parts': engines of the parts' size computing the same shares
        launches = 0
        for k in range(n):
            a, b = k * mb // n, (k + 1) * mb // n
            if a < b:
                with api.Engine(FW, FH, max_batch=cap, device=devs[k]) as part:
                    part.set_sgbm_params(**SGBM)
                    part.compute(L[a:b], R[a:b], api.STAGE_SGBM)
                    launches += part.launch_count
        assert e.launch_count == launches > 0


@pytest.mark.gpu
def test_one_device_list_is_mvsv_init():
    L, R = frames(3, seed=50)
    with api.Engine(FW, FH, max_batch=3, devices=[0]) as e, api.Engine(FW, FH, max_batch=3) as one:
        assert e.devices == [0] and e.stream is not None
        for eng in (e, one):
            eng.set_sgbm_params(**SGBM)
            eng.compute(L, R, api.STAGE_SGBM)
        assert_same(e.download(3), one.download(3), "sgbm")


@pytest.mark.gpu
def test_pinned_host_buffers():
    """mvsv_host_alloc memory is pinned for every device (unified addressing makes it portable), and a compute from it
    followed by a download into it gives what one engine gives"""
    torch = pytest.importorskip("torch")
    mb = 7
    L, R = frames(mb, seed=60)
    bufs = [api.pinned((mb, FH, FW), np.uint8) for _ in range(2)] + [api.pinned((mb, FH, FW), np.int16)]
    for d in range(max(NDEV, 1)):
        with torch.cuda.device(d):
            assert all(torch.from_numpy(b.array).is_pinned() for b in bufs), d
    bufs[0].array[:], bufs[1].array[:] = L, R
    with api.Engine(FW, FH, max_batch=mb, devices=[0, 0, 0]) as e, api.Engine(FW, FH, max_batch=mb) as one:
        for eng in (e, one):
            eng.set_sgbm_params(**SGBM)
        e.compute(bufs[0].array, bufs[1].array, api.STAGE_SGBM)
        e.download(mb, out={"disp": bufs[2].array})
        one.compute(L, R, api.STAGE_SGBM)
        assert np.array_equal(bufs[2].array, one.download(mb)["disp"])
    for b in bufs:
        b.close()


@pytest.mark.gpu
def test_init_devices_rejections():
    import ctypes as C
    lib = api.load_library()
    for devs, mb in (([], 4), ([0, 0, 0], 2), ([0, 4096], 4), ([-1, 0], 4), ([0, 0], 0)):
        ctx = C.c_void_p(1234)
        ids = np.array(devs, np.int32)
        assert lib.mvsv_init_devices(ids.ctypes.data if devs else None, len(devs), FW, FH, mb, C.byref(ctx)) == ERR_INVALID
        assert not ctx.value, devs
    ctx = C.c_void_p(1234)
    assert lib.mvsv_init_devices(None, 2, FW, FH, 4, C.byref(ctx)) == ERR_INVALID and not ctx.value
    ids = np.array([0, 4096], np.int32)
    assert lib.mvsv_init_devices(ids.ctypes.data, 2, FW, FH, 4, C.byref(ctx)) == ERR_INVALID and not ctx.value
    assert "part 1 (device 4096)" in lib.mvsv_last_error(None).decode()


def test_init_devices_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(api.MvsvError) as e:
        api.Engine(FW, FH, max_batch=4, devices=[0, 0])
    assert e.value.code == ERR_CUDA and "no CPU fallback" in str(e.value)
    lib = api.load_library()
    assert lib.mvsv_get_devices(None, None, 0) == ERR_INVALID
