"""Several stereo rigs in one batch (mvsv_set_frame_rigs): every frame is rectified with its own rig's maps and
reprojected with its own rig's Q, and gives what a single-rig engine holding that rig's calibration gives, bit for bit.

Four rigs from perturbed versions of the reference's calibrations (tests/golden/calibrations.json), rectified with
cv2.stereoRectify; all share one ROI size, placed at a different offset inside each rig's display ROI."""
import json
import os

import numpy as np
import pytest

import cases
from mvstereovision3_b200 import api, synth

with open(os.path.join(cases.GOLDEN_DIR, "calibrations.json")) as f:
    CAL = json.load(f)["rigs"]

FW, FH = 752, 480
MAXB = 48
RIG_IDS = (0, 5, 17, 63)             # engine rig of calibration k
SGBM = dict(minDisp=1, numDisp=64, blockSize=13, disp12MaxDiff=0, preFilterCap=0, uniquenessRatio=0,
            speckleWindowSize=150, speckleRange=2, disparityMode=0)
BM = dict(numDisp=64, blockSize=21, preFilterCap=31, textureThreshold=10, uniquenessRatio=15)
ERR_INVALID, ERR_STATE = -1, -4


def _perturbed(name, seed):
    """cv2.stereoRectify of a calibration near one of the reference's: (K, D, R, P) per camera, Q, display ROI."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(seed)
    r = CAL[name]
    KL, KR = np.array(r["KL"]), np.array(r["KR"])
    for K in (KL, KR):
        K[0, 0] *= 1 + rng.uniform(-0.04, 0.04)
        K[1, 1] *= 1 + rng.uniform(-0.04, 0.04)
        K[0, 2] += rng.uniform(-15, 15)
        K[1, 2] += rng.uniform(-15, 15)
    DL = np.array(r["DL"]) * rng.uniform(0.5, 1.5, 5)
    DR = np.array(r["DR"]) * rng.uniform(0.5, 1.5, 5)
    rv, _ = cv2.Rodrigues(np.array(r["R"]))
    R, _ = cv2.Rodrigues(rv + rng.uniform(-0.01, 0.01, (3, 1)))
    T = np.array(r["T"]).reshape(3, 1) * rng.uniform(0.8, 1.2)
    R0, R1, P0, P1, Q, roi0, roi1 = cv2.stereoRectify(KL, DL, KR, DR, (FW, FH), R, T, flags=cv2.CALIB_ZERO_DISPARITY,
                                                      alpha=0, newImageSize=(FW, FH))
    x0, y0 = max(roi0[0], roi1[0]), max(roi0[1], roi1[1])
    x1, y1 = min(roi0[0] + roi0[2], roi1[0] + roi1[2]), min(roi0[1] + roi0[3], roi1[1] + roi1[3])
    return [(KL, DL, R0, P0), (KR, DR, R1, P1)], Q.astype(np.float32), (x0, y0, x1 - x0, y1 - y0)


@pytest.fixture(scope="module")
def rigs():
    cv2 = pytest.importorskip("cv2")
    out = []
    for k in range(4):
        cams, Q, droi = _perturbed(sorted(CAL)[k % len(CAL)], 300 + k)
        out.append(dict(cams=cams, Q=Q, droi=droi))
    w = min(r["droi"][2] for r in out) - 30
    h = min(r["droi"][3] for r in out) - 20
    assert w >= 300 and h >= 200, [r["droi"] for r in out]
    for k, r in enumerate(out):
        dx, dy, dw, dh = r["droi"]
        r["roi"] = (dx + (3 + 9 * k) % (dw - w + 1), dy + (2 + 6 * k) % (dh - h + 1), w, h)
        r["maps"] = [cv2.initUndistortRectifyMap(K, D, R, P, (FW, FH), cv2.CV_32FC1) for K, D, R, P in r["cams"]]
    assert len({r["roi"][:2] for r in out}) == 4
    return out


@pytest.fixture(scope="module")
def frames():
    raw = [synth.stereogram(FH, FW, 1, 64, seed=40 + i)[:2] for i in range(MAXB)]
    return np.stack([x[0] for x in raw]), np.stack([x[1] for x in raw])


def install(e, rig, r, how):
    for cam in range(2):
        if how == "device":
            K, D, R, P = r["cams"][cam]
            e.set_rectification(cam, K, D, R, P, r["roi"], rig=rig)
        else:
            e.upload_rectify_maps(cam, *r["maps"][cam], r["roi"], rig=rig)
    e.set_Q(r["Q"], rig=rig)


# Tables of calibration indices (-> RIG_IDS) and the batch they are computed with.  Frames past a table come from rig 0.
def _table(name):
    if name == "unsorted":              # all four rigs, groups of 17, 9, 8 and 7 frames around the 8-frame remap chunks
        t = np.random.default_rng(1).permutation([3] * 17 + [1] * 9 + [2] * 8 + [0] * 7)
        return [int(v) for v in t], 41
    if name == "short":                 # a rig of one frame; calibration 3 (rig 63) installed but unused; rig 0 past the table
        return [1, 1, 0, 1, 2, 1, 1, 0, 1, 1, 1], 30
    if name == "long":                  # a table of max_batch frames, computed with a batch of 20
        return [int(v) for v in np.random.default_rng(2).integers(0, 4, MAXB)], 20
    raise KeyError(name)


def rig_of_frames(t, batch):
    """calibration index of every frame of the batch"""
    return [t[i] if i < len(t) else 0 for i in range(batch)]


def setup(e, matcher, resize):
    if resize:
        e.set_resize(resize)
    if matcher == "sgbm":
        e.set_sgbm_params(**SGBM)
    else:
        e.set_bm_params(**BM)
    W, H = e.info.width, e.info.height
    e.set_mean_rois(api.subimage_rois(W, H) + api.samplepoint_rois(W, H))


STAGES = api.STAGE_RECTIFY | api.STAGE_XYZ | api.STAGE_MEANS


def stages_of(matcher):
    return STAGES | (api.STAGE_SGBM if matcher == "sgbm" else api.STAGE_BM)


def reference(rigs, how, L, R, cal, matcher, resize):
    """per frame: the outputs of a single-rig engine holding that frame's calibration as rig 0"""
    out = [None] * len(cal)
    for k in sorted(set(cal)):
        idx = [i for i, c in enumerate(cal) if c == k]
        with api.Engine(FW, FH, max_batch=len(idx)) as e:
            install(e, 0, rigs[k], how)
            setup(e, matcher, resize)
            e.compute(L[idx], R[idx], stages_of(matcher))
            o = e.download(len(idx), rect=True, xyz=True, means=True)
        for j, i in enumerate(idx):
            out[i] = {key: v[j] for key, v in o.items()}
    return out


def assert_frames_equal(got, want, cal):
    for i, w in enumerate(want):
        for key in ("rectL", "rectR", "disp", "means"):
            np.testing.assert_array_equal(got[key][i], w[key], err_msg="frame %d (calibration %d): %s" % (i, cal[i], key))
        # XYZ bit for bit, NaN payloads included
        assert np.array_equal(got["xyz"][i].view(np.uint32), w["xyz"].view(np.uint32)), "frame %d: xyz" % i


def assert_rectified_like_cv2(rigs, got, L, R, cal, resize):
    cv2 = pytest.importorskip("cv2")
    for i, k in enumerate(cal):
        x, y, w, h = rigs[k]["roi"]
        for key, img, (mx, my) in (("rectL", L[i], rigs[k]["maps"][0]), ("rectR", R[i], rigs[k]["maps"][1])):
            want = cv2.remap(img, mx, my, cv2.INTER_LINEAR)[y:y + h, x:x + w]
            if resize:
                want = cv2.resize(want, (0, 0), fx=resize, fy=resize)
            np.testing.assert_array_equal(got[key][i], want, err_msg="frame %d (calibration %d): %s" % (i, k, key))


def cv2_sgbm(l, r):
    cv2 = pytest.importorskip("cv2")
    m = cv2.StereoSGBM_create(minDisparity=SGBM["minDisp"], numDisparities=SGBM["numDisp"], blockSize=SGBM["blockSize"],
                              P1=0, P2=0, disp12MaxDiff=SGBM["disp12MaxDiff"], preFilterCap=SGBM["preFilterCap"],
                              uniquenessRatio=SGBM["uniquenessRatio"], speckleWindowSize=SGBM["speckleWindowSize"],
                              speckleRange=SGBM["speckleRange"], mode=cv2.STEREO_SGBM_MODE_SGBM)
    return m.compute(l, r)


def compute_rigs(e, rigs, how, L, R, table, batch, matcher, resize):
    for k, r in enumerate(rigs):
        install(e, RIG_IDS[k], r, how)
    setup(e, matcher, resize)
    e.set_frame_rigs([RIG_IDS[k] for k in table])
    e.compute(L[:batch], R[:batch], stages_of(matcher))
    return e.download(batch, rect=True, xyz=True, means=True)


CASES = [("device", "unsorted", "sgbm", 0), ("upload", "unsorted", "sgbm", 0), ("device", "short", "sgbm", 0),
         ("upload", "long", "sgbm", 0), ("device", "unsorted", "sgbm", 0.5), ("upload", "short", "sgbm", 0.5),
         ("device", "unsorted", "bm", 0), ("upload", "long", "bm", 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("how,table,matcher,resize", CASES)
def test_rigs_equal_single_rig_engines(rigs, frames, how, table, matcher, resize):
    L, R = frames
    t, batch = _table(table)
    cal = rig_of_frames(t, batch)
    with api.Engine(FW, FH, max_batch=MAXB) as e:
        got = compute_rigs(e, rigs, how, L, R, t, batch, matcher, resize)
        launches = e.launch_count
    assert launches > 0
    assert_rectified_like_cv2(rigs, got, L, R, cal, resize)
    assert_frames_equal(got, reference(rigs, how, L[:batch], R[:batch], cal, matcher, resize), cal)
    if matcher == "sgbm" and not resize:
        # a frame of each rig the batch holds (the first one) against cv2 on the cv2-rectified pair
        for k in sorted(set(cal))[:3]:
            i = cal.index(k)
            np.testing.assert_array_equal(got["disp"][i], cv2_sgbm(got["rectL"][i], got["rectR"][i]))


@pytest.mark.gpu
def test_rigs_device_inputs(rigs, frames):
    torch = pytest.importorskip("torch")
    L, R = frames
    t, batch = _table("unsorted")
    cal = rig_of_frames(t, batch)
    dl, dr = torch.from_numpy(L[:batch]).cuda(), torch.from_numpy(R[:batch]).cuda()
    with api.Engine(FW, FH, max_batch=MAXB) as e:
        for k, r in enumerate(rigs):
            install(e, RIG_IDS[k], r, "device")
        setup(e, "sgbm", 0)
        e.set_frame_rigs([RIG_IDS[k] for k in t])
        torch.cuda.synchronize()
        e.compute_device(dl.data_ptr(), FW, dr.data_ptr(), FW, FH * FW, batch, stages_of("sgbm"))
        got = e.download(batch, rect=True, xyz=True, means=True)
    assert_frames_equal(got, reference(rigs, "device", L[:batch], R[:batch], cal, "sgbm", 0), cal)


@pytest.mark.gpu
def test_rigs_two_io_slots_table_changed_between_computes(rigs, frames):
    """a compute keeps the assignment it was submitted with: the table changes while the first one's results wait"""
    L, R = frames
    ta, ba = _table("unsorted")
    tb, bb = _table("short")
    with api.Engine(FW, FH, max_batch=MAXB) as e:
        e.set_io_slots(2)
        for k, r in enumerate(rigs):
            install(e, RIG_IDS[k], r, "upload")
        setup(e, "sgbm", 0)
        e.set_frame_rigs([RIG_IDS[k] for k in ta])
        e.compute(L[:ba], R[:ba], stages_of("sgbm"))
        e.set_frame_rigs([RIG_IDS[k] for k in tb])
        e.compute(L[MAXB - bb:], R[MAXB - bb:], stages_of("sgbm"))
        got_a = e.download(ba, rect=True, xyz=True, means=True, age=1)
        got_b = e.download(bb, rect=True, xyz=True, means=True)
    cal_a, cal_b = rig_of_frames(ta, ba), rig_of_frames(tb, bb)
    assert_frames_equal(got_a, reference(rigs, "upload", L[:ba], R[:ba], cal_a, "sgbm", 0), cal_a)
    assert_frames_equal(got_b, reference(rigs, "upload", L[MAXB - bb:], R[MAXB - bb:], cal_b, "sgbm", 0), cal_b)


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", ((37, 5), (64, 48)))
def test_rigs_debug_postfilter_xyz(rigs, W, H):
    """XYZ of caller-supplied maps (no rectification): each pixel with its frame's Q, also where a thread's four pixels
    cross a frame boundary (37 x 5 = 185 pixels per frame)"""
    B = 21
    rng = np.random.default_rng(W)
    maps = rng.integers(-40, 1100, (B, H, W)).astype(np.int16)
    t = [3, 0, 1, 1, 2, 3, 3, 1, 0, 2, 2, 2, 1, 3, 0, 1]            # frames 16..20: rig 0
    cal = rig_of_frames(t, B)
    with api.Engine(W, H, max_batch=B) as e:
        for k, r in enumerate(rigs):
            e.set_Q(r["Q"], rig=RIG_IDS[k])
        e.set_frame_rigs([RIG_IDS[k] for k in t])
        e.debug_postfilter(maps, median=False, stages=api.STAGE_XYZ)
        got = e.download(B, disp=False, xyz=True)["xyz"]
    for k in sorted(set(cal)):
        idx = [i for i, c in enumerate(cal) if c == k]
        with api.Engine(W, H, max_batch=B) as e:
            e.set_Q(rigs[k]["Q"])
            e.debug_postfilter(maps[idx], median=False, stages=api.STAGE_XYZ)
            want = e.download(len(idx), disp=False, xyz=True)["xyz"]
        assert np.array_equal(got[idx].view(np.uint32), want.view(np.uint32)), k


@pytest.mark.gpu
def test_rigs_rejections(rigs, frames):
    L, R = frames
    r0, r1, r2 = rigs[:3]
    with api.Engine(FW, FH, max_batch=8) as e:
        for bad in (-1, api.MAX_RIGS):
            for call in (lambda: e.set_Q(r0["Q"], rig=bad),
                         lambda: install(e, bad, r0, "device"),
                         lambda: install(e, bad, r0, "upload"),
                         lambda: e.set_frame_rigs([0, bad])):
                with pytest.raises(api.MvsvError) as ei:
                    call()
                assert ei.value.code == ERR_INVALID
        with pytest.raises(api.MvsvError) as ei:
            e.set_frame_rigs([0] * 9)                                 # more frames than max_batch
        assert ei.value.code == ERR_INVALID

        install(e, 0, r0, "device")
        x, y, w, h = r1["roi"]
        K, D, Rm, P = r1["cams"][0]
        with pytest.raises(api.MvsvError) as ei:
            e.set_rectification(0, K, D, Rm, P, (x, y, w - 2, h), rig=5)      # another ROI size than rig 0's
        assert ei.value.code == ERR_INVALID
        with pytest.raises(api.MvsvError) as ei:
            e.upload_rectify_maps(1, *r1["maps"][1], (x, y, w, h - 1), rig=5)
        assert ei.value.code == ERR_INVALID
        e.set_rectification(0, K, D, Rm, P, r1["roi"], rig=5)                 # camera 0 of rig 5 only
        with pytest.raises(api.MvsvError) as ei:
            e.set_rectification(1, *r1["cams"][1], (x + 1, y, w, h), rig=5)   # both cameras of a rig share its ROI
        assert ei.value.code == ERR_INVALID
        with pytest.raises(api.MvsvError) as ei:
            e.set_rectification(0, *r2["cams"][0], (x, y, w + 1, h), rig=17)    # rigs 0 and 5 hold maps of another size
        assert ei.value.code == ERR_INVALID

        setup(e, "sgbm", 0)
        st = stages_of("sgbm")
        e.compute(L[:4], R[:4], st)                                   # rig 0 only
        before = e.download(4, rect=True, xyz=True, means=True)

        def rejected(table, stages):
            e.set_frame_rigs(table)
            with pytest.raises(api.MvsvError) as ei:
                e.compute(L[4:8], R[4:8], stages)
            assert ei.value.code == ERR_STATE
            after = e.download(4, rect=True, xyz=True, means=True)      # the earlier results, untouched
            for key in before:
                assert np.array_equal(after[key].view(np.uint8), before[key].view(np.uint8)), key

        rejected([0, 5, 0, 0], st & ~api.STAGE_XYZ)    # rig 5: camera 1 has no map
        rejected([0, 0, 0, 9], st)                     # rig 9: nothing installed
        e.set_rectification(1, *r1["cams"][1], r1["roi"], rig=5)
        rejected([0, 5, 0, 0], st)                     # rig 5: maps, but no Q
        e.set_frame_rigs([0, 5, 0, 0])
        e.compute(L[4:8], R[4:8], st & ~api.STAGE_XYZ)  # without XYZ rig 5 needs no Q
        e.set_Q(r1["Q"], rig=5)
        e.compute(L[4:8], R[4:8], st)
        e.set_frame_rigs([5, 5, 5])                    # frames past the table: rig 0
        e.compute(L[:4], R[:4], st)
        e.set_frame_rigs([])
        e.compute(L[:4], R[:4], st)
        np.testing.assert_array_equal(e.download(4)["disp"], before["disp"])

        e.reset_rectification()                        # drops the maps of every rig
        assert (e.info.width, e.info.height) == (FW, FH)
        e.set_frame_rigs([5])
        with pytest.raises(api.MvsvError) as ei:
            e.compute(L[:1], R[:1], api.STAGE_RECTIFY)
        assert ei.value.code == ERR_STATE


def test_rig_calls_without_engine():
    lib = api.load_library()
    q = np.zeros(16, np.float32)
    assert lib.mvsv_set_Q_rig(None, 0, q.ctypes.data) == ERR_INVALID
    assert lib.mvsv_set_frame_rigs(None, None, 0) == ERR_INVALID
    assert lib.mvsv_upload_rectify_maps_rig(None, 0, 0, None, None, 0, 0, 0, 2, 1) == ERR_INVALID
    assert lib.mvsv_set_rectification_rig(None, 0, 0, None, None, 0, None, None, 0, 0, 2, 1) == ERR_INVALID
