"""Rectification-map generation (SURVEY section 8f row f3): cv::initUndistortRectifyMap of
Stereosystem::initRectification (reference src/Stereosystem.cpp:214-217) restated in the oracle and built on the
device by mvsv_set_rectification.  The yardstick is the fixed-point form rint(map * 32) that cv::remap consumes:
it must be identical to cv2 4.13's for the reference's three calibrations (tests/golden/calibrations.json)."""
import json
import os
import zlib

import numpy as np
import pytest

import cases

with open(os.path.join(cases.GOLDEN_DIR, "calibrations.json")) as f:
    CAL = json.load(f)["rigs"]
RIGS = sorted(CAL)
MODES = ("full", "binned")


def cameras(rig, mode):
    """[(K, D, R, P)] for left, right as initRectification passes them (camera matrices halved when binned)."""
    r, m = CAL[rig], CAL[rig]["modes"][mode]
    s = 0.5 if mode == "binned" else 1.0
    return [(np.array(r["KL"]) * s, np.array(r["DL"]), np.array(m["R0"]), np.array(m["P0"])),
            (np.array(r["KR"]) * s, np.array(r["DR"]), np.array(m["R1"]), np.array(m["P1"]))], tuple(m["size"]), m


def fixed(mx, my):
    return np.stack([np.rint(mx * np.float32(32)), np.rint(my * np.float32(32))], -1).astype(np.int32)


def perturbed(rig, seed):
    """A calibration near one of the reference's: jittered intrinsics/distortion and a small extra rotation."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(seed)
    r = CAL[rig]
    KL, KR = np.array(r["KL"]), np.array(r["KR"])
    for K in (KL, KR):
        K[0, 0] *= 1 + rng.uniform(-0.05, 0.05)
        K[1, 1] *= 1 + rng.uniform(-0.05, 0.05)
        K[0, 2] += rng.uniform(-20, 20)
        K[1, 2] += rng.uniform(-20, 20)
    DL = np.array(r["DL"]) * rng.uniform(0.5, 1.5, 5)
    DR = np.array(r["DR"]) * rng.uniform(0.5, 1.5, 5)
    rv, _ = cv2.Rodrigues(np.array(r["R"]))
    R, _ = cv2.Rodrigues(rv + rng.uniform(-0.01, 0.01, (3, 1)))
    T = np.array(r["T"]).reshape(3, 1) * rng.uniform(0.8, 1.2)
    size = (752, 480)
    R0, R1, P0, P1, Q, roi0, roi1 = cv2.stereoRectify(KL, DL, KR, DR, size, R, T, flags=cv2.CALIB_ZERO_DISPARITY, alpha=0,
                                                      newImageSize=size)
    return [(KL, DL, R0, P0), (KR, DR, R1, P1)], size


# ------------------------------------------------------------------------------------------ oracle (CPU)
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("rig", RIGS)
def test_oracle_maps_match_committed_crc(oracle, rig, mode):
    cams, size, m = cameras(rig, mode)
    for (K, D, R, P), key in zip(cams, ("crc_fixed_left", "crc_fixed_right")):
        mx, my = oracle.rectify_maps(K, D, R, P, size)
        assert mx.shape == (size[1], size[0])
        assert zlib.crc32(np.ascontiguousarray(fixed(mx, my)).tobytes()) == m[key], (rig, mode, key)


def test_oracle_maps_match_committed_float_maps(oracle):
    """the float maps committed for parameters/baseline_small (the fixture of the remap tests)"""
    g = cases.synth.load_rectification(cases.GOLDEN_DIR)
    cams, size, _ = cameras("baseline_small", "full")
    for (K, D, R, P), kx, ky in zip(cams, ("m1x", "m2x"), ("m1y", "m2y")):
        mx, my = oracle.rectify_maps(K, D, R, P, size)
        np.testing.assert_array_equal(fixed(mx, my), fixed(g[kx], g[ky]))
        assert np.mean((mx == g[kx]) & (my == g[ky])) > 0.9999     # float maps: equal up to isolated last-bit cases
        np.testing.assert_allclose(mx, g[kx], rtol=0, atol=1e-4)
        np.testing.assert_allclose(my, g[ky], rtol=0, atol=1e-4)


@pytest.mark.parametrize("seed", range(4))
def test_oracle_maps_match_cv2_on_perturbed_calibrations(oracle, seed):
    cv2 = pytest.importorskip("cv2")
    cams, size = perturbed(RIGS[seed % len(RIGS)], seed)
    for K, D, R, P in cams:
        mx, my = oracle.rectify_maps(K, D, R, P, size)
        cx, cy = cv2.initUndistortRectifyMap(K, D, R, P, size, cv2.CV_32FC1)
        np.testing.assert_array_equal(fixed(mx, my), fixed(cx, cy))


def test_oracle_maps_identity():
    """K == P[:, :3], no distortion, R = I  ->  the identity map"""
    from oracle import loader
    K = np.array([[400.0, 0, 100.5], [0, 410.0, 60.25], [0, 0, 1]])
    P = np.hstack([K, np.zeros((3, 1))])
    mx, my = loader.rectify_maps(K, np.zeros(5), np.eye(3), P, (200, 120))
    np.testing.assert_allclose(mx, np.tile(np.arange(200, dtype=np.float32), (120, 1)), atol=1e-4)
    np.testing.assert_allclose(my, np.tile(np.arange(120, dtype=np.float32)[:, None], (1, 200)), atol=1e-4)


# ------------------------------------------------------------------------------------------ device
@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("rig", RIGS)
def test_device_maps_match_cv2(oracle, rig, mode):
    from mvstereovision3_b200 import api
    cams, size, m = cameras(rig, mode)
    roi = m["display_roi"]
    with api.Engine(size[0], size[1]) as e:
        for cam, (K, D, R, P) in enumerate(cams):
            e.set_rectification(cam, K, D, R, P, roi)
        assert (e.info.width, e.info.height) == (roi[2], roi[3])
        for cam, ((K, D, R, P), key) in enumerate(zip(cams, ("crc_fixed_left", "crc_fixed_right"))):
            got = e.read_rectify_map(cam, roi)
            mx, my = oracle.rectify_maps(K, D, R, P, size)
            want = fixed(mx, my)        # == cv2's (test_oracle_maps_match_committed_crc)
            assert zlib.crc32(np.ascontiguousarray(want).tobytes()) == m[key]
            np.testing.assert_array_equal(got, want[roi[1]:roi[1] + roi[3], roi[0]:roi[0] + roi[2]])


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_device_maps_match_cv2_live(seed):
    cv2 = pytest.importorskip("cv2")
    from mvstereovision3_b200 import api
    cams, size = perturbed(RIGS[seed % len(RIGS)], 100 + seed)
    roi = (8, 5, size[0] - 19, size[1] - 11)            # a display ROI that is not the full frame
    with api.Engine(size[0], size[1]) as e:
        for cam, (K, D, R, P) in enumerate(cams):
            e.set_rectification(cam, K, D[:4] if seed == 1 else D, R, P, roi)
            cx, cy = cv2.initUndistortRectifyMap(K, D[:4] if seed == 1 else D, R, P, size, cv2.CV_32FC1)
            np.testing.assert_array_equal(e.read_rectify_map(cam, roi),
                                          fixed(cx, cy)[roi[1]:roi[1] + roi[3], roi[0]:roi[0] + roi[2]])


@pytest.mark.gpu
def test_pipeline_with_device_maps_equals_uploaded_maps():
    """raw pair -> rectify -> SGBM: building the maps on the device gives the same images and disparities as
    uploading the committed cv2 float maps (Stereosystem::getRectifiedImagepair, src/Stereosystem.cpp:244-277)."""
    from mvstereovision3_b200 import api, synth
    g = synth.load_rectification(cases.GOLDEN_DIR)
    cams, size, m = cameras("baseline_small", "full")
    roi = tuple(int(v) for v in g["roi"])
    assert list(roi) == m["display_roi"]
    l, r, _ = synth.stereogram(480, 752, 1, 64, seed=7)
    p = dict(minDisp=1, numDisp=64, blockSize=13, speckleWindowSize=150, speckleRange=2)
    outs = []
    for device_maps in (False, True):
        with api.Engine(752, 480) as e:
            if device_maps:
                for cam, (K, D, R, P) in enumerate(cams):
                    e.set_rectification(cam, K, D, R, P, roi)
            else:
                e.upload_rectify_maps(0, g["m1x"], g["m1y"], roi)
                e.upload_rectify_maps(1, g["m2x"], g["m2y"], roi)
            e.set_sgbm_params(**p)
            e.compute(l, r, api.STAGE_RECTIFY | api.STAGE_SGBM)
            outs.append(e.download(1, rect=True))
    np.testing.assert_array_equal(outs[1]["rectL"][0], g["rectL"])
    np.testing.assert_array_equal(outs[1]["rectR"][0], g["rectR"])
    for k in ("rectL", "rectR", "disp"):
        np.testing.assert_array_equal(outs[0][k], outs[1][k])


@pytest.mark.gpu
def test_set_rectification_errors():
    from mvstereovision3_b200 import api
    cams, size, m = cameras("smallBL", "full")
    K, D, R, P = cams[0]
    with api.Engine(size[0], size[1]) as e:
        with pytest.raises(api.MvsvError) as ei:
            e.set_rectification(0, K, np.zeros(8), R, P, m["display_roi"])       # rational model: not the reference's
        assert ei.value.code == -5
        with pytest.raises(api.MvsvError):
            e.set_rectification(0, K, D, R, np.zeros((3, 4)), m["display_roi"])  # singular projection
        with pytest.raises(api.MvsvError):
            e.set_rectification(0, K, D, R, P, (0, 0, size[0] + 1, size[1]))     # ROI outside the frame
        with pytest.raises(api.MvsvError):
            e.read_rectify_map(0, m["display_roi"])                               # nothing installed yet
        e.set_rectification(0, K, D, R, P, m["display_roi"])
        with pytest.raises(api.MvsvError):
            e.set_rectification(1, K, D, R, P, (1, 1, 100, 100))                  # cameras must share the display ROI


# ------------------------------------------------------------------------------------------ resize(factor)
RESIZE_FACTORS = (0.5, 0.25, 0.75, 0.6, 1.5, 0.3333, 2.0, 0.9, 1.25, float(np.float32(0.7)))
RESIZE_SIZES = ((479, 752), (97, 131), (120, 200), (33, 50), (31, 47))


@pytest.mark.parametrize("size", RESIZE_SIZES)
def test_oracle_resize_matches_cv2(oracle, size):
    """Stereosystem::getRectifiedImagepair(sip, factor): cv::resize(.., Size(0,0), factor, factor), reference
    src/Stereosystem.cpp:294-295 (trgt/test.cpp:213 passes 0.5)"""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(size[0])
    img = rng.integers(0, 256, size, dtype=np.uint8)
    for f in RESIZE_FACTORS:
        want = cv2.resize(img, (0, 0), fx=f, fy=f)
        got = oracle.resize(img, f)
        assert got.shape == want.shape, (size, f)
        np.testing.assert_array_equal(got, want, err_msg="%s x %s" % (size, f))


@pytest.mark.gpu
@pytest.mark.parametrize("factor", (0.5, 0.75, 1.5, 0.3333))
def test_rectify_resize_sgbm_pipeline(oracle, factor):
    """raw pair -> remap -> crop -> resize(factor) -> SGBM, against the oracle chain and (resize) live cv2"""
    from mvstereovision3_b200 import api, synth
    g = synth.load_rectification(cases.GOLDEN_DIR)
    cams, size, m = cameras("baseline_small", "full")
    roi = m["display_roi"]
    B = 2
    raws = [synth.stereogram(480, 752, 1, 64, seed=20 + b)[:2] for b in range(B)]
    p = cases.sgbm_params(minDisp=1, numDisp=32, blockSize=9, speckleWindowSize=100, speckleRange=2)
    with api.Engine(752, 480, max_batch=B) as e:
        e.set_resize(factor)                                  # before the maps exist: takes effect once they do
        for cam, (K, D, R, P) in enumerate(cams):
            e.set_rectification(cam, K, D, R, P, roi)
        e.set_sgbm_params(**{k: v for k, v in p.items() if k != "mode"}, disparityMode=p["mode"])
        e.compute(np.stack([x[0] for x in raws]), np.stack([x[1] for x in raws]), api.STAGE_RECTIFY | api.STAGE_SGBM)
        out = e.download(B, rect=True)
        info = e.info
        for b in range(B):
            rl = oracle.resize(oracle.remap(raws[b][0], g["m1x"], g["m1y"], roi), factor)
            rr = oracle.resize(oracle.remap(raws[b][1], g["m2x"], g["m2y"], roi), factor)
            assert (info.height, info.width) == rl.shape
            np.testing.assert_array_equal(out["rectL"][b], rl)
            np.testing.assert_array_equal(out["rectR"][b], rr)
            np.testing.assert_array_equal(out["disp"][b], oracle.sgbm(rl, rr, p))
        try:
            import cv2
            full = cv2.remap(raws[0][0], g["m1x"], g["m1y"], cv2.INTER_LINEAR)[roi[1]:roi[1] + roi[3], roi[0]:roi[0] + roi[2]]
            np.testing.assert_array_equal(out["rectL"][0], cv2.resize(full, (0, 0), fx=factor, fy=factor))
        except ImportError:
            pass
        # switching the resize off restores the display-ROI geometry
        e.set_resize(0)
        assert (e.info.width, e.info.height) == (roi[2], roi[3])
        e.compute(raws[0][0], raws[0][1], api.STAGE_RECTIFY | api.STAGE_SGBM)
        o2 = e.download(1, rect=True)
        rl = oracle.remap(raws[0][0], g["m1x"], g["m1y"], roi)
        rr = oracle.remap(raws[0][1], g["m2x"], g["m2y"], roi)
        np.testing.assert_array_equal(o2["rectL"][0], rl)
        np.testing.assert_array_equal(o2["disp"][0], oracle.sgbm(rl, rr, p))


@pytest.mark.gpu
def test_resize_odd_roi_and_errors(oracle):
    """odd display ROI (clipped 2x2 blocks at the far edges) and argument checks"""
    from mvstereovision3_b200 import api, synth
    H, W = 97, 131
    mx, my = cases.warp_maps(H, W, 3)
    l, r = synth.random_pair(H, W, seed=5)
    roi = (0, 0, W, H)
    with api.Engine(W, H) as e:
        with pytest.raises(api.MvsvError):
            e.set_resize(100.0)
        with pytest.raises(api.MvsvError):
            e.set_resize(float("nan"))
        e.upload_rectify_maps(0, mx, my, roi)
        e.upload_rectify_maps(1, mx, my, roi)
        for f in (0.5, 0.6, 2.0):
            e.set_resize(f)
            e.compute(l, r, api.STAGE_RECTIFY)
            out = e.download(1, disp=False, rect=True)
            np.testing.assert_array_equal(out["rectL"][0], oracle.resize(oracle.remap(l, mx, my, roi), f))
            np.testing.assert_array_equal(out["rectR"][0], oracle.resize(oracle.remap(r, mx, my, roi), f))
        e.reset_rectification()
        assert (e.info.width, e.info.height) == (W, H)


@pytest.mark.gpu
def test_device_maps_4k_frame():
    """a 3840x2160 frame (BASELINE.json cfg 5 size) with the first rig's calibration scaled up: the device maps still
    equal cv2's fixed-point maps, and remap + crop through them equals cv2.remap"""
    cv2 = pytest.importorskip("cv2")
    from mvstereovision3_b200 import api
    r = CAL[RIGS[0]]
    s = 3840 / 752.0
    size = (3840, 2160)
    KL, KR = np.array(r["KL"]) * s, np.array(r["KR"]) * s
    KL[2, 2] = KR[2, 2] = 1.0
    DL, DR = np.array(r["DL"]), np.array(r["DR"])
    R0, R1, P0, P1, Q, roi0, roi1 = cv2.stereoRectify(KL, DL, KR, DR, size, np.array(r["R"]), np.array(r["T"]).reshape(3, 1),
                                                      flags=cv2.CALIB_ZERO_DISPARITY, alpha=0, newImageSize=size)
    x0, y0 = max(roi0[0], roi1[0]), max(roi0[1], roi1[1])
    x1, y1 = min(roi0[0] + roi0[2], roi1[0] + roi1[2]), min(roi0[1] + roi0[3], roi1[1] + roi1[3])
    roi = (x0, y0, x1 - x0, y1 - y0)
    rng = np.random.default_rng(4)
    raw = rng.integers(0, 256, (size[1], size[0]), dtype=np.uint8)
    with api.Engine(size[0], size[1]) as e:
        for cam, (K, D, R, P) in enumerate(((KL, DL, R0, P0), (KR, DR, R1, P1))):
            e.set_rectification(cam, K, D, R, P, roi)
            mx, my = cv2.initUndistortRectifyMap(K, D, R, P, size, cv2.CV_32FC1)
            np.testing.assert_array_equal(e.read_rectify_map(cam, roi), fixed(mx, my)[y0:y1, x0:x1])
        e.compute(raw, raw, api.STAGE_RECTIFY)
        out = e.download(1, disp=False, rect=True)
        np.testing.assert_array_equal(out["rectR"][0], cv2.remap(raw, mx, my, cv2.INTER_LINEAR)[y0:y1, x0:x1])
