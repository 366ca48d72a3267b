"""Generates tests/golden/*.npz from cv2 4.13.0 -- the OpenCV build standing in for the un-vendored OpenCV the
reference calls (src/disparity.cpp:8,20; src/Stereosystem.cpp:210-217,252-253).  Inputs are re-created from
seeds by tests/cases.py; only cv2's OUTPUTS are stored.  Run from the repo root:  python tests/golden/make_golden.py
(`... make_golden.py rectify` writes the rectification fixture alone)."""
import json
import os
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402

OUT = cases.GOLDEN_DIR


def cv_sgbm(l, r, p):
    m = cv2.StereoSGBM_create(minDisparity=p["minDisp"], numDisparities=p["numDisp"], blockSize=p["blockSize"],
                              P1=p["P1"], P2=p["P2"], disp12MaxDiff=p["disp12MaxDiff"], preFilterCap=p["preFilterCap"],
                              uniquenessRatio=p["uniquenessRatio"], speckleWindowSize=p["speckleWindowSize"],
                              speckleRange=p["speckleRange"],
                              mode=cv2.STEREO_SGBM_MODE_HH if p["mode"] == 1 else cv2.STEREO_SGBM_MODE_SGBM)
    return m.compute(l, r)


def cv_bm(l, r, p):
    m = cv2.StereoBM_create(numDisparities=p["numDisp"], blockSize=p["blockSize"])
    m.setPreFilterCap(p["preFilterCap"])
    m.setUniquenessRatio(p["uniquenessRatio"])
    m.setTextureThreshold(p["textureThreshold"])
    return m.compute(l, r)


def main():
    out = {}
    for name, p, H, W in cases.SGBM_CASES:
        for kind in ("ramp", "noise"):
            l, r = cases.sgbm_inputs(name, p, H, W, kind)
            out["sgbm/%s/%s" % (name, kind)] = cv_sgbm(l, r, p)
    for name, p, H, W in cases.BM_CASES:
        for kind in ("ramp", "noise"):
            l, r = cases.bm_inputs(name, p, H, W, kind)
            out["bm/%s/%s" % (name, kind)] = cv_bm(l, r, p)
    for seed in range(3):
        H, W = 96, 140
        img, _ = cases.synth.random_pair(H, W, seed=seed)
        mx, my = cases.warp_maps(H, W, seed)
        out["remap/%d" % seed] = cv2.remap(img, mx, my, cv2.INTER_LINEAR)
    rng = np.random.default_rng(11)
    d = (rng.integers(-2, 40, size=(41, 67)) * 16).astype(np.int16)
    out["median/in"] = d
    out["median/out"] = cv2.medianBlur(d, 3)
    s = d.copy()
    cv2.filterSpeckles(s, -16, 9, 32)
    out["speckle/out"] = s
    disp = rng.integers(-16, 64 * 16, size=(40, 60)).astype(np.int16)
    out["xyz/in"] = disp
    out["xyz/out"] = cv2.reprojectImageTo3D(disp.astype(np.float32) / 16, cases.Q_REFERENCE)
    np.savez_compressed(os.path.join(OUT, "cv2_golden.npz"), **out)

    rectify_fixture()


def rectify_fixture():
    """Rectification maps of the reference's parameters/baseline_small calibration (src/Stereosystem.cpp:193-242),
    whose numbers calibrations.json holds.  The maps are written delta-coded (synth.encode_map) to a file of their
    own: as floats they would not compress below 1 MB."""
    with open(os.path.join(OUT, "calibrations.json")) as f:
        cal = {k: np.array(v) for k, v in json.load(f)["rigs"]["baseline_small"].items() if k != "modes"}
    KL, KR, DL, DR, R, T = (cal[k] for k in ("KL", "KR", "DL", "DR", "R", "T"))
    size = (752, 480)
    R0, R1, P0, P1, Q, roi0, roi1 = cv2.stereoRectify(KL, DL, KR, DR, size, R, T.reshape(3, 1),
                                                      flags=cv2.CALIB_ZERO_DISPARITY, alpha=0, newImageSize=size)
    m1x, m1y = cv2.initUndistortRectifyMap(KL, DL, R0, P0, size, cv2.CV_32FC1)
    m2x, m2y = cv2.initUndistortRectifyMap(KR, DR, R1, P1, size, cv2.CV_32FC1)
    x0, y0 = max(roi0[0], roi1[0]), max(roi0[1], roi1[1])
    x1 = min(roi0[0] + roi0[2], roi1[0] + roi1[2])
    y1 = min(roi0[1] + roi0[3], roi1[1] + roi1[3])
    roi = np.array([x0, y0, x1 - x0, y1 - y0], np.int32)
    print("display ROI", roi)
    l, r, _ = cases.synth.stereogram(480, 752, 1, 64, seed=7)
    rl = cv2.remap(l, m1x, m1y, cv2.INTER_LINEAR)[y0:y1, x0:x1]
    rr = cv2.remap(r, m2x, m2y, cv2.INTER_LINEAR)[y0:y1, x0:x1]
    np.savez_compressed(os.path.join(OUT, "rectify_baseline_small.npz"), roi=roi, Q=Q.astype(np.float32),
                        rectL=rl, rectR=rr)
    maps = dict(m1x=m1x, m1y=m1y, m2x=m2x, m2y=m2y)
    np.savez_compressed(os.path.join(OUT, "rectify_baseline_small_maps.npz"),
                        **{k: cases.synth.encode_map(v) for k, v in maps.items()})


if __name__ == "__main__":
    rectify_fixture() if sys.argv[1:] == ["rectify"] else main()
