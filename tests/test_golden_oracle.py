"""CPU: the C oracle against the committed cv2 4.13.0 golden vectors (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest

import cases


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(cases.GOLDEN_DIR, "cv2_golden.npz"))


@pytest.mark.parametrize("case", cases.SGBM_CASES, ids=[c[0] for c in cases.SGBM_CASES])
def test_sgbm_oracle_vs_golden(oracle, golden, case):
    name, p, H, W = case
    for kind in ("ramp", "noise"):
        l, r = cases.sgbm_inputs(name, p, H, W, kind)
        np.testing.assert_array_equal(oracle.sgbm(l, r, p), golden["sgbm/%s/%s" % (name, kind)])


@pytest.mark.parametrize("case", cases.BM_CASES, ids=[c[0] for c in cases.BM_CASES])
def test_bm_oracle_vs_golden(oracle, golden, case):
    name, p, H, W = case
    for kind in ("ramp", "noise"):
        l, r = cases.bm_inputs(name, p, H, W, kind)
        np.testing.assert_array_equal(oracle.bm(l, r, p), golden["bm/%s/%s" % (name, kind)])


def test_remap_median_speckle_xyz_vs_golden(oracle, golden):
    for seed in range(3):
        img, _ = cases.synth.random_pair(96, 140, seed=seed)
        mx, my = cases.warp_maps(96, 140, seed)
        np.testing.assert_array_equal(oracle.remap(img, mx, my), golden["remap/%d" % seed])
    d = golden["median/in"]
    np.testing.assert_array_equal(oracle.median3(d), golden["median/out"])
    np.testing.assert_array_equal(oracle.speckle(d, -16, 9, 32), golden["speckle/out"])
    disp = golden["xyz/in"]
    xyz, valid = oracle.reproject(disp, cases.Q_REFERENCE)
    v = valid.astype(bool)
    np.testing.assert_allclose(xyz[v], golden["xyz/out"][v], rtol=1e-5)   # north_star: 1e-5 relative for float XYZ


def test_rectify_fixture(oracle):
    g = cases.synth.load_rectification(cases.GOLDEN_DIR)
    roi = tuple(int(v) for v in g["roi"])
    assert roi == (0, 0, 752, 479)          # SURVEY.md 8c: baseline_small yields a 752x479 display ROI
    l, r, _ = cases.synth.stereogram(480, 752, 1, 64, seed=7)
    np.testing.assert_array_equal(oracle.remap(l, g["m1x"], g["m1y"], roi), g["rectL"])
    np.testing.assert_array_equal(oracle.remap(r, g["m2x"], g["m2y"], roi), g["rectR"])
