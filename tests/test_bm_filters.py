"""StereoBM's post-filters: the left-right check (disp12MaxDiff) and the speckle filter (speckleWindowSize /
speckleRange): the reference (tests/bm_filters_ref.py, on top of the C oracle's StereoBM) against cv2 4.13.0, and the
GPU against the reference and cv2."""
import numpy as np
import pytest

import bm_filters_ref as ref
import cases
from mvstereovision3_b200 import api, synth

FILT = -16
STEREO_MATCH = dict(preFilterCap=31, textureThreshold=10, uniquenessRatio=15)     # OpenCV's stereo_match sample
STEREO_MATCH_FILTERS = dict(disp12MaxDiff=1, speckleWindowSize=100, speckleRange=32)
BM_YML = dict(numDisp=80, blockSize=21, preFilterCap=2, uniquenessRatio=0, textureThreshold=30)


def occluded_pair(H, W, D, seed):
    """A background plane at a small disparity, an occluding textured rectangle at D - 5 (its left edge is
    half-occluded in the right image: LR failures) and a few 5x5 noise patches in the left image (small islands)."""
    rng = np.random.default_rng(seed)
    dbg, dfg = max(2, D // 6), D - 5
    tex = synth._blur3(rng.integers(0, 256, size=(H, W + D + 8), dtype=np.uint8))
    fg = synth._blur3(rng.integers(0, 256, size=(H, W + D + 8), dtype=np.uint8))
    left = tex[:, :W].copy()
    right = tex[:, dbg:dbg + W].copy()
    y0, y1, x0, x1 = H // 4, 3 * H // 4, W // 3 + D // 2, 2 * W // 3 + D // 2
    left[y0:y1, x0:x1] = fg[y0:y1, x0:x1]
    right[y0:y1, x0 - dfg:x1 - dfg] = fg[y0:y1, x0:x1]
    for _ in range(6):
        yy, xx = rng.integers(0, H - 6), rng.integers(D, W - 6)
        left[yy:yy + 5, xx:xx + 5] = rng.integers(0, 256, size=(5, 5))
    n = rng.integers(-4, 5, size=right.shape)
    return left, np.clip(right.astype(np.int16) + n, 0, 255).astype(np.uint8)


def cv_bm(cv2, left, right, p):
    m = cv2.StereoBM_create(numDisparities=p["numDisp"], blockSize=p["blockSize"])
    m.setPreFilterCap(p["preFilterCap"])
    m.setUniquenessRatio(p["uniquenessRatio"])
    m.setTextureThreshold(p["textureThreshold"])
    m.setDisp12MaxDiff(p.get("disp12MaxDiff", -1))
    m.setSpeckleWindowSize(p.get("speckleWindowSize", 0))
    m.setSpeckleRange(p.get("speckleRange", 0))
    return m.compute(left, right)


def check(name, got, want):
    assert got.shape == want.shape, (name, got.shape, want.shape)
    n = int((got != want).sum())
    assert n == 0, "%s: %d pixels differ, first at %s" % (name, n, tuple(np.argwhere(got != want)[0]))


# ---- reference against cv2 (CPU) ------------------------------------------------------------------------------------
# cv2 4.13 runs its check on the exact cost only on its 16-bit path (preFilterCap <= 31 and blockSize <= 21); above
# that it reads its cost buffer in a layout its matcher does not write, and the result changes from run to run
# (DESIGN.md section 2).  The sweep stays on the deterministic path.
SWEEP = [(16, 5, 70, 200), (32, 9, 71, 180), (48, 15, 74, 203), (80, 21, 60, 230), (96, 7, 61, 240), (32, 21, 65, 181)]
SWEEP_BM = [(31, 10, 15), (2, 30, 0), (20, 0, 5)]      # preFilterCap, textureThreshold, uniquenessRatio
SPECKLE = [(50, 2), (100, 32), (150, 16)]              # speckleWindowSize, speckleRange


@pytest.mark.parametrize("D,bs,H,W", SWEEP, ids=["d%d_bs%d_h%d" % (D, bs, H) for D, bs, H, W in SWEEP])
def test_reference_filters_equal_cv2(oracle, D, bs, H, W):
    cv2 = pytest.importorskip("cv2")
    lr_changed = sp_changed = 0
    for kind_i, kind in enumerate(("occluded", "noise")):
        l, r = occluded_pair(H, W, D, D + bs) if kind == "occluded" else synth.random_pair(H, W, seed=D + bs)
        for cap, tex, uq in SWEEP_BM:
            base = dict(numDisp=D, blockSize=bs, preFilterCap=cap, textureThreshold=tex, uniquenessRatio=uq)
            plain = ref.bm(oracle, l, r, base)
            for j, d12 in enumerate((-1, 0, 1, 3)):
                lr = None
                for win, rng in ((0, 0), SPECKLE[(j + len(SWEEP_BM) * kind_i) % len(SPECKLE)]):
                    p = dict(base, disp12MaxDiff=d12, speckleWindowSize=win, speckleRange=rng)
                    got = ref.bm(oracle, l, r, p)
                    check("%s %s" % (kind, p), got, cv_bm(cv2, l, r, p))
                    if win == 0:
                        lr = got
                        lr_changed += int((got != plain).sum())
                    else:
                        sp_changed += int((got != lr).sum())
    # the inputs make both filters act (the test cannot pass with filters that do nothing)
    assert lr_changed > 100 and sp_changed > 100, (lr_changed, sp_changed)


def test_reference_stereo_match_configuration(oracle):
    cv2 = pytest.importorskip("cv2")
    for H, W, D, bs, seed in ((120, 300, 64, 9, 1), (121, 320, 48, 15, 2)):
        l, r = occluded_pair(H, W, D, seed)
        p = dict(numDisp=D, blockSize=bs, **STEREO_MATCH, **STEREO_MATCH_FILTERS)
        got = ref.bm(oracle, l, r, p)
        check("stereo_match", got, cv_bm(cv2, l, r, p))
        assert (got != ref.bm(oracle, l, r, dict(p, disp12MaxDiff=-1, speckleWindowSize=0))).sum() > 50


def test_filter_units_and_order(oracle):
    """speckleRange is used as given (x16 units), disp12MaxDiff = 0 is a real check, the check runs before speckle."""
    cv2 = pytest.importorskip("cv2")
    base = dict(numDisp=64, blockSize=15, **STEREO_MATCH)
    l, r = synth.random_pair(120, 300, seed=7)
    plain = cv_bm(cv2, l, r, base)
    want = plain.copy()
    cv2.filterSpeckles(want, FILT, 50, 2)
    check("range as given", ref.bm(oracle, l, r, dict(base, speckleWindowSize=50, speckleRange=2)), want)
    want32 = plain.copy()
    cv2.filterSpeckles(want32, FILT, 50, 32)
    assert not np.array_equal(want, want32)
    l, r = occluded_pair(120, 300, 64, 7)
    plain = cv_bm(cv2, l, r, base)
    d0 = ref.bm(oracle, l, r, dict(base, disp12MaxDiff=0))
    assert (d0 != plain).sum() > 0
    lr1 = ref.bm(oracle, l, r, dict(base, disp12MaxDiff=1))
    cv2.filterSpeckles(lr1, FILT, 50, 32)
    check("check before speckle", ref.bm(oracle, l, r, dict(base, disp12MaxDiff=1, speckleWindowSize=50, speckleRange=32)), lr1)


def test_reference_rejects_bad_speckle_values(oracle):
    l, r = synth.random_pair(40, 100, seed=1)
    for win, rng in ((-1, 0), (10, -1)):
        with pytest.raises(ValueError):
            ref.bm(oracle, l, r, dict(numDisp=16, blockSize=7, speckleWindowSize=win, speckleRange=rng))
    ref.bm(oracle, l, r, dict(numDisp=16, blockSize=7, speckleWindowSize=0, speckleRange=-1))


def test_load_bm_parameters_reads_the_filter_keys(tmp_path):
    class Fake:
        def set_bm_params(self, **kw):
            self.bm = kw

        def set_bm_filters(self, *a):
            self.filters = a
    f = tmp_path / "bm.yml"
    f.write_text("%YAML:1.0\nnumDisp: 80\nblockSize: 21\npreFilterCap: 2\n")
    e = Fake()
    assert api.loadBMParameters(str(f), e, {})
    assert not hasattr(e, "filters")
    f.write_text("%YAML:1.0\nnumDisp: 64\nblockSize: 9\nspeckleWindowSize: 100\nspeckleRange: 32\ndisp12MaxDiff: 1\n")
    assert api.loadBMParameters(str(f), e, {})
    assert e.filters == (1, 100, 32)
    f.write_text("%YAML:1.0\nnumDisp: 64\nblockSize: 9\nspeckleWindowSize: 100\n")
    assert api.loadBMParameters(str(f), e, {})
    assert e.filters == (-1, 100, 0)


# ---- GPU ------------------------------------------------------------------------------------------------------------
CASE_FILTERS = [dict(disp12MaxDiff=1, speckleWindowSize=100, speckleRange=32),
                dict(disp12MaxDiff=0, speckleWindowSize=50, speckleRange=2),
                dict(disp12MaxDiff=3, speckleWindowSize=150, speckleRange=16)]


@pytest.mark.gpu
@pytest.mark.parametrize("wide", [0, 2], ids=["auto", "u16"])
@pytest.mark.parametrize("case", cases.BM_CASES, ids=[c[0] for c in cases.BM_CASES])
def test_bm_filters_stages_vs_reference(oracle, case, wide):
    """Every BM geometry with both filters on, a batch of three different frames: the map after the LR check
    (debug_read 2) and the final map against the reference; both column-sum forms."""
    name, p, H, W = case
    if wide and p["blockSize"] * 2 * p["preFilterCap"] > 255:
        pytest.skip("the volume is 16 bits wide anyway")
    i = [c[0] for c in cases.BM_CASES].index(name)
    f = CASE_FILTERS[i % len(CASE_FILTERS)]
    frames = [occluded_pair(H, W, p["numDisp"], i), cases.bm_inputs(name, p, H, W, "ramp"), cases.bm_inputs(name, p, H, W, "noise")]
    with api.Engine(W, H, max_batch=3) as e:
        e.set_bm_params(**p)
        e.set_bm_filters(**f)
        e.debug_set_flags(wide)
        e.compute(np.stack([a for a, _ in frames]), np.stack([b for _, b in frames]), api.STAGE_BM)
        out = e.download(3)["disp"]
        lr = e.debug_read(2, 3)
    for b, (l, r) in enumerate(frames):
        check("%s/%d/lr" % (name, b), lr[b], ref.bm(oracle, l, r, dict(p, disp12MaxDiff=f["disp12MaxDiff"])))
        check("%s/%d/final" % (name, b), out[b], ref.bm(oracle, l, r, dict(p, **f)))


@pytest.mark.gpu
def test_bm_filters_one_at_a_time(oracle):
    p = dict(numDisp=48, blockSize=15, **STEREO_MATCH)
    H, W = 81, 250
    l, r = occluded_pair(H, W, 48, 11)
    with api.Engine(W, H) as e:
        e.set_bm_params(**p)
        for f in (dict(disp12MaxDiff=0), dict(speckleWindowSize=60, speckleRange=16), dict(disp12MaxDiff=2),
                  dict(disp12MaxDiff=-5, speckleWindowSize=0, speckleRange=-3)):
            e.set_bm_filters(**f)
            e.compute(l, r, api.STAGE_BM)
            want = ref.bm(oracle, l, r, dict(p, **{k: max(v, -1) for k, v in f.items()}))
            check(str(f), e.download(1)["disp"][0], want)


@pytest.mark.gpu
def test_bm_filters_survive_params_and_resize(oracle):
    """Filters set before set_bm_params and kept by it, set after it, and kept across a geometry change."""
    H, W = 100, 300
    p = dict(numDisp=32, blockSize=9, **STEREO_MATCH)
    f = STEREO_MATCH_FILTERS
    l, r = occluded_pair(H, W, 32, 5)
    ys, xs = np.mgrid[0:H, 0:W].astype(np.float32)
    with api.Engine(W, H) as e:
        e.set_bm_filters(**f)
        e.set_bm_params(**p)
        e.compute(l, r, api.STAGE_BM)
        check("before params", e.download(1)["disp"][0], ref.bm(oracle, l, r, dict(p, **f)))
        p2 = dict(p, numDisp=48)
        e.set_bm_params(**p2)
        e.set_bm_filters(disp12MaxDiff=0, speckleWindowSize=40, speckleRange=16)
        f2 = dict(disp12MaxDiff=0, speckleWindowSize=40, speckleRange=16)
        e.compute(l, r, api.STAGE_BM)
        check("after params", e.download(1)["disp"][0], ref.bm(oracle, l, r, dict(p2, **f2)))
        e.set_bm_params(**p)
        for cam in (0, 1):
            e.upload_rectify_maps(cam, xs, ys, (0, 0, W, H))
        e.set_resize(0.5)
        e.compute(l, r, api.STAGE_RECTIFY | api.STAGE_BM)
        res = e.download(1, rect=True)
        rl, rr = res["rectL"][0], res["rectR"][0]
        assert rl.shape == (H // 2, W // 2)
        check("after resize", res["disp"][0], ref.bm(oracle, rl, rr, dict(p, **f2)))


@pytest.mark.gpu
def test_bm_filters_with_xyz_means_and_two_slots(oracle):
    H, W, B = 90, 260, 2
    p = dict(BM_YML)
    f = STEREO_MATCH_FILTERS
    rois = [(100, 10, 40, 30), (150, 40, 60, 40), (90, 60, 5, 5)]
    batches = [[occluded_pair(H, W, 80, 20 + 2 * k + b) for b in range(B)] for k in range(3)]
    with api.Engine(W, H, max_batch=B) as e:
        e.set_bm_params(**p)
        e.set_bm_filters(**f)
        e.set_Q(cases.Q_REFERENCE)
        e.set_mean_rois(rois)
        e.set_io_slots(2)
        stages = api.STAGE_BM | api.STAGE_XYZ | api.STAGE_MEANS
        results = []
        for k, fr in enumerate(batches):
            e.compute(np.stack([a for a, _ in fr]), np.stack([b for _, b in fr]), stages)
            if k > 0:
                results.append(e.download(B, xyz=True, means=True, age=1))
        e.sync()
        results.append(e.download(B, xyz=True, means=True))
    for k, (fr, res) in enumerate(zip(batches, results)):
        for b, (l, r) in enumerate(fr):
            want = ref.bm(oracle, l, r, dict(p, **f))
            check("slots %d/%d" % (k, b), res["disp"][b], want)
            xyz, valid = oracle.reproject(want, cases.Q_REFERENCE)
            v = valid.astype(bool)
            np.testing.assert_allclose(res["xyz"][b][v], xyz[v], rtol=1e-5)
            assert np.all(res["xyz"][b][~v] == 0)
            np.testing.assert_array_equal(res["means"][b], [oracle.mean(want, roi) for roi in rois])


@pytest.mark.gpu
def test_bm_explicit_defaults_change_nothing():
    H, W, B = 90, 260, 3
    frames = [occluded_pair(H, W, 80, 30 + b) for b in range(B)]
    L, R = np.stack([a for a, _ in frames]), np.stack([b for _, b in frames])
    outs = []
    for explicit in (False, True):
        with api.Engine(W, H, max_batch=B) as e:
            e.set_bm_params(**BM_YML)
            if explicit:
                e.set_bm_filters(1, 100, 32)
                e.set_bm_filters(-1, 0, 0)
            e.compute(L, R, api.STAGE_BM)
            outs.append(e.download(B)["disp"])
    assert np.array_equal(outs[0], outs[1])


@pytest.mark.gpu
def test_bm_filters_rejections():
    with api.Engine(200, 60) as e:
        for bad in (dict(speckleWindowSize=-1), dict(speckleWindowSize=10, speckleRange=-1)):
            with pytest.raises(api.MvsvError) as ei:
                e.set_bm_filters(**bad)
            assert ei.value.code == -1
    W = 4112
    l, r = synth.random_pair(40, W, seed=3)
    with api.Engine(W, 40) as e:
        e.set_bm_params(numDisp=16, blockSize=9, **STEREO_MATCH)
        with pytest.raises(api.MvsvError) as ei:
            e.set_bm_filters(disp12MaxDiff=0)
        assert ei.value.code == -5
        e.set_bm_filters(disp12MaxDiff=-1, speckleWindowSize=20, speckleRange=16)     # the speckle filter has no limit
        e.compute(l, r, api.STAGE_BM)
    # a narrow engine with the check on that is widened by a geometry change: the compute refuses
    ys, xs = np.mgrid[0:40, 0:2100].astype(np.float32)
    with api.Engine(2100, 40) as e:
        e.set_bm_params(numDisp=16, blockSize=9, **STEREO_MATCH)
        e.set_bm_filters(disp12MaxDiff=1)
        for cam in (0, 1):
            e.upload_rectify_maps(cam, xs, ys, (0, 0, 2100, 40))
        e.set_resize(2.0)
        lw, rw = synth.random_pair(40, 2100, seed=4)
        with pytest.raises(api.MvsvError) as ei:
            e.compute(lw, rw, api.STAGE_RECTIFY | api.STAGE_BM)
        assert ei.value.code == -5


@pytest.mark.gpu
def test_cfg1_stereo_match_filters_vs_cv2():
    """configs/bm.yml at 752x480 with the stereo_match filters, a batch of 148 frames: several frames against cv2."""
    cv2 = pytest.importorskip("cv2")
    H, W, B = 480, 752, 148
    p = dict(BM_YML, **STEREO_MATCH_FILTERS)
    gen = [occluded_pair(H, W, 80, 60 + s) for s in range(4)]
    L = np.stack([gen[b % 4][0] for b in range(B)])
    R = np.stack([gen[b % 4][1] for b in range(B)])
    with api.Engine(W, H, max_batch=B) as e:
        e.set_bm_params(**BM_YML)
        e.set_bm_filters(**STEREO_MATCH_FILTERS)
        e.compute(L, R, api.STAGE_BM)
        out = e.download(B)["disp"]
    for b in (0, 1, 2, 3, 73, 146, 147):
        check("cfg1 filters/%d" % b, out[b], cv_bm(cv2, gen[b % 4][0], gen[b % 4][1], p))
    plain = cv_bm(cv2, gen[0][0], gen[0][1], BM_YML)
    assert (out[0] != plain).sum() > 1000
