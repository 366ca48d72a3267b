"""SGBM with numDisp in (256, 512]: the oracle against cv2 4.13 at the new range (CPU), and the CUDA path stage by stage
against the oracle, through every aggregation route, against cv2 at full size, at the contract's boundaries and through a
multi-device ctx with several rigs (GPU).

Above 256 the volumes take the pixel stride of the sweep's eight-lane layout (Dp = 320 / 384 / 448 / 512), the row scans
keep a pixel in one warp with 16 disparities per lane, and the cost kernel runs once per block of 256 disparities."""
import numpy as np
import pytest

import cases
from mvstereovision3_b200 import api, synth

ERR_INVALID, ERR_UNSUPPORTED = -1, -5


def gpu_params(p):
    d = dict(p)
    d["disparityMode"] = d.pop("mode")
    return d


def check(name, got, want):
    assert got.shape == want.shape, (name, got.shape, want.shape)
    if not np.array_equal(got, want):
        idx = np.argwhere(got != want)
        raise AssertionError("%s: %d mismatches, first at %s: got %s want %s" % (
            name, len(idx), tuple(idx[0]), got[tuple(idx[0])], want[tuple(idx[0])]))


def cv_sgbm(cv2, l, r, p):
    m = cv2.StereoSGBM_create(minDisparity=p["minDisp"], numDisparities=p["numDisp"], blockSize=p["blockSize"],
                              P1=p["P1"], P2=p["P2"], disp12MaxDiff=p["disp12MaxDiff"], preFilterCap=p["preFilterCap"],
                              uniquenessRatio=p["uniquenessRatio"], speckleWindowSize=p["speckleWindowSize"],
                              speckleRange=p["speckleRange"],
                              mode=cv2.STEREO_SGBM_MODE_HH if p["mode"] == 1 else cv2.STEREO_SGBM_MODE_SGBM)
    return m.compute(l, r)


# ---- CPU: the oracle against cv2 at the new range -------------------------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1], ids=["sgbm", "hh"])
@pytest.mark.parametrize("minD", [-5, 0, 3])
@pytest.mark.parametrize("D", [264, 320, 392, 512])
def test_oracle_equals_cv2_wide(oracle, D, minD, mode):
    cv2 = pytest.importorskip("cv2")
    p = oracle.make_sgbm_params(minDisp=minD, numDisp=D, blockSize=5, P1=40, P2=160, uniquenessRatio=10, disp12MaxDiff=2,
                                speckleWindowSize=60, speckleRange=2, mode=mode)
    H, W = 48, D + 120
    pairs = [synth.stereogram(H, W, minD, D, seed=D + minD)[:2], synth.random_pair(H, W, seed=D - minD)]
    for l, r in pairs:
        check("oracle vs cv2", oracle.sgbm(l, r, p), cv_sgbm(cv2, l, r, p))


# ---- GPU: stage by stage against the oracle -------------------------------------------------------------------------
STAGE_CASES = [
    ("d264_neg", dict(minDisp=-5, numDisp=264, blockSize=5, P1=40, P2=160, uniquenessRatio=10, disp12MaxDiff=2)),
    ("d392_hh", dict(minDisp=3, numDisp=392, blockSize=3, P1=20, P2=90, uniquenessRatio=5, disp12MaxDiff=1, mode=1)),
    ("d384_hh_neg", dict(minDisp=-2, numDisp=384, blockSize=7, P1=30, P2=200, uniquenessRatio=15, disp12MaxDiff=3, mode=1)),
    ("d512", dict(minDisp=0, numDisp=512, blockSize=5, P1=200, P2=800, uniquenessRatio=10, disp12MaxDiff=1,
                  speckleWindowSize=50, speckleRange=2)),
    ("d448_uniq100", dict(minDisp=1, numDisp=448, blockSize=3, P1=8, P2=32, uniquenessRatio=100)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("sweep", [0, 0xfe], ids=["auto", "sweep"])
@pytest.mark.parametrize("name,kw", STAGE_CASES, ids=[c[0] for c in STAGE_CASES])
def test_stages_vs_oracle(oracle, name, kw, sweep):
    """C, the final S, the raw and the final disparities of a ramp and a noise pair (MODE_SGBM and MODE_HH, padded
    lanes at D = 264 / 392, negative minDisp); "auto" lets the engine choose the independent passes for a batch of two,
    "sweep" forces the fused sweep."""
    p = cases.sgbm_params(**kw)
    H, W = 40, p["numDisp"] + 130
    pairs = [synth.stereogram(H, W, max(p["minDisp"], 0), p["numDisp"], seed=7)[:2], synth.random_pair(H, W, seed=8)]
    with api.Engine(W, H, max_batch=2) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.debug_set_flags(1 | (sweep << 8))
        e.compute(np.stack([a for a, _ in pairs]), np.stack([b for _, b in pairs]), api.STAGE_SGBM)
        out = e.download(2)["disp"]
        Cg, Sg, raw = (e.debug_read(w, 2) for w in (0, 1, 2))
    for b, (l, r) in enumerate(pairs):
        disp, Cv, Sv, rawv = oracle.sgbm(l, r, p, want_volumes=True, want_raw=True)
        check("%s/C/%d" % (name, b), Cg[b], Cv)
        check("%s/S/%d" % (name, b), Sg[b], Sv)
        check("%s/raw/%d" % (name, b), raw[b], rawv)
        check("%s/disp/%d" % (name, b), out[b], disp)


@pytest.mark.gpu
@pytest.mark.parametrize("kw,s8", [
    (dict(numDisp=384, blockSize=5, mode=1), 1),                                 # P1 = P2 = 0 -> 2 / 5: 8 * 5 <= 255
    (dict(numDisp=512, blockSize=3, uniquenessRatio=10), 1),
    (dict(numDisp=264, blockSize=5, P1=200, P2=800, mode=1), 0),                 # NR = 20: no byte form
    (dict(numDisp=392, blockSize=3, P1=10, P2=30, minDisp=-3), 0),               # NR = 28: no byte form
], ids=["d384_hh", "d512", "d264_p800", "d392"])
def test_byte_form_and_16bit_form_of_S(oracle, kw, s8):
    """The byte form of S where the sweep's layout and npaths * P2 <= 255 allow it, the 16-bit form when debug flag
    bit 1 forces it: the same final S and disparities as the oracle."""
    p = cases.sgbm_params(**kw)
    H, W = 33, p["numDisp"] + 93
    l, r = synth.random_pair(H, W, seed=11)
    l2, r2, _ = synth.stereogram(H, W, max(p["minDisp"], 0), p["numDisp"], seed=12)
    want = [oracle.sgbm(a, b, p, want_volumes=True) for a, b in ((l, r), (l2, r2))]
    for flags in (1, 3):
        with api.Engine(W, H, max_batch=2) as e:
            e.set_sgbm_params(**gpu_params(p))
            e.debug_set_flags(flags | (0xfe << 8))
            e.compute(np.stack([l, l2]), np.stack([r, r2]), api.STAGE_SGBM)
            out, Sg = e.download(2)["disp"], e.debug_read(1, 2)
            assert e.info.sgbm_s8 == (s8 if flags == 1 else 0)
        for b in range(2):
            check("S/%d/%d" % (flags, b), Sg[b], want[b][2])
            check("disp/%d/%d" % (flags, b), out[b], want[b][0])


# ---- GPU: every aggregation route -----------------------------------------------------------------------------------
ROUTE_CASES = [
    ("d384_hh_s8", dict(minDisp=0, numDisp=384, blockSize=3, P1=10, P2=30, uniquenessRatio=5, disp12MaxDiff=1, mode=1)),
    ("d264_pad", dict(minDisp=2, numDisp=264, blockSize=5, P1=40, P2=300, uniquenessRatio=10, disp12MaxDiff=2)),
    ("d504_pad_hh", dict(minDisp=0, numDisp=504, blockSize=3, P1=20, P2=90, mode=1)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("nc", [1, 4, 16, 0xfe, 0xff])
@pytest.mark.parametrize("name,kw", ROUTE_CASES, ids=[c[0] for c in ROUTE_CASES])
def test_aggregation_routes(oracle, name, kw, nc):
    """Forced strip counts of the fused sweep (1; 4: the cluster transport; 16: global memory), the engine's own strip
    count (0xfe) and the independent passes (0xff) give the oracle's bits."""
    p = cases.sgbm_params(**kw)
    H = 23
    W = p["minDisp"] + p["numDisp"] + (40 if nc == 1 else 150)       # a strip holds at most 40-44 pixels
    l, r = synth.random_pair(H, W, seed=21)
    l2, r2, _ = synth.stereogram(H, W, p["minDisp"], p["numDisp"], seed=22)
    with api.Engine(W, H, max_batch=2) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.debug_set_flags(1 | (nc << 8))
        if nc != 0xfe:
            assert e.info.sgbm_td_cluster == (0 if nc == 0xff else nc)
        e.compute(np.stack([l, l2]), np.stack([r, r2]), api.STAGE_SGBM)
        out, Sg = e.download(2)["disp"], e.debug_read(1, 2)
    for b, (a_, b_) in enumerate(((l, r), (l2, r2))):
        disp, _, Sv, _ = oracle.sgbm(a_, b_, p, want_volumes=True)
        check("%s/S/%d" % (name, b), Sg[b], Sv)
        check("%s/disp/%d" % (name, b), out[b], disp)


@pytest.mark.gpu
@pytest.mark.parametrize("D,nc,B", [(384, 37, 9), (264, 30, 11)])
def test_sweep_walks_several_frames_per_cta(oracle, D, nc, B):
    """More frames than frame slots: every CTA of the persistent sweep walks several frames (MODE_HH: two sweeps)."""
    p = cases.sgbm_params(minDisp=0, numDisp=D, blockSize=3, P1=20, P2=90, uniquenessRatio=5, disp12MaxDiff=1, mode=1)
    H, W = 9, D + 150
    ls, rs = zip(*[synth.random_pair(H, W, seed=300 + s) for s in range(6)])
    L, R = np.stack([ls[b % 6] for b in range(B)]), np.stack([rs[b % 6] for b in range(B)])
    want = [oracle.sgbm(ls[b], rs[b], p) for b in range(6)]
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.debug_set_flags(nc << 8)
        assert e.info.sgbm_td_cluster == nc and B > 148 // nc
        for it in range(5):
            e.compute(L, R, api.STAGE_SGBM)
            got = e.download(B)["disp"]
            for b in range(B):
                check("iteration %d frame %d" % (it, b), got[b], want[b % 6])


@pytest.mark.gpu
@pytest.mark.parametrize("fpc", [1, 2])
def test_chunked_cost_and_first_scan(oracle, fpc):
    """The cost kernel (one launch per block of 256 disparities) and the first row scan of different chunks of frames
    side by side on two streams: every stage of five different frames, byte form of S and 16-bit form."""
    p = cases.sgbm_params(minDisp=1, numDisp=384, blockSize=5, uniquenessRatio=10, disp12MaxDiff=1, mode=1)
    H, W, B = 30, 384 + 110, 5
    frames = [synth.random_pair(H, W, seed=50 + b) if b % 2 else synth.stereogram(H, W, 1, 384, seed=50 + b)[:2]
              for b in range(B)]
    L, R = np.stack([f[0] for f in frames]), np.stack([f[1] for f in frames])
    want = [oracle.sgbm(f[0], f[1], p, want_volumes=True) for f in frames]
    for flags in (1, 3):
        with api.Engine(W, H, max_batch=B) as e:
            e.set_sgbm_params(**gpu_params(p))
            e.debug_set_flags(flags | (0xfe << 8) | (fpc << 16))
            e.compute(L, R, api.STAGE_SGBM)
            out, Cg, Sg = e.download(B)["disp"], e.debug_read(0, B), e.debug_read(1, B)
        for b in range(B):
            check("C/%d/%d" % (flags, b), Cg[b], want[b][1])
            check("S/%d/%d" % (flags, b), Sg[b], want[b][2])
            check("disp/%d/%d" % (flags, b), out[b], want[b][0])


# ---- GPU: against cv2 at full size ----------------------------------------------------------------------------------
CFG4_D512 = cases.sgbm_params(numDisp=512, blockSize=5, P1=200, P2=800, disp12MaxDiff=1, uniquenessRatio=10,
                              speckleWindowSize=150, speckleRange=2, mode=1)
SGBM_YML_D384 = cases.sgbm_params(minDisp=1, numDisp=384, blockSize=13, speckleWindowSize=150, speckleRange=2)


@pytest.mark.gpu
@pytest.mark.parametrize("p,H,W,B,ramp", [(CFG4_D512, 1080, 1920, 2, True), (SGBM_YML_D384, 720, 1280, 1, False)],
                         ids=["1080p_d512_hh", "720p_d384_sgbm_yml"])
def test_full_size_vs_cv2(p, H, W, B, ramp):
    cv2 = pytest.importorskip("cv2")
    gen = [synth.stereogram(H, W, p["minDisp"], p["numDisp"], seed=b) for b in range(B)]
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.compute(np.stack([g[0] for g in gen]), np.stack([g[1] for g in gen]), api.STAGE_SGBM)
        out = e.download(B)["disp"]
    for b in range(B):
        check("full/%d" % b, out[b], cv_sgbm(cv2, gen[b][0], gen[b][1], p))
    if not ramp:
        return      # (blockSize 13 and speckle range 2 keep only ~10 % of this ramp's pixels, as in cv2)
    # the ramp is recovered: median |error| of valid pixels below one disparity step
    valid = out[0] > (p["minDisp"] - 1) * 16
    err = np.abs(out[0].astype(np.float32) / 16 - gen[0][2][:, None].astype(np.float32))[valid]
    assert valid.mean() > 0.5 and np.median(err) < 1.0


@pytest.mark.gpu
def test_full_batch_twins_agree():
    """A full-size batch at 720p, D = 384 (every sweep CTA walks several frames): every copy equals its twin on every
    repetition, and one copy of each pair equals cv2."""
    cv2 = pytest.importorskip("cv2")
    p, H, W, B = SGBM_YML_D384, 720, 1280, 12
    gen = [synth.stereogram(H, W, p["minDisp"], p["numDisp"], seed=50 + s)[:2] for s in range(3)]
    L, R = np.stack([gen[b % 3][0] for b in range(B)]), np.stack([gen[b % 3][1] for b in range(B)])
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**gpu_params(p))
        for it in range(3):
            e.compute(L, R, api.STAGE_SGBM)
            d = e.download(B)["disp"]
            for b in range(3, B):
                check("repetition %d frame %d vs its twin" % (it, b), d[b], d[b % 3])
    for s in range(3):
        check("vs cv2 / %d" % s, d[s], cv_sgbm(cv2, gen[s][0], gen[s][1], p))


# ---- GPU: the boundaries of the contract ----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("sweep", [0, 0xfe], ids=["auto", "sweep"])
def test_single_column_domain(oracle, sweep):
    """W = maxD + 1: one column of the cost domain (W1 = 1)."""
    p = cases.sgbm_params(minDisp=0, numDisp=264, blockSize=3, P1=10, P2=60, uniquenessRatio=5, disp12MaxDiff=1, mode=1)
    H, W = 21, 265
    l, r = synth.random_pair(H, W, seed=31)
    with api.Engine(W, H) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.debug_set_flags(sweep << 8)
        assert e.info.sgbm_W1 == 1
        e.compute(l, r, api.STAGE_SGBM)
        check("W1 = 1", e.download(1)["disp"][0], oracle.sgbm(l, r, p))


@pytest.mark.gpu
def test_contract_rejections():
    with api.Engine(700, 40) as e:
        for bad, code in ((dict(numDisp=520), ERR_INVALID), (dict(numDisp=512, minDisp=200), ERR_INVALID),
                          (dict(numDisp=264, minDisp=-700), ERR_INVALID)):
            with pytest.raises(api.MvsvError) as ex:
                e.set_sgbm_params(**gpu_params(cases.sgbm_params(**bad)))
            assert ex.value.code == code, bad
        e.set_sgbm_params(**gpu_params(cases.sgbm_params(numDisp=512, minDisp=187)))      # W1 = 1 is accepted
        assert e.info.sgbm_W1 == 1
        with pytest.raises(api.MvsvError) as ex:
            e.set_bm_params(numDisp=272, blockSize=9, preFilterCap=31, textureThreshold=10, uniquenessRatio=15)
        assert ex.value.code == ERR_INVALID                                                 # StereoBM stays at <= 256
    with api.Engine(3840, 2160) as e:
        with pytest.raises(api.MvsvError) as ex:
            e.set_sgbm_params(**gpu_params(cases.sgbm_params(numDisp=512, blockSize=5, P1=200, P2=800)))
        assert ex.value.code == ERR_UNSUPPORTED                                             # > 2^31 cells per frame


@pytest.mark.gpu
def test_rejected_resize_keeps_the_results(oracle):
    """A 700-wide ROI at numDisp 512 leaves a cost domain of 188 columns; resizing it by 0.5 would empty it and is
    rejected: the engine keeps its size and the results of its last compute."""
    fw, fh = 720, 40
    roi = (10, 0, 700, fh)
    p = cases.sgbm_params(numDisp=512, blockSize=5, P1=40, P2=160, uniquenessRatio=10)
    l, r, _ = synth.stereogram(fh, 700, 0, 512, seed=41)
    with api.Engine(fw, fh) as e:
        for cam in range(2):
            mx, my = cases.warp_maps(fh, fw, seed=cam)
            e.upload_rectify_maps(cam, mx, my, roi)
        e.set_sgbm_params(**gpu_params(p))
        e.compute(l, r, api.STAGE_SGBM)
        before = e.download(1)["disp"]
        with pytest.raises(api.MvsvError) as ex:
            e.set_resize(0.5)
        assert ex.value.code == ERR_INVALID
        assert (e.info.width, e.info.height) == (700, fh)
        check("earlier results", e.download(1)["disp"], before)
        check("vs oracle", before[0], oracle.sgbm(l, r, p))
        e.compute(l, r, api.STAGE_SGBM)
        check("computed again", e.download(1)["disp"], before)


@pytest.mark.gpu
@pytest.mark.parametrize("D,Dpad,s8", [(264, 320, 0), (320, 320, 0), (384, 384, 1), (392, 448, 0), (448, 448, 0),
                                       (456, 512, 1), (512, 512, 1)])
def test_info_reports_the_layout(D, Dpad, s8):
    """sgbm_D, the pixel stride sgbm_Dpad, and whether S was kept as bytes (P2 = 5, MODE_HH: 8 * 5 <= 255, and NR a
    multiple of 8, i.e. D in (320, 384] or (448, 512])."""
    H, W = 12, D + 60
    l, r = synth.random_pair(H, W, seed=D)
    with api.Engine(W, H, max_batch=2) as e:
        e.set_sgbm_params(**gpu_params(cases.sgbm_params(numDisp=D, blockSize=3, mode=1)))
        e.debug_set_flags(0xfe << 8)
        e.compute(l, r, api.STAGE_SGBM)
        i = e.info
        assert (i.sgbm_D, i.sgbm_Dpad, i.sgbm_s8) == (D, Dpad, s8)


# ---- GPU: composition ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_devices_and_rigs_equal_one_engine(oracle):
    """One D = 384 batch from two rigs through a ctx over [0, 0] equals the single engine, bit for bit, and the oracle
    on the frames remapped with each frame's rig.  The rigs' maps shift both cameras alike (sub-pixel in x, half a row
    in y), so the stereo correspondence survives rectification."""
    FW, FH, ROI = 560, 40, (6, 3, 520, 32)
    kw = cases.sgbm_params(minDisp=1, numDisp=384, blockSize=5, uniquenessRatio=10, disp12MaxDiff=1, mode=1)
    p = gpu_params(kw)
    ys, xs = np.mgrid[0:FH, 0:FW].astype(np.float32)
    maps = {rig: (xs + 0.25 * (rig + 1), ys + 0.5 * rig) for rig in (0, 1)}
    rois = {rig: (ROI[0] + 4 * rig, ROI[1], ROI[2], ROI[3]) for rig in (0, 1)}
    B = 5
    pairs = [synth.stereogram(FH, FW, 1, 384, seed=60 + b)[:2] for b in range(B)]
    L, R = np.stack([a for a, _ in pairs]), np.stack([b for _, b in pairs])
    rigs = [0, 1, 1, 0, 1]

    def run(e):
        for rig in (0, 1):
            for cam in range(2):
                e.upload_rectify_maps(cam, maps[rig][0], maps[rig][1], rois[rig], rig=rig)
        e.set_sgbm_params(**p)
        e.set_frame_rigs(rigs)
        e.compute(L, R, api.STAGE_RECTIFY | api.STAGE_SGBM)
        return e.download(B, rect=True)

    with api.Engine(FW, FH, max_batch=B, devices=[0, 0]) as e, api.Engine(FW, FH, max_batch=B) as one:
        got, want = run(e), run(one)
    assert got.keys() == want.keys()
    for k in want:
        check(k, got[k], want[k])
    for b, rig in enumerate(rigs):
        l, r = (oracle.remap(img[b], maps[rig][0], maps[rig][1], rois[rig]) for img in (L, R))
        check("oracle/%d" % b, want["disp"][b], oracle.sgbm(l, r, kw))
    assert (want["disp"] > 0).mean() > 0.05          # the cost domain is 135 of 520 columns
