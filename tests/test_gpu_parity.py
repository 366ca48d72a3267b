"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle, the committed cv2 golden
vectors and (when cv2 is importable) cv2 4.13.0 live at the BASELINE.json sizes.  Integer outputs are bit-exact;
float XYZ within 1e-5 relative (north_star)."""
import os

import numpy as np
import pytest

import cases
from mvstereovision3_b200 import api, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(cases.GOLDEN_DIR, "cv2_golden.npz"))


def gpu_params(p):
    d = dict(p)
    d["disparityMode"] = d.pop("mode")
    return d


def first_diff(a, b):
    idx = np.argwhere(a != b)
    return "%d mismatches, first at %s: got %s want %s" % (len(idx), tuple(idx[0]), a[tuple(idx[0])], b[tuple(idx[0])])


def check(name, got, want):
    assert got.shape == want.shape, (name, got.shape, want.shape)
    assert np.array_equal(got, want), "%s: %s" % (name, first_diff(got, want))


@pytest.mark.parametrize("sweep", [0, 0xfe], ids=["auto", "sweep"])
@pytest.mark.parametrize("case", cases.SGBM_CASES, ids=[c[0] for c in cases.SGBM_CASES])
def test_sgbm_stages_vs_oracle(oracle, golden, case, sweep):
    """Every stage against the oracle and the cv2 golden vectors.  "auto": the engine's own choice for a batch of two
    (the independent one-direction passes); "sweep": the fused strip sweep the throughput configurations use."""
    name, p, H, W = case
    with api.Engine(W, H, max_batch=2) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.debug_set_flags(1 | (sweep << 8))
        pair = [cases.sgbm_inputs(name, p, H, W, k) for k in ("ramp", "noise")]
        left = np.stack([pair[0][0], pair[1][0]])
        right = np.stack([pair[0][1], pair[1][1]])
        e.compute(left, right, api.STAGE_SGBM)
        out = e.download(2)["disp"]
        Cg, Sg, raw, med = (e.debug_read(w, 2) for w in (0, 1, 2, 4))
        for b, kind in enumerate(("ramp", "noise")):
            disp, Cv, Sv, rawv = oracle.sgbm(pair[b][0], pair[b][1], p, want_volumes=True, want_raw=True)
            check(name + "/C/" + kind, Cg[b], Cv)
            check(name + "/S/" + kind, Sg[b], Sv)
            check(name + "/raw/" + kind, raw[b], rawv)
            check(name + "/median/" + kind, med[b], oracle.median3(rawv))
            check(name + "/disp/" + kind, out[b], disp)
            check(name + "/golden/" + kind, out[b], golden["sgbm/%s/%s" % (name, kind)])


@pytest.mark.parametrize("nc", [1, 2, 4, 8, 0xff])
@pytest.mark.parametrize("ci", [0, 1, 3, 7])
def test_fused_sweep_cluster_sizes(oracle, ci, nc):
    """The fused previous-row sweep (csrc/sweep.cu) with 1, 2, 4 and 8 column strips per frame, and the
    independent-pass fallback (0xff), give the same bits as the oracle (MODE_SGBM and MODE_HH, D = 64, 32, 48, 128)."""
    name, p, H, W = cases.SGBM_CASES[ci]
    l, r = cases.sgbm_inputs(name, p, H, W, "noise")
    with api.Engine(W, H, max_batch=2) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.debug_set_flags(1 | (nc << 8))
        assert e.info.sgbm_td_cluster == (0 if nc == 0xff else nc)
        e.compute(np.stack([l, l[::-1].copy()]), np.stack([r, r[::-1].copy()]), api.STAGE_SGBM)
        out = e.download(2)["disp"]
        Sg = e.debug_read(1, 2)
    disp, Cv, Sv, rawv = oracle.sgbm(l, r, p, want_volumes=True, want_raw=True)
    check("S", Sg[0], Sv)
    check("disp", out[0], disp)
    check("disp flipped", out[1], oracle.sgbm(l[::-1].copy(), r[::-1].copy(), p))


@pytest.mark.parametrize("wide", [0, 2], ids=["auto", "u16"])
@pytest.mark.parametrize("case", cases.BM_CASES, ids=[c[0] for c in cases.BM_CASES])
def test_bm_vs_oracle(oracle, golden, case, wide):
    """Prefilter and disparity against the oracle and the cv2 golden vectors.  "auto": the column-sum volume is one byte
    per cell where blockSize * 2 * cap <= 255 (bm.yml); "u16": debug flag bit 1 keeps it 16 bits wide."""
    name, p, H, W = case
    if wide and p["blockSize"] * 2 * p["preFilterCap"] > 255:
        pytest.skip("the volume is 16 bits wide anyway")
    with api.Engine(W, H, max_batch=2) as e:
        e.set_bm_params(**p)
        e.debug_set_flags(wide)
        pair = [cases.bm_inputs(name, p, H, W, k) for k in ("ramp", "noise")]
        e.compute(np.stack([pair[0][0], pair[1][0]]), np.stack([pair[0][1], pair[1][1]]), api.STAGE_BM)
        out = e.download(2)["disp"]
        preL, preR = e.debug_read(5, 2), e.debug_read(6, 2)
        for b, kind in enumerate(("ramp", "noise")):
            disp, pl, pr = oracle.bm(pair[b][0], pair[b][1], p, want_prefilter=True)
            check(name + "/preL/" + kind, preL[b], pl)
            check(name + "/preR/" + kind, preR[b], pr)
            check(name + "/disp/" + kind, out[b], disp)
            check(name + "/golden/" + kind, out[b], golden["bm/%s/%s" % (name, kind)])


@pytest.mark.parametrize("fpc", [1, 2, 3])
@pytest.mark.parametrize("name", ["sgbm_yml_d64", "hh_cfg4_style", "d48_hh", "d128_shipped"])
def test_chunked_cost_and_first_scan(oracle, name, fpc):
    """The cost kernel and the first row scan of different chunks of frames run side by side on two streams at large
    batches; the debug flag forces `fpc` frames per chunk here: five different frames, every stage of every frame
    against the oracle, byte form of S and 16-bit form."""
    _, p, H, W = next(c for c in cases.SGBM_CASES if c[0] == name)
    B = 5
    frames = [synth.random_pair(H, W, seed=50 + b) if b % 2 else synth.stereogram(H, W, max(p["minDisp"], 0), p["numDisp"], seed=50 + b)[:2]
              for b in range(B)]
    L, R = np.stack([f[0] for f in frames]), np.stack([f[1] for f in frames])
    for flags in (1, 3):
        with api.Engine(W, H, max_batch=B) as e:
            e.set_sgbm_params(**gpu_params(p))
            e.debug_set_flags(flags | (0xfe << 8) | (fpc << 16))
            e.compute(L, R, api.STAGE_SGBM)
            out, Cg, Sg = e.download(B)["disp"], e.debug_read(0, B), e.debug_read(1, B)
        for b in range(B):
            disp, Cv, Sv, _ = oracle.sgbm(frames[b][0], frames[b][1], p, want_volumes=True)
            check("%s/C/%d/%d" % (name, flags, b), Cg[b], Cv)
            check("%s/S/%d/%d" % (name, flags, b), Sg[b], Sv)
            check("%s/disp/%d/%d" % (name, flags, b), out[b], disp)


@pytest.mark.parametrize("W", [16, 17, 18, 19, 20, 21, 22, 23, 119, 120, 121, 122, 123, 124, 125, 239, 240, 241, 244])
def test_widths_around_the_lane_tiling(oracle, W):
    """The prefilter and the median handle four columns per lane and 120 columns per warp (vector path when the width
    allows it, scalar tails otherwise): every width class around those tilings, two heights, every stage."""
    p = cases.sgbm_params(numDisp=8, blockSize=3, P1=7, P2=40, uniquenessRatio=5, speckleWindowSize=20, speckleRange=2)
    for H in (5, 33):
        pair = [synth.random_pair(H, W, seed=W + b) for b in range(2)]
        with api.Engine(W, H, max_batch=2) as e:
            e.set_sgbm_params(**gpu_params(p))
            e.debug_set_flags(1)
            e.compute(np.stack([pair[0][0], pair[1][0]]), np.stack([pair[0][1], pair[1][1]]), api.STAGE_SGBM)
            out = e.download(2)["disp"]
            Cg, raw, med = (e.debug_read(w, 2) for w in (0, 2, 4))
        for b in range(2):
            disp, Cv, Sv, rawv = oracle.sgbm(pair[b][0], pair[b][1], p, want_volumes=True, want_raw=True)
            check("C/%d/%d" % (H, b), Cg[b], Cv)
            check("raw/%d/%d" % (H, b), raw[b], rawv)
            check("median/%d/%d" % (H, b), med[b], oracle.median3(rawv))
            check("disp/%d/%d" % (H, b), out[b], disp)


def test_remap_vs_oracle_and_golden(oracle, golden):
    H, W = 96, 140
    for seed in range(3):
        img, img2 = synth.random_pair(H, W, seed=seed)
        mx, my = cases.warp_maps(H, W, seed)
        with api.Engine(W, H, max_batch=1) as e:
            e.upload_rectify_maps(0, mx, my, (0, 0, W, H))
            e.upload_rectify_maps(1, mx, my, (0, 0, W, H))
            e.compute(img, img2, api.STAGE_RECTIFY)
            r = e.download(1, disp=False, rect=True)
            check("remap/golden/%d" % seed, r["rectL"][0], golden["remap/%d" % seed])
            check("remap/oracle/%d" % seed, r["rectR"][0], oracle.remap(img2, mx, my))
        roi = (5, 3, W - 11, H - 9)
        with api.Engine(W, H, max_batch=1) as e:
            e.upload_rectify_maps(0, mx, my, roi)
            e.upload_rectify_maps(1, mx, my, roi)
            assert (e.info.width, e.info.height) == (W - 11, H - 9)
            e.compute(img, img2, api.STAGE_RECTIFY)
            r = e.download(1, disp=False, rect=True)
            check("remap/crop/%d" % seed, r["rectL"][0], oracle.remap(img, mx, my, roi))


def test_strided_roi_views_and_batches(oracle):
    """cv::Mat ROI views (stride > width, reference src/Stereosystem.cpp:255-256) and batch == per-frame."""
    name, p, H, W = cases.SGBM_CASES[0]
    big_l = np.zeros((3, H + 4, W + 24), np.uint8)
    big_r = np.zeros_like(big_l)
    frames = []
    for b in range(3):
        l, r, _ = synth.stereogram(H, W, p["minDisp"], p["numDisp"], seed=40 + b)
        big_l[b, 2:2 + H, 8:8 + W] = l
        big_r[b, 2:2 + H, 8:8 + W] = r
        frames.append((l, r))
    with api.Engine(W, H, max_batch=3) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.compute(big_l[:, 2:2 + H, 8:8 + W], big_r[:, 2:2 + H, 8:8 + W], api.STAGE_SGBM)
        out = e.download(3)["disp"]
        for b in range(3):
            check("batch/%d" % b, out[b], oracle.sgbm(frames[b][0], frames[b][1], p))
        # single-frame call through the disparity.h mirror
        d = api.sgbm(api.Stereopair(frames[1][0], frames[1][1]), e)
        check("mirror", d, out[1])


def test_speckle_median_xyz_means(oracle, golden):
    """Post-filters on a crafted map are reached through SGBM above; here: consumers on a real SGBM output."""
    name, p, H, W = cases.SGBM_CASES[0]
    l, r = cases.sgbm_inputs(name, p, H, W, "ramp")
    with api.Engine(W, H, max_batch=1) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.set_Q(cases.Q_REFERENCE)
        off = api.dmap_roi_offset(p["numDisp"], W)
        rois = api.subimage_rois(W - off, H, off) + api.samplepoint_rois(W - off, H, off)
        e.set_mean_rois(rois)
        e.compute(l, r, api.STAGE_SGBM | api.STAGE_XYZ | api.STAGE_MEANS)
        out = e.download(1, xyz=True, means=True)
    disp = oracle.sgbm(l, r, p)
    check("disp", out["disp"][0], disp)
    xyz, valid = oracle.reproject(disp, cases.Q_REFERENCE)
    v = valid.astype(bool)
    assert v.any()
    np.testing.assert_allclose(out["xyz"][0][v], xyz[v], rtol=1e-5)
    assert not out["xyz"][0][~v].any()
    want = np.array([oracle.mean(disp, roi) for roi in rois], np.float32)
    np.testing.assert_array_equal(out["means"][0], want)      # integer sums + truncating division: exact


def test_parameter_contract_rejections():
    with api.Engine(320, 200) as e:
        for bad in (dict(numDisp=0), dict(numDisp=20), dict(numDisp=512), dict(numDisp=64, blockSize=21, P2=32 * 441),
                    dict(numDisp=64, blockSize=5, P2=32000), dict(numDisp=64, preFilterCap=200)):
            kw = gpu_params(cases.sgbm_params(**bad))
            with pytest.raises(api.MvsvError) as ex:
                e.set_sgbm_params(**kw)
            assert ex.value.code == -1
        with pytest.raises(api.MvsvError):
            e.set_bm_params(numDisp=24, blockSize=9, preFilterCap=31, textureThreshold=10, uniquenessRatio=15)
        l, r = synth.random_pair(200, 320, seed=1)
        with pytest.raises(api.MvsvError) as ex:
            e.compute(l, r, api.STAGE_SGBM)                 # params not set
        assert ex.value.code == -4


def test_degenerate_width(oracle):
    # W1 <= 0: whole map INVALID (SURVEY.md A.2)
    p = cases.sgbm_params(numDisp=64, blockSize=3)
    l, r = synth.random_pair(20, 50, seed=3)
    with api.Engine(50, 20) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.compute(l, r, api.STAGE_SGBM)
        check("w1<=0", e.download(1)["disp"][0], oracle.sgbm(l, r, p))


# ---- BASELINE.json configurations at full size, against cv2 live (cv2 ships in the image) ---------------------
def _cv2():
    return pytest.importorskip("cv2")


def _cv_sgbm(cv2, l, r, p):
    m = cv2.StereoSGBM_create(minDisparity=p["minDisp"], numDisparities=p["numDisp"], blockSize=p["blockSize"],
                              P1=p["P1"], P2=p["P2"], disp12MaxDiff=p["disp12MaxDiff"], preFilterCap=p["preFilterCap"],
                              uniquenessRatio=p["uniquenessRatio"], speckleWindowSize=p["speckleWindowSize"],
                              speckleRange=p["speckleRange"],
                              mode=cv2.STEREO_SGBM_MODE_HH if p["mode"] == 1 else cv2.STEREO_SGBM_MODE_SGBM)
    return m.compute(l, r)


CFG2 = cases.sgbm_params(minDisp=1, numDisp=64, blockSize=13, speckleWindowSize=150, speckleRange=2)
CFG2_SHIPPED = cases.sgbm_params(minDisp=1, numDisp=128, blockSize=13, speckleWindowSize=150, speckleRange=2)
CFG4 = cases.sgbm_params(numDisp=256, blockSize=5, P1=200, P2=800, disp12MaxDiff=1, uniquenessRatio=10,
                         speckleWindowSize=150, speckleRange=2, mode=1)
CFG5 = cases.sgbm_params(numDisp=256, blockSize=5, P1=200, P2=800)


@pytest.mark.parametrize("p,H,W,B", [(CFG2, 480, 752, 4), (CFG2_SHIPPED, 480, 752, 2), (CFG4, 1080, 1920, 1),
                                     (CFG5, 2160, 3840, 1)],
                         ids=["cfg2_752x480_d64", "sgbm_yml_d128", "cfg4_1080p_d256_hh", "cfg5_4k_d256"])
def test_full_size_vs_cv2(p, H, W, B):
    cv2 = _cv2()
    ls, rs = [], []
    for b in range(B):
        l, r, _ = synth.stereogram(H, W, p["minDisp"], p["numDisp"], seed=b)
        ls.append(l); rs.append(r)
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.compute(np.stack(ls), np.stack(rs), api.STAGE_SGBM)
        out = e.download(B)["disp"]
    for b in range(B):
        check("full/%d" % b, out[b], _cv_sgbm(cv2, ls[b], rs[b], p))
    # the ramp is recovered: median |error| of valid pixels below one disparity step
    l, r, d = synth.stereogram(H, W, p["minDisp"], p["numDisp"], seed=0)
    valid = out[0] > (p["minDisp"] - 1) * 16
    err = np.abs(out[0].astype(np.float32) / 16 - d[:, None].astype(np.float32))[valid]
    assert valid.mean() > 0.5 and np.median(err) < 1.0


def test_cfg1_bm_full_size_vs_cv2():
    cv2 = _cv2()
    p = dict(numDisp=80, blockSize=21, preFilterCap=2, uniquenessRatio=0, textureThreshold=30)   # configs/bm.yml
    l, r, _ = synth.stereogram(480, 752, 0, 80, seed=42)
    m = cv2.StereoBM_create(numDisparities=80, blockSize=21)
    m.setPreFilterCap(2); m.setUniquenessRatio(0); m.setTextureThreshold(30)
    with api.Engine(752, 480) as e:
        e.set_bm_params(**p)
        d = api.bm(api.Stereopair(l, r), e)
    check("cfg1", d, m.compute(l, r))


@pytest.mark.parametrize("nd,bs,cap,uniq,H,W,B", [(80, 21, 2, 0, 480, 752, 7), (256, 21, 31, 10, 1080, 1920, 2),
                                                  (128, 11, 2, 5, 1080, 1920, 3)],
                         ids=["bm_yml_batch7", "1080p_d256_u16", "1080p_d128_bytes"])
def test_bm_batches_full_size_vs_cv2(nd, bs, cap, uniq, H, W, B):
    """StereoBM at full sizes against cv2 live, several different frames per call (a warp's rows straddle frames):
    configs/bm.yml, a 16-bit volume at D = 256 and a byte volume at D = 128."""
    cv2 = _cv2()
    p = dict(numDisp=nd, blockSize=bs, preFilterCap=cap, uniquenessRatio=uniq, textureThreshold=30)
    m = cv2.StereoBM_create(numDisparities=nd, blockSize=bs)
    m.setPreFilterCap(cap); m.setUniquenessRatio(uniq); m.setTextureThreshold(30)
    frames = [synth.stereogram(H, W, 0, nd, seed=100 + b)[:2] for b in range(B)]
    with api.Engine(W, H, max_batch=B) as e:
        e.set_bm_params(**p)
        assert e.info.bm_col8 == (1 if bs * 2 * cap <= 255 else 0)
        e.compute(np.stack([f[0] for f in frames]), np.stack([f[1] for f in frames]), api.STAGE_BM)
        out = e.download(B)["disp"]
    for b in range(B):
        check("bm full/%d" % b, out[b], m.compute(frames[b][0], frames[b][1]))


def test_cfg3_pipeline(oracle):
    """remap(maps of parameters/baseline_small) -> crop -> SGBM cfg 2 -> XYZ -> 81 sub-image + sample-point means."""
    g = synth.load_rectification(cases.GOLDEN_DIR)
    roi = tuple(int(v) for v in g["roi"])
    B = 3
    raws = [synth.stereogram(480, 752, 1, 64, seed=7 + b)[:2] for b in range(B)]
    with api.Engine(752, 480, max_batch=B) as e:
        e.upload_rectify_maps(0, g["m1x"], g["m1y"], roi)
        e.upload_rectify_maps(1, g["m2x"], g["m2y"], roi)
        W, H = e.info.width, e.info.height
        assert (W, H) == (roi[2], roi[3])
        e.set_sgbm_params(**gpu_params(CFG2))
        e.set_Q(g["Q"])
        off = api.dmap_roi_offset(CFG2["numDisp"], W)
        rois = api.subimage_rois(W - off, H, off) + api.samplepoint_rois(W - off, H, off)
        e.set_mean_rois(rois)
        e.compute(np.stack([x[0] for x in raws]), np.stack([x[1] for x in raws]),
                  api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_XYZ | api.STAGE_MEANS)
        out = e.download(B, rect=True, xyz=True, means=True)
    check("rectL/golden", out["rectL"][0], g["rectL"])
    check("rectR/golden", out["rectR"][0], g["rectR"])
    for b in range(B):
        rl = oracle.remap(raws[b][0], g["m1x"], g["m1y"], roi)
        rr = oracle.remap(raws[b][1], g["m2x"], g["m2y"], roi)
        check("rectL/%d" % b, out["rectL"][b], rl)
        check("rectR/%d" % b, out["rectR"][b], rr)
        disp = oracle.sgbm(rl, rr, CFG2)
        check("disp/%d" % b, out["disp"][b], disp)
        xyz, valid = oracle.reproject(disp, g["Q"])
        v = valid.astype(bool)
        np.testing.assert_allclose(out["xyz"][b][v], xyz[v], rtol=1e-5)
        want = np.array([oracle.mean(disp, r_) for r_ in rois], np.float32)
        np.testing.assert_array_equal(out["means"][b], want)


def test_determinism_and_linearity_properties():
    """Size-independent properties at full size: rerun == same bits; a frame's result does not depend on its
    batch neighbours; shifting both images by a constant intensity leaves the x-Sobel channel unchanged but not
    the raw channel, so only idempotence-type properties are asserted."""
    p, H, W, B = CFG2, 480, 752, 6
    ls, rs = zip(*[synth.stereogram(H, W, 1, 64, seed=100 + b)[:2] for b in range(B)])
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.compute(np.stack(ls), np.stack(rs), api.STAGE_SGBM)
        a = e.download(B)["disp"]
        e.compute(np.stack(ls[::-1]), np.stack(rs[::-1]), api.STAGE_SGBM)
        b = e.download(B)["disp"]
        check("permuted batch", b[::-1], a)
        e.compute(ls[2], rs[2], api.STAGE_SGBM)
        check("single", e.download(1)["disp"][0], a[2])


def test_cpp_mirror_end_to_end(oracle, tmp_path):
    """C++ host code -> disparity.h mirror -> C ABI -> CUDA, on ROI views with step > cols, against the oracle."""
    import subprocess
    from test_host_cpu import _build_shim_demo
    exe = _build_shim_demo(tmp_path)
    H, W = 120, 300
    l, r, _ = synth.stereogram(H, W, 1, 128, seed=9)
    (tmp_path / "l.raw").write_bytes(l.tobytes())
    (tmp_path / "r.raw").write_bytes(r.tobytes())
    yml = tmp_path / "sgbm.yml"     # verbatim reference configs/sgbm.yml
    yml.write_text("%YAML:1.0\nminDisp: 1\nnumDisp: 128\nblockSize: 13\ndisp12MaxDiff: 0\npreFilterCap: 0\n"
                   "uniquenessRatio: 0\nspeckleWindowSize: 150\nspeckleWindowRange: 2\nmode: 0\n")
    subprocess.check_call([exe, str(yml), str(tmp_path / "l.raw"), str(tmp_path / "r.raw"), str(W), str(H),
                           str(tmp_path / "out.raw")])
    got = np.frombuffer((tmp_path / "out.raw").read_bytes(), np.int16).reshape(H, W)
    check("cpp mirror", got, oracle.sgbm(l, r, CFG2_SHIPPED))


def test_d256_large_block_fits_shared_memory(oracle):
    """D = 256 with the largest block size the contract allows (bs 11: 121*93 + P2 <= 32767) -- the cost kernel's
    shared-memory footprint (staging copies + row ring + producer ring) is at its maximum here."""
    p = cases.sgbm_params(numDisp=256, blockSize=11, P1=8, P2=32, uniquenessRatio=5)
    H, W = 30, 300
    l, r = synth.random_pair(H, W, seed=77)
    with api.Engine(W, H) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.compute(l, r, api.STAGE_SGBM)
        check("d256 bs11", e.download(1)["disp"][0], oracle.sgbm(l, r, p))


def test_worst_case_cost_kernel_footprint(oracle):
    """The parameter set with the largest shared-memory footprint of the cost kernel inside the contract:
    D = 256, preFilterCap 97 (pixel cost no longer fits a byte -> 16-bit row ring), blockSize 11."""
    p = cases.sgbm_params(numDisp=256, blockSize=11, P1=8, P2=32, preFilterCap=97)
    H, W = 28, 290
    l, r = synth.random_pair(H, W, seed=78)
    with api.Engine(W, H) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.compute(l, r, api.STAGE_SGBM)
        check("d256 cap97 bs11", e.download(1)["disp"][0], oracle.sgbm(l, r, p))


def test_cpp_frame_loop_demo(tmp_path):
    """examples/mean_plain_demo.cpp: the reference's application skeleton (worker std::thread + condition variable,
    trgt/mean_plain.cpp:62-82, trgt/demo.cpp:215-276) running on the engine with a synthetic frame source."""
    import subprocess
    root = os.path.dirname(cases.GOLDEN_DIR.rstrip("/").rsplit("/", 1)[0])
    libdir = os.path.join(root, "mvstereovision3_b200")
    exe = str(tmp_path / "mean_plain_demo")
    subprocess.check_call(["g++", "-std=c++11", "-O2", "-pthread", "-Wall", "-I" + os.path.join(root, "include"),
                           os.path.join(root, "examples", "mean_plain_demo.cpp"), "-L" + libdir, "-lmvsv",
                           "-Wl,-rpath," + libdir, "-o", exe])
    out = subprocess.check_output([exe, "--frames", "30"], timeout=120).decode()
    assert "Disparity Framerate:" in out and "Detection Framerate:" in out, out
    first = out.splitlines()[0].split()
    assert first[0] == "frames" and int(first[1]) >= 30 and first[3] == "752x479"
    assert int(first[first.index("map") + 7]) > 100000        # most of the last map is valid


@pytest.mark.parametrize("H", [1, 2, 3, 4, 7])
@pytest.mark.parametrize("nc", [2, 4])
def test_fused_sweep_degenerate_strips(oracle, H, nc):
    """Border hand-off corner cases: frames of 1..7 rows (fewer rows than border-record slots) and column strips of
    one or two pixels (a strip's first pixel is also its last), MODE_HH so that both sweeps run."""
    p = cases.sgbm_params(numDisp=16, blockSize=3, P1=7, P2=40, uniquenessRatio=5, mode=1)
    W = 16 + 5                                   # W1 = 5 -> strips of 1 or 2 columns with 4 strips
    l, r = synth.random_pair(H, W, seed=90 + H)
    with api.Engine(W, H) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.debug_set_flags(nc << 8)
        assert e.info.sgbm_td_cluster == nc
        e.compute(l, r, api.STAGE_SGBM)
        check("H=%d nc=%d" % (H, nc), e.download(1)["disp"][0], oracle.sgbm(l, r, p))


def test_io_slots_pipeline_in_one_engine(oracle):
    """mvsv_set_io_slots(2): compute k+1 is submitted before the results of compute k are fetched (age 1); the
    copies overlap the kernels inside ONE engine and every batch still equals the oracle (bench.py's e2e loop)."""
    p = cases.sgbm_params(minDisp=1, numDisp=32, blockSize=5, P1=20, P2=90, uniquenessRatio=5, speckleWindowSize=30, speckleRange=2)
    H, W, B = 60, 200, 6
    batches = []
    for k in range(5):
        ls, rs = zip(*[synth.random_pair(H, W, seed=100 * k + b) for b in range(B)])
        batches.append((np.stack(ls), np.stack(rs)))
    want = [np.stack([oracle.sgbm(L[b], R[b], p) for b in range(B)]) for L, R in batches]
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.set_Q(cases.Q_REFERENCE)
        e.set_mean_rois([(40, 5, 50, 40), (100, 10, 20, 20)])
        e.set_io_slots(2)
        got, means = [None] * len(batches), [None] * len(batches)
        stages = api.STAGE_SGBM | api.STAGE_MEANS
        e.compute(batches[0][0], batches[0][1], stages)
        for k in range(1, len(batches)):
            e.compute(batches[k][0], batches[k][1], stages)
            r = e.download(B, means=True, age=1)
            got[k - 1], means[k - 1] = r["disp"], r["means"]
        r = e.download(B, means=True)
        got[-1], means[-1] = r["disp"], r["means"]
        with pytest.raises(api.MvsvError):
            e.download(B, age=2)
        e.set_io_slots(1)
        e.compute(batches[2][0], batches[2][1], api.STAGE_SGBM)
        check("back to one slot", e.download(B)["disp"], want[2])
    for k in range(len(batches)):
        check("batch %d" % k, got[k], want[k])
        for b in range(B):
            m = np.array([oracle.mean(want[k][b], roi) for roi in [(40, 5, 50, 40), (100, 10, 20, 20)]], np.float32)
            np.testing.assert_array_equal(means[k][b], m)


def test_rejected_compute_keeps_the_last_results(oracle):
    """Two I/O slots, three computes, the third rejected (row stride below the width): the rejected call takes no slot,
    so download() still returns the second batch and age 1 the first, never the frames of an older compute."""
    p = cases.sgbm_params(numDisp=16, blockSize=5)
    H, W, B = 40, 96, 2
    batches = []
    for k in range(3):
        ls, rs = zip(*[synth.random_pair(H, W, seed=500 + 10 * k + b) for b in range(B)])
        batches.append((np.stack(ls), np.stack(rs)))
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.set_io_slots(2)
        for L, R in batches[:2]:
            e.compute(L, R, api.STAGE_SGBM)
        L, R = batches[2]
        rc = e._lib.mvsv_compute(e._ctx, L.ctypes.data, W - 1, R.ctypes.data, W, L.strides[0], B, api.STAGE_SGBM)
        assert rc == -1, rc                                  # MVSV_ERR_INVALID
        got = e.download(B)["disp"], e.download(B, age=1)["disp"]
    for b in range(B):
        check("second batch/%d" % b, got[0][b], oracle.sgbm(batches[1][0][b], batches[1][1][b], p))
        check("first batch/%d" % b, got[1][b], oracle.sgbm(batches[0][0][b], batches[0][1][b], p))


def test_io_slots_with_rectification_and_resize(oracle):
    """Two I/O slots with the cfg-3 stage set (RECTIFY | SGBM | XYZ | MEANS), maps and ROIs installed before
    set_io_slots(2) as bench.py does, then a geometry change (set_resize) while both slots are live: the change drops
    the results the slots held, and every batch, fetched one call late, equals the oracle."""
    H, W, B = 96, 140, 2
    mx, my = cases.warp_maps(H, W, 2)
    roi = (4, 2, W - 20, H - 10)
    p = cases.sgbm_params(numDisp=16, blockSize=5)
    stages = api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_XYZ | api.STAGE_MEANS
    raws = []
    for k in range(6):
        ls, rs = zip(*[synth.random_pair(H, W, seed=600 + 10 * k + b) for b in range(B)])
        raws.append((np.stack(ls), np.stack(rs)))
    with api.Engine(W, H, max_batch=B) as e:
        e.upload_rectify_maps(0, mx, my, roi)
        e.upload_rectify_maps(1, mx, my, roi)
        e.set_sgbm_params(**gpu_params(p))
        e.set_Q(cases.Q_REFERENCE)
        for factor, batches in ((0, raws[:3]), (0.5, raws[3:])):
            if factor:
                e.set_resize(factor)
                with pytest.raises(api.MvsvError) as ex:
                    e.download(B, age=1)
                assert ex.value.code == -4
            w, h = e.info.width, e.info.height
            rois = [(w // 2, h // 4, w // 3, h // 2), (2, 2, 10, 10)]
            e.set_mean_rois(rois)
            if not factor:
                e.set_io_slots(2)
            got = []
            e.compute(batches[0][0], batches[0][1], stages)
            for L, R in batches[1:]:
                e.compute(L, R, stages)
                got.append(e.download(B, rect=True, xyz=True, means=True, age=1))
            got.append(e.download(B, rect=True, xyz=True, means=True))
            for k, (L, R) in enumerate(batches):
                for b in range(B):
                    rl, rr = oracle.remap(L[b], mx, my, roi), oracle.remap(R[b], mx, my, roi)
                    if factor:
                        rl, rr = oracle.resize(rl, factor), oracle.resize(rr, factor)
                    tag = "x%s/batch %d/%d" % (factor, k, b)
                    check(tag + "/rectL", got[k]["rectL"][b], rl)
                    check(tag + "/rectR", got[k]["rectR"][b], rr)
                    disp = oracle.sgbm(rl, rr, p)
                    check(tag + "/disp", got[k]["disp"][b], disp)
                    xyz, valid = oracle.reproject(disp, cases.Q_REFERENCE)
                    v = valid.astype(bool)
                    np.testing.assert_allclose(got[k]["xyz"][b][v], xyz[v], rtol=1e-5)
                    want = np.array([oracle.mean(disp, r_) for r_ in rois], np.float32)
                    np.testing.assert_array_equal(got[k]["means"][b], want)


def test_mean_rois_dropped_on_geometry_change(oracle):
    """ROIs are coordinates of the current map: a geometry change drops them, MEANS then fails with MVSV_ERR_STATE
    until they are set again (and never launches with stale ROIs or a freed result buffer)."""
    H, W = 96, 140
    img, img2 = synth.random_pair(H, W, seed=5)
    mx, my = cases.warp_maps(H, W, 1)
    p = cases.sgbm_params(numDisp=16, blockSize=5)
    with api.Engine(W, H, max_batch=1) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.set_mean_rois([(100, 60, 30, 30)])
        e.compute(img, img2, api.STAGE_SGBM | api.STAGE_MEANS)
        e.download(1, means=True)
        roi = (4, 2, W - 40, H - 30)                      # the old ROI now lies outside the map
        e.upload_rectify_maps(0, mx, my, roi)
        e.upload_rectify_maps(1, mx, my, roi)
        assert e.info.num_rois == 0
        with pytest.raises(api.MvsvError) as ex:
            e.compute(img, img2, api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_MEANS)
        assert ex.value.code == -4
        e.set_mean_rois([(10, 10, 30, 30)])
        e.compute(img, img2, api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_MEANS)
        out = e.download(1, means=True)
        rl, rr = oracle.remap(img, mx, my, roi), oracle.remap(img2, mx, my, roi)
        disp = oracle.sgbm(rl, rr, p)
        check("disp", out["disp"][0], disp)
        np.testing.assert_array_equal(out["means"][0], np.array([oracle.mean(disp, (10, 10, 30, 30))], np.float32))
        with pytest.raises(ValueError):
            e.download(2)                                  # more frames than the last compute held


@pytest.mark.parametrize("nc", [1, 2, 4, 8])
def test_halo_handoff_soak(oracle, nc):
    """Determinism soak of the strip-border hand-off of the fused sweep (tagged records through L2, neighbouring
    warps paced by shared-memory progress counters): 100 x 24 small MODE_HH frames (two sweeps each) at 1, 2, 4 and
    8 strips per frame, each result identical to the oracle."""
    p = cases.sgbm_params(minDisp=1, numDisp=32, blockSize=5, P1=20, P2=90, uniquenessRatio=5, disp12MaxDiff=1,
                          speckleWindowSize=30, speckleRange=2, mode=1)
    H, W, B = 37, 171, 24
    ls, rs = zip(*[synth.random_pair(H, W, seed=s) for s in range(B)])
    L, R = np.stack(ls), np.stack(rs)
    want = np.stack([oracle.sgbm(ls[b], rs[b], p) for b in range(B)])
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.debug_set_flags(nc << 8)
        assert e.info.sgbm_td_cluster == nc
        for it in range(100):
            e.compute(L, R, api.STAGE_SGBM)
            got = e.download(B)["disp"]
            assert np.array_equal(got, want), "cluster %d, iteration %d: %d pixels differ" % (nc, it, int((got != want).sum()))


@pytest.mark.parametrize("D,nc,B", [(32, 8, 60), (128, 16, 30), (256, 37, 9)])
def test_sweep_walks_several_frames_per_cta(oracle, D, nc, B):
    """More frames than frame slots (B > floor(148 / strips)): every CTA of the persistent sweep walks several frames,
    warps and strips drift across the frame boundaries, and all frames (MODE_HH: two sweeps) still equal the oracle --
    the frame-boundary case of the border hand-off, at one, two and four lanes per pixel."""
    p = cases.sgbm_params(minDisp=0, numDisp=D, blockSize=3, P1=20, P2=90, uniquenessRatio=5, disp12MaxDiff=1, mode=1)
    H, W = 9, D + 150
    ls, rs = zip(*[synth.random_pair(H, W, seed=300 + s) for s in range(6)])
    L, R = np.stack([ls[b % 6] for b in range(B)]), np.stack([rs[b % 6] for b in range(B)])
    want = [oracle.sgbm(ls[b], rs[b], p) for b in range(6)]
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.debug_set_flags(nc << 8)
        assert e.info.sgbm_td_cluster == nc and B > 148 // nc
        for it in range(20):
            e.compute(L, R, api.STAGE_SGBM)
            got = e.download(B)["disp"]
            for b in range(B):
                assert np.array_equal(got[b], want[b % 6]), "iteration %d frame %d: %d pixels differ" % (
                    it, b, int((got[b] != want[b % 6]).sum()))


@pytest.mark.parametrize("kw", [
    dict(minDisp=1, numDisp=64, blockSize=13, speckleWindowSize=150, speckleRange=2),             # cfg 2 (P2 -> 5)
    dict(numDisp=32, blockSize=5, P1=3, P2=30, mode=1, uniquenessRatio=10, disp12MaxDiff=1),      # MODE_HH, 8 * 30 <= 255
    dict(numDisp=128, blockSize=9, P1=8, P2=51, uniquenessRatio=5),                               # two lanes per pixel
    dict(numDisp=256, blockSize=3, P1=2, P2=31, mode=1),                                          # four lanes, MODE_HH
    dict(numDisp=48, blockSize=7, P1=10, P2=50, preFilterCap=63),                                 # 24 registers per lane
    dict(numDisp=16, blockSize=11, P1=1, P2=2, preFilterCap=100),                                 # costs near the int16 limit
    dict(numDisp=16, blockSize=11, P1=1, P2=2, preFilterCap=31, mode=1),                          # byte form with saturated sums
], ids=["cfg2", "hh_d32", "d128", "d256_hh", "d48", "d16_wide", "d16_hh_saturating"])
def test_byte_form_of_S_equals_16bit_form(oracle, kw):
    """When npaths * P2 <= 255 the aggregated volume is kept as one byte per cell (sum of the paths' excesses over
    C); the same parameters with the byte form forced off (debug flag bit 1) and the oracle must give the same final S
    volume and the same disparities."""
    p = cases.sgbm_params(**kw)
    H, W = 41, p["numDisp"] + 93
    l, r = synth.random_pair(H, W, seed=11)
    l2, r2, _ = synth.stereogram(H, W, p["minDisp"], p["numDisp"], seed=12)
    L, R = np.stack([l, l2]), np.stack([r, r2])
    res = {}
    for flags in (1, 3):
        with api.Engine(W, H, max_batch=2) as e:
            e.set_sgbm_params(**gpu_params(p))
            e.debug_set_flags(flags | (0xfe << 8))          # the sweep also for this batch of two
            e.compute(L, R, api.STAGE_SGBM)
            res[flags] = (e.download(2)["disp"], e.debug_read(1, 2), e.info.sgbm_s8)
    bs = p["blockSize"] | 1
    fast = 3 * (bs * bs * (2 * (max(p["preFilterCap"], 15) | 1) + 63) + max(p["P2"], 5)) <= 65535
    assert res[1][2] == (1 if fast else 0) and res[3][2] == 0, "byte form expected by default (row sums fit 16 bits), 16-bit form when forced"
    for b, (a_, b_) in enumerate(((l, r), (l2, r2))):
        disp, Cv, Sv, rawv = oracle.sgbm(a_, b_, p, want_volumes=True, want_raw=True)
        if kw.get("mode") == 1 and kw["blockSize"] == 11 and b == 0:
            assert (Sv == 32767).sum() > 10, "this case is meant to saturate some path sums"
        for flags in (1, 3):
            check("S/%d/%d" % (flags, b), res[flags][1][b], Sv)
            check("disp/%d/%d" % (flags, b), res[flags][0][b], disp)


def test_two_devices_in_one_process(oracle):
    """One process, one engine per GPU (INTEGRATION.md section 5): kernel attributes (dynamic shared memory of the sweep
    and the StereoBM column sums) are configured per device.  Needs two GPUs; skipped otherwise."""
    import ctypes
    try:
        rt = ctypes.CDLL("libcudart.so")
    except OSError:
        rt = None
    n = ctypes.c_int(0)
    if rt is None or rt.cudaGetDeviceCount(ctypes.byref(n)) != 0 or n.value < 2:
        pytest.skip("needs two CUDA devices")
    p = cases.sgbm_params(minDisp=1, numDisp=64, blockSize=9, speckleWindowSize=50, speckleRange=2)
    bmp = dict(numDisp=32, blockSize=9, preFilterCap=31, uniquenessRatio=5, textureThreshold=10)
    H, W = 60, 260
    l, r, _ = synth.stereogram(H, W, 1, 64, seed=3)
    want = oracle.sgbm(l, r, p)
    want_bm = oracle.bm(l, r, bmp)
    for dev in (1, 0, 1):
        with api.Engine(W, H, max_batch=1, device=dev) as e:
            e.set_sgbm_params(**gpu_params(p))
            e.compute(l, r, api.STAGE_SGBM)
            check("sgbm on device %d" % dev, e.download(1)["disp"][0], want)
            e.set_bm_params(**bmp)
            e.compute(l, r, api.STAGE_BM)
            check("bm on device %d" % dev, e.download(1)["disp"][0], want_bm)


@pytest.mark.parametrize("p,B", [(CFG2, 148), (CFG2_SHIPPED, 74)], ids=["cfg2_b148", "sgbm_yml_d128_b74"])
def test_full_bench_batch_twins_agree(p, B):
    """The bench batches at full size (every sweep CTA walks several frames, all SMs busy): the batch holds four distinct
    pairs repeated, every copy must equal its twin on every repetition, and one copy of each must equal cv2.  This is the
    configuration in which the frame-boundary pacing race of the sweep showed (tools/determinism_check.py)."""
    cv2 = _cv2()
    H, W = 480, 752
    gen = [synth.stereogram(H, W, p["minDisp"], p["numDisp"], seed=50 + s)[:2] for s in range(4)]
    L = np.stack([gen[b % 4][0] for b in range(B)])
    R = np.stack([gen[b % 4][1] for b in range(B)])
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**gpu_params(p))
        for it in range(3):
            e.compute(L, R, api.STAGE_SGBM)
            d = e.download(B)["disp"]
            for b in range(4, B):
                assert np.array_equal(d[b], d[b % 4]), "repetition %d: frame %d differs from its twin in %d pixels" % (
                    it, b, int((d[b] != d[b % 4]).sum()))
    for s in range(4):
        check("vs cv2 / %d" % s, d[s], _cv_sgbm(cv2, gen[s][0], gen[s][1], p))
