"""SGBM and StereoBM on inputs where costs tie (tests/hard_inputs.py): textureless, saturated and black regions, exact
matches, periodic structure.  The matchers' winner-take-all, uniqueness, sub-pixel and left-right-check code decides
ties by explicit rules (first minimum; lowest cost and then the largest / smallest x in the scatter tables), and blurred
noise almost never reaches those rules.

CPU: the references (the C oracle, tests/bm_filters_ref.py) against cv2 4.13.0 on every family, and coverage: every
family reaches the case it is named for (measured on the reference's own volumes, so the generators cannot quietly
degenerate).  GPU: the CUDA path against the references stage by stage, on every code path, bit-exact."""
import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

import bm_filters_ref as ref
import cases
import hard_inputs as hi
from test_bm_filters import cv_bm
from test_gpu_parity import CFG2, CFG2_SHIPPED, CFG4, _cv_sgbm, check, gpu_params
from test_property import bm_case, sgbm_case

FAMILIES = list(hi.FAMILIES) + ["scene"]
MAX_COST = 32767


def frame(fam, H, W, minD, D, seed=0):
    if fam == "scene":
        return hi.scene(H, W, max(minD, 0), D, seed)
    return hi.pair(fam, H, W, D, seed)


# ---- coverage measures on the references' volumes -------------------------------------------------------------------
def _scatter_ties(cost, target, ok):
    """Fraction of the pixels `ok` whose scatter target (same row) also receives another pixel at the same, lowest cost:
    the case that the left-right check's tie rule decides.  target: column index per pixel, any integer range."""
    H, W = cost.shape
    ys, xs = np.nonzero(ok)
    if len(ys) == 0:
        return 0.0
    t = target[ys, xs]
    key = ys.astype(np.int64) * (int(t.max() - t.min()) + 1) + (t - t.min())
    c = cost[ys, xs].astype(np.int64)
    best = np.full(int(key.max()) + 1, np.iinfo(np.int64).max)
    np.minimum.at(best, key, c)
    at_min = c == best[key]
    n = np.bincount(key[at_min], minlength=len(best))
    return float((at_min & (n[key] >= 2)).sum()) / (H * W)


def sgbm_coverage(oracle, l, r, p):
    """Per-pixel fractions (over the H x W1 domain) of the tie cases of SGBM's winner-take-all, from the oracle's S."""
    _, _, S, _ = oracle.sgbm(l, r, p, want_volumes=True)
    S = S.astype(np.int64)
    D = S.shape[2]
    best = S.argmin(2)
    minS = S.min(2)
    k = np.arange(D)
    far = np.abs(k[None, None] - best[..., None]) > 1
    far_tie = ((S == minS[..., None]) & far).any(2)
    live = minS < MAX_COST
    xs = np.arange(S.shape[1])[None, :]
    return dict(
        sgbm_far_tie=float((far_tie & live).mean()),
        sgbm_zero=float((minS == 0).mean()),
        sgbm_uniq_tie=float((far_tie & (minS > 0) & live).mean()),     # rejected by any uniquenessRatio > 0
        sgbm_lr_tie=_scatter_ties(minS, xs - best, live),
    )


def bm_volume(pl, pr, p):
    """Texture sums and the SAD volume [D, rows, width1 columns] of StereoBM's match domain (bm_filters_ref's clamps)."""
    H, W = pl.shape
    D, bs, cap = p["numDisp"], p["blockSize"], p["preFilterCap"]
    w2, lofs, width1 = bs // 2, D - 1, W - D + 1
    j = np.arange(-w2, width1 + w2)
    cl = np.clip(j, -lofs, W - lofs - 1) + lofs
    cr = np.clip(j, 0, W - D)
    L, R = pl.astype(np.int64), pr.astype(np.int64)
    tex = ref._box(np.abs(L[:, cl] - cap), bs)
    return tex, np.stack([ref._box(np.abs(L[:, cl] - R[:, cr + k]), bs) for k in range(D)])


def bm_coverage(oracle, l, r, p):
    """Fractions of StereoBM's match domain in each tie case, and of prefiltered pixels at the clip limits."""
    _, pl, pr = oracle.bm(l, r, p, want_prefilter=True)
    cap, D = p["preFilterCap"], p["numDisp"]
    tex, sad = bm_volume(pl, pr, p)
    mind = sad.argmin(0)
    minsad = sad.min(0)
    k = np.arange(D)[:, None, None]
    far = np.abs(k - mind[None]) > 1
    pk = np.take_along_axis(sad, np.where(mind + 1 < D, mind + 1, D - 2)[None], 0)[0]
    nk = np.take_along_axis(sad, np.where(mind > 0, mind - 1, 1)[None], 0)[0]
    den = pk + nk - 2 * minsad + np.abs(pk - nk)
    disp, cost = ref.match_domain(pl, pr, dict(p, textureThreshold=0, uniquenessRatio=0))
    X = np.arange(disp.shape[1])[None, :]
    both = np.concatenate([pl.ravel(), pr.ravel()])
    return dict(
        bm_far_tie=float(((sad == minsad[None]) & far).any(0).mean()),
        bm_zero=float((minsad == 0).mean()),
        bm_next_tie=float(((pk == minsad) | (nk == minsad)).mean()),       # ties at mind +- 1: the uniqueness count's exemptions
        bm_den0=float((den == 0).mean()),
        bm_notex=float((tex == 0).mean()),
        bm_pre_lo=float((both == 0).mean()),
        bm_pre_hi=float((both == 2 * cap).mean()),
        bm_lr_tie=_scatter_ties(cost, X - ((disp + 8) >> 4), disp != ref.FILT),
    )


COV_SGBM = cases.sgbm_params(numDisp=32, blockSize=5, P1=8, P2=32, uniquenessRatio=10)
COV_BM = dict(numDisp=32, blockSize=9, preFilterCap=31, uniquenessRatio=0, textureThreshold=0)
COV_H, COV_W = 60, 200

# what each family must reach: minimum fractions of the measures above (about half of what each one measures at
# COV_H x COV_W; SGBM scatter ties are rare on any input, so their floor is low)
REACHES = {
    "zeros": dict(sgbm_zero=0.9, bm_zero=0.9, bm_far_tie=0.9, bm_next_tie=0.9, bm_den0=0.9, bm_notex=0.9),
    "whites": dict(sgbm_zero=0.9, bm_zero=0.9, bm_far_tie=0.9, bm_next_tie=0.9, bm_den0=0.9, bm_notex=0.9),
    "flat_levels": dict(sgbm_far_tie=0.3, sgbm_uniq_tie=0.3, bm_far_tie=0.9, bm_den0=0.9),
    "same": dict(sgbm_zero=0.5, bm_zero=0.5, bm_pre_lo=0.2, bm_pre_hi=0.2),
    "exact_shift": dict(sgbm_zero=0.5, bm_zero=0.5, bm_pre_lo=0.2, bm_pre_hi=0.2),
    "stripes": dict(sgbm_far_tie=0.5, sgbm_zero=0.5, bm_far_tie=0.5, bm_zero=0.5, bm_pre_lo=0.1, bm_pre_hi=0.1),
    "stripes_offset": dict(sgbm_far_tie=0.5, sgbm_uniq_tie=0.5, bm_far_tie=0.5),
    "stripes_noise": dict(sgbm_far_tie=0.01, sgbm_uniq_tie=0.01, sgbm_lr_tie=0.01, bm_lr_tie=0.3),
    "checker": dict(sgbm_far_tie=0.5, sgbm_zero=0.5, bm_far_tie=0.5, bm_zero=0.5),
    "quantised": dict(sgbm_zero=0.5, bm_zero=0.5),
    "dots": dict(sgbm_zero=0.5, bm_zero=0.5, bm_pre_lo=0.08, bm_pre_hi=0.08),
    "hramp": dict(sgbm_zero=0.5, bm_far_tie=0.4, bm_next_tie=0.4, bm_den0=0.4, bm_lr_tie=0.03),
    "vramp": dict(sgbm_zero=0.5, bm_far_tie=0.5, bm_den0=0.5, bm_notex=0.5),
    "flat_patches": dict(sgbm_zero=0.5, bm_zero=0.5, bm_far_tie=0.05, bm_notex=0.05, bm_lr_tie=0.03),
    "scene": dict(sgbm_zero=0.35, bm_far_tie=0.05, bm_den0=0.01, bm_notex=0.03, bm_lr_tie=0.02),
}


@pytest.fixture(scope="module")
def coverage(oracle):
    out = {}
    for i, fam in enumerate(FAMILIES):
        l, r = frame(fam, COV_H, COV_W, 0, 32, seed=i)
        out[fam] = dict(sgbm_coverage(oracle, l, r, COV_SGBM), **bm_coverage(oracle, l, r, COV_BM))
    return out


@pytest.mark.parametrize("fam", FAMILIES)
def test_family_reaches_its_case(coverage, fam):
    got = coverage[fam]
    low = {k: (round(got[k], 3), v) for k, v in REACHES[fam].items() if not got[k] >= v}
    assert not low, "%s: measure (got, wanted at least): %s" % (fam, low)


def test_families_are_deterministic():
    for fam in FAMILIES:
        a, b = frame(fam, 30, 120, 1, 32, seed=5), frame(fam, 30, 120, 1, 32, seed=5)
        assert a[0].dtype == np.uint8 and a[0].shape == (30, 120) and a[1].shape == (30, 120)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), fam


# ---- A. the references against cv2 (CPU) ----------------------------------------------------------------------------
@pytest.mark.parametrize("case", cases.SGBM_CASES, ids=[c[0] for c in cases.SGBM_CASES])
def test_oracle_sgbm_vs_cv2_on_hard_inputs(oracle, case):
    cv2 = pytest.importorskip("cv2")
    name, p, H, W = case
    for i, fam in enumerate(FAMILIES):
        l, r = frame(fam, H, W, p["minDisp"], p["numDisp"], seed=i)
        check("%s/%s" % (name, fam), oracle.sgbm(l, r, p), _cv_sgbm(cv2, l, r, p))


def bm_families(p):
    """Every family; above blockSize 63, where the oracle's StereoBM (O(blockSize^2) per pixel) takes about a second per
    frame, a flat, a periodic, a ramp and the scene family."""
    return FAMILIES if p["blockSize"] <= 63 else ["flat_levels", "stripes", "hramp", "scene"]


def bm_variants(p):
    """The case itself; textureThreshold 0 (flat windows reach the sub-pixel step) with uniquenessRatio 10 and 0; the
    left-right check (disp12MaxDiff 0, 1) and the speckle filter where cv2 computes them deterministically
    (preFilterCap <= 31, blockSize <= 21)."""
    lr = p["preFilterCap"] <= 31 and p["blockSize"] <= 21
    return [p, dict(p, textureThreshold=0, uniquenessRatio=10, **(dict(disp12MaxDiff=0) if lr else {})),
            dict(p, textureThreshold=0, uniquenessRatio=0, **(dict(disp12MaxDiff=1, speckleWindowSize=50, speckleRange=16) if lr else {}))]


@pytest.mark.parametrize("case", cases.BM_CASES, ids=[c[0] for c in cases.BM_CASES])
def test_reference_bm_vs_cv2_on_hard_inputs(oracle, case):
    cv2 = pytest.importorskip("cv2")
    name, p, H, W = case
    for i, fam in enumerate(bm_families(p)):
        l, r = frame(fam, H, W, 0, p["numDisp"], seed=i)
        for v in bm_variants(p):
            check("%s/%s/%s" % (name, fam, v), ref.bm(oracle, l, r, v), cv_bm(cv2, l, r, v))


# ---- GPU ------------------------------------------------------------------------------------------------------------
def family_pairs():
    """Two different families per batch of two; every family appears."""
    f = FAMILIES
    return [(f[i], f[(i + 1) % len(f)]) for i in range(0, len(f), 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("sweep", [0, 0xfe], ids=["auto", "sweep"])
@pytest.mark.parametrize("case", cases.SGBM_CASES, ids=[c[0] for c in cases.SGBM_CASES])
def test_sgbm_stages_on_hard_inputs(oracle, case, sweep):
    """B. C, S, raw (before median and speckle, which can hide a wrong winner), median and the final map of every
    family against the oracle, two different families per batch; the independent passes and the fused sweep."""
    from mvstereovision3_b200 import api
    name, p, H, W = case
    with api.Engine(W, H, max_batch=2) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.debug_set_flags(1 | (sweep << 8))
        for j, fams in enumerate(family_pairs()):
            frames = [frame(f, H, W, p["minDisp"], p["numDisp"], seed=j) for f in fams]
            e.compute(np.stack([a for a, _ in frames]), np.stack([b for _, b in frames]), api.STAGE_SGBM)
            out = e.download(2)["disp"]
            Cg, Sg, raw, med = (e.debug_read(w, 2) for w in (0, 1, 2, 4))
            for b, f in enumerate(fams):
                disp, Cv, Sv, rawv = oracle.sgbm(frames[b][0], frames[b][1], p, want_volumes=True, want_raw=True)
                tag = "%s/%s/" % (name, f)
                if Cv is not None:
                    check(tag + "C", Cg[b], Cv)
                    check(tag + "S", Sg[b], Sv)
                check(tag + "raw", raw[b], rawv)
                check(tag + "median", med[b], oracle.median3(rawv))
                check(tag + "disp", out[b], disp)


TIE_FAMILIES = ["stripes", "stripes_offset", "checker", "flat_levels", "flat_patches", "stripes_noise", "scene", "hramp"]


@pytest.mark.gpu
@pytest.mark.parametrize("nc", [1, 2, 4, 8, 0xff], ids=["nc1", "nc2", "nc4", "nc8", "passes"])
@pytest.mark.parametrize("mode", [0, 1], ids=["sgbm", "hh"])
@pytest.mark.parametrize("D", [32, 64, 128, 256])
def test_sgbm_paths_on_tie_frames(oracle, D, mode, nc):
    """C. Every aggregation path on tie-heavy frames: 1, 2, 4, 8 strips per frame and the independent passes; the byte
    and the 16-bit form of S (flag bit 1) with the vector and the scalar 3x3 median (flag bit 2, W % 4 == 0); one, two
    and four lanes per pixel; MODE_SGBM and MODE_HH; uniquenessRatio 0 and > 0, disp12MaxDiff -1, 0 and 1."""
    from mvstereovision3_b200 import api
    H, W = 26, D + 60
    i = [32, 64, 128, 256].index(D) * 2 + mode
    fams = (TIE_FAMILIES[i % len(TIE_FAMILIES)], TIE_FAMILIES[(i + 3) % len(TIE_FAMILIES)])
    frames = [frame(f, H, W, 0, D, seed=i) for f in fams]
    L, R = np.stack([a for a, _ in frames]), np.stack([b for _, b in frames])
    for uniq, d12 in ((0, -1), (10, 0), (5, 1)):
        p = cases.sgbm_params(numDisp=D, blockSize=5, P1=8, P2=30, uniquenessRatio=uniq, disp12MaxDiff=d12, mode=mode,
                              speckleWindowSize=20, speckleRange=1)
        want = [oracle.sgbm(a, b, p, want_volumes=True, want_raw=True) for a, b in frames]
        for flags in (1, 1 | 2 | 4):
            with api.Engine(W, H, max_batch=2) as e:
                e.set_sgbm_params(**gpu_params(p))
                e.debug_set_flags(flags | (nc << 8))
                assert e.info.sgbm_td_cluster == (0 if nc == 0xff else nc)
                e.compute(L, R, api.STAGE_SGBM)
                assert e.info.sgbm_s8 == (1 if nc != 0xff and not flags & 2 else 0)
                out, Sg, raw, med = e.download(2)["disp"], e.debug_read(1, 2), e.debug_read(2, 2), e.debug_read(4, 2)
            for b, f in enumerate(fams):
                disp, _, Sv, rawv = want[b]
                tag = "%s/u%d/d12 %d/flags %d/" % (f, uniq, d12, flags)
                check(tag + "S", Sg[b], Sv)
                check(tag + "raw", raw[b], rawv)
                check(tag + "median", med[b], oracle.median3(rawv))
                check(tag + "disp", out[b], disp)


@pytest.mark.gpu
@pytest.mark.parametrize("wide", [0, 2], ids=["auto", "u16"])
@pytest.mark.parametrize("case", cases.BM_CASES, ids=[c[0] for c in cases.BM_CASES])
def test_bm_on_hard_inputs(oracle, case, wide):
    """D. StereoBM prefilter and map of every family in one batch, with the case's parameters and with textureThreshold
    0 (flat windows reach the sub-pixel guard) at uniquenessRatio 0 and 10; then the left-right check and the speckle
    filter (k_bm_lrcheck) against the reference."""
    from mvstereovision3_b200 import api
    name, p, H, W = case
    if wide and p["blockSize"] * 2 * p["preFilterCap"] > 255:
        pytest.skip("the volume is 16 bits wide anyway")
    fams = bm_families(p)
    B = len(fams)
    frames = [frame(f, H, W, 0, p["numDisp"], seed=i) for i, f in enumerate(fams)]
    L, R = np.stack([a for a, _ in frames]), np.stack([b for _, b in frames])
    with api.Engine(W, H, max_batch=B) as e:
        for v in (p, dict(p, textureThreshold=0, uniquenessRatio=0), dict(p, textureThreshold=0, uniquenessRatio=10)):
            e.set_bm_params(**v)
            e.debug_set_flags(wide)
            e.compute(L, R, api.STAGE_BM)
            out = e.download(B)["disp"]
            preL, preR = e.debug_read(5, B), e.debug_read(6, B)
            for b, f in enumerate(fams):
                disp, pl, pr = oracle.bm(frames[b][0], frames[b][1], v, want_prefilter=True)
                tag = "%s/%s/tex %d/u %d/" % (name, f, v["textureThreshold"], v["uniquenessRatio"])
                check(tag + "preL", preL[b], pl)
                check(tag + "preR", preR[b], pr)
                check(tag + "disp", out[b], disp)
        filters = [(dict(p, textureThreshold=0, uniquenessRatio=10), dict(disp12MaxDiff=0)),
                   (p, dict(disp12MaxDiff=1, speckleWindowSize=50, speckleRange=16)),
                   (dict(p, textureThreshold=0, uniquenessRatio=0), dict(disp12MaxDiff=1))]
        for v, f in filters[:1 if p["blockSize"] > 63 else 3]:
            e.set_bm_params(**v)
            e.set_bm_filters(**f)
            e.compute(L, R, api.STAGE_BM)
            out = e.download(B)["disp"]
            # the map after the check is an intermediate (debug_read 2) only when the speckle filter follows it;
            # without the filter it is the final map
            lr = e.debug_read(2, B) if f.get("speckleWindowSize", 0) > 0 else out
            for b, fam in enumerate(fams):
                tag = "%s/%s/%s/%s/" % (name, fam, v, f)
                check(tag + "lr", lr[b], ref.bm(oracle, frames[b][0], frames[b][1], dict(v, disp12MaxDiff=f["disp12MaxDiff"])))
                check(tag + "final", out[b], ref.bm(oracle, frames[b][0], frames[b][1], dict(v, **f)))
        e.set_bm_filters()


@pytest.mark.gpu
@settings(max_examples=30, deadline=None, suppress_health_check=list(HealthCheck))
@given(sgbm_case(max_d=128), st.sampled_from(FAMILIES))
def test_cuda_sgbm_vs_oracle_random_hard(oracle, case, fam):
    """E. Random in-contract SGBM parameters and shapes (tests/test_property.py), with the image family drawn too."""
    from mvstereovision3_b200 import api
    p, H, W, seed, _ = case
    l, r = frame(fam, H, W, p["minDisp"], p["numDisp"], seed=seed)
    want = oracle.sgbm(l, r, p)
    for flags in (0, 0xfe << 8):
        with api.Engine(W, H) as e:
            e.set_sgbm_params(**gpu_params(p))
            e.debug_set_flags(flags)
            e.compute(l, r, api.STAGE_SGBM)
            got = e.download(1)["disp"][0]
        assert np.array_equal(got, want), (fam, p, H, W, seed, hex(flags), int((got != want).sum()))


@pytest.mark.gpu
@settings(max_examples=40, deadline=None, suppress_health_check=list(HealthCheck))
@given(bm_case(), st.sampled_from(FAMILIES), st.sampled_from(FAMILIES))
def test_cuda_bm_vs_oracle_random_hard(oracle, case, fam0, fam1):
    from mvstereovision3_b200 import api
    nd, bs, cap, uniq, tex, H, W, seed, flags = case
    pairs = [frame(fam0, H, W, 0, nd, seed=seed), frame(fam1, H, W, 0, nd, seed=seed + 1)]
    p = dict(numDisp=nd, blockSize=bs, preFilterCap=cap, textureThreshold=tex, uniquenessRatio=uniq)
    with api.Engine(W, H, max_batch=2) as e:
        e.set_bm_params(**p)
        e.debug_set_flags(flags)
        e.compute(np.stack([pairs[0][0], pairs[1][0]]), np.stack([pairs[0][1], pairs[1][1]]), api.STAGE_BM)
        got = e.download(2)["disp"]
    for b, fam in enumerate((fam0, fam1)):
        want = oracle.bm(pairs[b][0], pairs[b][1], p)
        assert np.array_equal(got[b], want), (fam, p, H, W, seed, flags, int((got[b] != want).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("p,B", [(CFG2, 148), (CFG2_SHIPPED, 74)], ids=["cfg2_b148", "sgbm_yml_d128_b74"])
def test_full_size_scene_batch_vs_cv2(p, B):
    """F. The bench batches at full size on scene frames of four seeds repeated through the batch: every copy equals
    its twin, one copy of each equals cv2."""
    from mvstereovision3_b200 import api
    cv2 = pytest.importorskip("cv2")
    H, W = 480, 752
    gen = [hi.scene(H, W, p["minDisp"], p["numDisp"], seed=s) for s in range(4)]
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**gpu_params(p))
        e.compute(np.stack([gen[b % 4][0] for b in range(B)]), np.stack([gen[b % 4][1] for b in range(B)]), api.STAGE_SGBM)
        d = e.download(B)["disp"]
    for b in range(4, B):
        assert np.array_equal(d[b], d[b % 4]), "frame %d differs from its twin in %d pixels" % (b, int((d[b] != d[b % 4]).sum()))
    for s in range(4):
        check("scene %d vs cv2" % s, d[s], _cv_sgbm(cv2, gen[s][0], gen[s][1], p))


@pytest.mark.gpu
def test_1080p_hh_d256_scene_vs_cv2():
    from mvstereovision3_b200 import api
    cv2 = pytest.importorskip("cv2")
    l, r = hi.scene(1080, 1920, 0, 256, seed=3)
    with api.Engine(1920, 1080) as e:
        e.set_sgbm_params(**gpu_params(CFG4))
        e.compute(l, r, api.STAGE_SGBM)
        check("1080p hh d256 scene", e.download(1)["disp"][0], _cv_sgbm(cv2, l, r, CFG4))


@pytest.mark.gpu
def test_bm_yml_scene_batch_vs_cv2():
    from mvstereovision3_b200 import api
    cv2 = pytest.importorskip("cv2")
    p = dict(numDisp=80, blockSize=21, preFilterCap=2, uniquenessRatio=0, textureThreshold=30)     # configs/bm.yml
    frames = [hi.scene(480, 752, 0, 80, seed=20 + b) for b in range(7)]
    with api.Engine(752, 480, max_batch=7) as e:
        e.set_bm_params(**p)
        e.compute(np.stack([a for a, _ in frames]), np.stack([b for _, b in frames]), api.STAGE_BM)
        out = e.download(7)["disp"]
    for b, (l, r) in enumerate(frames):
        check("bm.yml scene %d" % b, out[b], cv_bm(cv2, l, r, p))


@pytest.mark.gpu
@pytest.mark.parametrize("fpc", [1, 2, 3])
@pytest.mark.parametrize("name", ["sgbm_yml_d64", "hh_cfg4_style", "d128_shipped"])
def test_flat_and_stripe_frames_between_textured_ones(oracle, name, fpc):
    """G. A flat frame and a stripe frame between textured frames, `fpc` frames per chunk of the cost kernel and the
    first row scan (flag bits 16..23), byte and 16-bit form of S: every frame equals its single-frame result and the
    oracle."""
    from mvstereovision3_b200 import api
    _, p, H, W = next(c for c in cases.SGBM_CASES if c[0] == name)
    kinds = ["exact_shift", "flat_levels", "scene", "stripes", "exact_shift", "zeros", "quantised"]
    frames = [frame(k, H, W, p["minDisp"], p["numDisp"], seed=b) for b, k in enumerate(kinds)]
    B = len(frames)
    L, R = np.stack([a for a, _ in frames]), np.stack([b for _, b in frames])
    for flags in (1, 3):
        with api.Engine(W, H, max_batch=B) as e:
            e.set_sgbm_params(**gpu_params(p))
            e.debug_set_flags(flags | (0xfe << 8) | (fpc << 16))
            e.compute(L, R, api.STAGE_SGBM)
            out, Sg = e.download(B)["disp"], e.debug_read(1, B)
            single = []
            for a, b in frames:
                e.compute(a, b, api.STAGE_SGBM)
                single.append(e.download(1)["disp"][0])
        for b, k in enumerate(kinds):
            disp, _, Sv, _ = oracle.sgbm(frames[b][0], frames[b][1], p, want_volumes=True)
            tag = "%s/%d/%s/%d" % (name, flags, k, b)
            check(tag + "/S", Sg[b], Sv)
            check(tag + "/disp", out[b], disp)
            check(tag + "/single", single[b], out[b])
