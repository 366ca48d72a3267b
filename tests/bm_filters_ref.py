"""Reference for StereoBM's post-filters (SURVEY.md A.4): the left-right check (disp12MaxDiff) and the speckle filter,
on top of the C oracle's StereoBM.  Test infrastructure, pinned against cv2 4.13.0 by tests/test_bm_filters.py.

cv::StereoBM matches every column of its width1 domain, X in [D - 1, W), with windows clamped to the image, and runs
the check before it clears the columns outside the valid rectangle; the border pixels therefore take part in the
check's scatter.  The oracle's orc_bm evaluates the valid rectangle only, so this module re-evaluates the whole domain
with numpy from the oracle's prefiltered images (the same clamps as orc_bm), asserts that the valid rectangle equals
orc_bm's map, and keeps the winner's SAD as the check's cost."""
import numpy as np

FILT = -16


def _box(a, bs):
    """Sums of bs x bs windows of a (rows r..r+bs-1, columns c..c+bs-1) for every full window."""
    c = np.pad(a.astype(np.int64), ((1, 0), (1, 0))).cumsum(0).cumsum(1)
    return c[bs:, bs:] - c[:-bs, bs:] - c[bs:, :-bs] + c[:-bs, :-bs]


def match_domain(pl, pr, p):
    """Disparity and winner SAD of every pixel of the width1 domain (rows [w2, H - w2), columns [D - 1, W)); FILT and 0
    elsewhere and where the texture or uniqueness test rejects."""
    H, W = pl.shape
    D, bs, cap = p["numDisp"], p["blockSize"], p["preFilterCap"]
    w2, lofs, width1 = bs // 2, D - 1, W - D + 1
    disp = np.full((H, W), FILT, np.int64)
    cost = np.zeros((H, W), np.int64)
    if width1 < 1 or H - 2 * w2 <= 0:
        return disp, cost
    j = np.arange(-w2, width1 + w2)                       # window columns in the width1 domain
    cl = np.clip(j, -lofs, W - lofs - 1) + lofs
    cr = np.clip(j, 0, W - D)
    L, R = pl.astype(np.int64), pr.astype(np.int64)
    tex = _box(np.abs(L[:, cl] - cap), bs)
    sad = np.stack([_box(np.abs(L[:, cl] - R[:, cr + k]), bs) for k in range(D)])
    mind = sad.argmin(0)                                  # first minimum
    minsad = np.take_along_axis(sad, mind[None], 0)[0]
    reject = tex < p["textureThreshold"]
    if p["uniquenessRatio"] > 0:
        thresh = minsad + minsad * p["uniquenessRatio"] // 100
        far = np.abs(np.arange(D)[:, None, None] - mind[None]) > 1
        reject |= (far & (sad <= thresh[None])).any(0)
    pk = np.take_along_axis(sad, np.where(mind + 1 < D, mind + 1, D - 2)[None], 0)[0]
    nk = np.take_along_axis(sad, np.where(mind > 0, mind - 1, 1)[None], 0)[0]
    den = pk + nk - 2 * minsad + np.abs(pk - nk)
    num = (pk - nk) * 256
    frac = np.where(den != 0, np.sign(num) * (np.abs(num) // np.maximum(den, 1)), 0)      # C division
    d = ((D - 1 - mind) * 256 + frac + 15) >> 4
    disp[w2:H - w2, lofs:] = np.where(reject, FILT, d)
    cost[w2:H - w2, lofs:] = np.where(reject, 0, minsad)
    return disp, cost


def lr_check(disp, cost, D, d12):
    """cv::validateDisparity per row: scatter x in [D, W) ascending, first strict minimum of the cost per x2, then
    every pixel whose disp2 at both integer neighbours differs by more than 16 * d12 becomes FILT."""
    H, W = disp.shape
    out = disp.copy()
    none = np.iinfo(np.int64).max
    table = np.full((H, W), none, np.int64)
    ys, xs = np.nonzero(disp[:, D:] != FILT)
    xs = xs + D
    d = disp[ys, xs]
    np.minimum.at(table, (ys, xs - ((d + 8) >> 4)), cost[ys, xs] * 4096 + xs)
    bad = np.ones(len(xs), bool)
    for xi in (xs - (d >> 4), xs - ((d + 15) >> 4)):
        inside = (xi >= 0) & (xi < W)
        key = np.where(inside, table[ys, np.clip(xi, 0, W - 1)], none)
        found = key != none
        d2 = disp[ys, np.where(found, key % 4096, 0)]
        bad &= found & (np.abs(d2 - d) > 16 * d12)
    out[ys[bad], xs[bad]] = FILT
    return out


def bm(oracle, left, right, p):
    """cv::StereoBM::compute with p's disp12MaxDiff / speckleWindowSize / speckleRange (defaults -1 / 0 / 0)."""
    d12, win, rng = p.get("disp12MaxDiff", -1), p.get("speckleWindowSize", 0), p.get("speckleRange", 0)
    if win < 0 or (win > 0 and rng < 0):
        raise ValueError("speckleWindowSize < 0, or speckleRange < 0 with a window")
    base = dict(numDisp=64, blockSize=21, preFilterCap=31, textureThreshold=10, uniquenessRatio=15)   # oracle.bm's
    base.update((k, v) for k, v in p.items() if k not in ("disp12MaxDiff", "speckleWindowSize", "speckleRange"))
    plain, pl, pr = oracle.bm(left, right, base, want_prefilter=True)
    out = plain.astype(np.int64)
    if d12 >= 0:
        H, W = plain.shape
        w2, D = base["blockSize"] // 2, base["numDisp"]
        disp, cost = match_domain(pl, pr, base)
        valid = np.zeros((H, W), bool)
        valid[w2:H - w2, D - 1 + w2:W - w2] = True
        assert np.array_equal(np.where(valid, disp, FILT), out), "the domain re-evaluation differs from orc_bm"
        out = np.where(valid, lr_check(disp, cost, D, d12), FILT)
    out = out.astype(np.int16)
    if win > 0:
        out = oracle.speckle(out, FILT, win, rng)
    return out
