"""The disparity post-filters and consumers of csrc/filters.cu on crafted maps: the 3x3 median (k_median3_w4,
k_median3), the speckle filter (k_ccl_rows, k_ccl_vmerge, k_ccl_flatten, k_ccl_apply), the reprojection (k_xyz), the
ROI means (k_means) and the min / max reduction (k_minmax).

The GPU runs them on caller-supplied maps through the test hook mvsv_debug_postfilter (Engine.debug_postfilter), so
that the maps can hold what a matcher rarely produces: values at the int16 limits, components of exactly maxSpeckleSize
pixels, runs across the warp chunks of the row scan, sums past 2^31.  The references are exact and live in this file:
cv2.medianBlur and cv2.filterSpeckles, a numpy transcription of k_xyz / orc_reproject, and integer ROI means and
min / max.  The CPU part checks every reference against the C oracle (and the XYZ transcription against
cv2.reprojectImageTo3D); the GPU part compares the kernels with the references bit for bit."""
import functools
import json
import os

import numpy as np
import pytest
from scipy import ndimage, sparse
from scipy.sparse import csgraph

import cases
from mvstereovision3_b200 import api

cv2 = pytest.importorskip("cv2")

NEWVALS = (-16, 0, -64)
FAR = (20000, 26000)          # background: a checkerboard of these connects to nothing below a range of 6000


# ------------------------------------------------------------------------------------------------ references
def ref_median(m):
    """medianBlur(CV_16S, 3), replicate border, frame by frame."""
    return np.stack([cv2.medianBlur(np.ascontiguousarray(f), 3) for f in m.reshape((-1,) + m.shape[-2:])]).reshape(m.shape)


def ref_speckle(m, new_val, max_size, max_diff):
    out = [cv2.filterSpeckles(np.ascontiguousarray(f).copy(), new_val, max_size, max_diff)[0]
           for f in m.reshape((-1,) + m.shape[-2:])]
    return np.stack(out).reshape(m.shape)


def ref_xyz(disp, Q):
    """k_xyz / orc_reproject in numpy: Q[r] . (x, y, d, 1) accumulated left to right in float64 (the products of two
    floats are exact there), rounded to float32, divided in float32; Z = 0 where Z / 1000 is infinite; (0, 0, 0) where
    d <= 0.  disp [B, H, W] int16 -> [B, H, W, 3] float32."""
    q = np.asarray(Q, np.float32).astype(np.float64).reshape(4, 4)
    _, H, W = disp.shape
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    d = (disp.astype(np.float32) / np.float32(16)).astype(np.float64)
    cc = [(((q[r, 0] * x) + q[r, 1] * y) + q[r, 2] * d + q[r, 3]).astype(np.float32) for r in range(4)]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        X, Y, Z = cc[0] / cc[3], cc[1] / cc[3], cc[2] / cc[3]
        Z = np.where(np.isinf(Z / np.float32(1000)), np.float32(0), Z)
    out = np.stack([X, Y, Z], -1)
    out[disp <= 0] = 0
    return out


def ref_means(disp, rois):
    """Utility::calcMeanDisparity: pixels with v > 1 are summed in an int (wrapping past 2^31) and counted; the mean is
    the C (truncating) quotient, 0 when the sum or the count is 0.  disp [B, H, W] -> [B, nrois] float32."""
    B = disp.shape[0]
    v = disp.astype(np.int64)
    sel = v > 1
    sat_v = np.zeros((B, disp.shape[1] + 1, disp.shape[2] + 1), np.int64)
    sat_n = np.zeros_like(sat_v)
    sat_v[:, 1:, 1:] = np.where(sel, v, 0).cumsum(1).cumsum(2)
    sat_n[:, 1:, 1:] = sel.cumsum(1).cumsum(2)
    r = np.asarray(rois, np.int64).reshape(-1, 4)
    x0, y0, x1, y1 = r[:, 0], r[:, 1], r[:, 0] + r[:, 2], r[:, 1] + r[:, 3]
    box = lambda s: s[:, y1, x1] - s[:, y0, x1] - s[:, y1, x0] + s[:, y0, x0]
    total, n = box(sat_v), box(sat_n)
    total = (total + 2 ** 31) % 2 ** 32 - 2 ** 31
    q = np.abs(total) // np.maximum(n, 1) * np.sign(total)
    return np.where((total == 0) | (n == 0), 0, q).astype(np.float32)


def ref_minmax(disp):
    out = np.zeros((disp.shape[0], 2), np.int16)
    for b, f in enumerate(disp):
        p = f[f > 0]
        if p.size:
            out[b] = p.min(), p.max()
    return out


# ------------------------------------------------------------------------------------------------ map helpers
def components(m, new_val, max_diff):
    """Per pixel, the size of its 4-connected speckle component (|difference| <= max_diff, new_val pixels belong to
    none: 0 there)."""
    H, W = m.shape
    v = m.astype(np.int64)
    ok = m != new_val
    idx = np.arange(H * W).reshape(H, W)
    eh = ok[:, 1:] & ok[:, :-1] & (np.abs(v[:, 1:] - v[:, :-1]) <= max_diff)
    ev = ok[1:] & ok[:-1] & (np.abs(v[1:] - v[:-1]) <= max_diff)
    a = np.concatenate([idx[:, :-1][eh], idx[:-1][ev]])
    b = np.concatenate([idx[:, 1:][eh], idx[1:][ev]])
    g = sparse.coo_matrix((np.ones(len(a)), (a, b)), shape=(H * W, H * W))
    _, lab = csgraph.connected_components(g, directed=False)
    return np.where(ok, np.bincount(lab)[lab].reshape(H, W), 0)


def steps(m, new_val):
    """The set of |differences| between 4-neighbours that are both not new_val."""
    v = m.astype(np.int64)
    ok = m != new_val
    h = np.abs(v[:, 1:] - v[:, :-1])[ok[:, 1:] & ok[:, :-1]]
    w = np.abs(v[1:] - v[:-1])[ok[1:] & ok[:-1]]
    return set(np.unique(np.concatenate([h, w])).tolist())


def background(H, W):
    """Pixels that connect to nothing (a checkerboard of two far-apart values)."""
    return np.where((np.arange(H)[:, None] + np.arange(W)) % 2 == 0, FAR[0], FAR[1]).astype(np.int16)


def tri(t, n):
    """Triangle wave 0, 1, .., n-1, n-1, .., 0, 0, 1, ..: consecutive values differ by 0 or 1."""
    t = np.asarray(t) % (2 * n)
    return np.where(t < n, t, 2 * n - 1 - t)


# ------------------------------------------------------------------------------------------------ speckle maps
# Each generator returns (map [H, W] or [B, H, W], maxSpeckleSize, maxDiff) and asserts that the map hits its target.
def sp_serpentine(new_val, H=70, W=300, max_diff=16, over=0):
    """A 1-pixel-wide path: full rows at even y, joined by one pixel at alternating ends; it crosses every 16-row CCL
    strip and every 128-column CTA.  Its values climb and fall in steps of exactly maxDiff.  maxSize = its size - over:
    over 0 removes it, over 1 keeps it."""
    m = background(H, W)
    path = []
    for y in range(H):
        if y % 2 == 0:
            xs = range(W) if (y // 2) % 2 == 0 else range(W - 1, -1, -1)
            path += [(y, x) for x in xs]
        else:
            path.append((y, W - 1 if (y // 2) % 2 == 0 else 0))
    ys, xs = np.array(path).T
    m[ys, xs] = 1000 + max_diff * tri(np.arange(len(path)) // 5, 20)
    size = len(path)
    comp = components(m, new_val, max_diff)
    assert comp[0, 0] == size, "this case is meant to be one component"
    assert set(ys // 16) == set(range((H + 15) // 16)) and set(xs // 128) == set(range((W + 127) // 128))
    assert max_diff in steps(m, new_val), "the path is meant to step by maxDiff"
    return m, size - over, max_diff


def sp_comb(new_val, H=50, W=261, max_diff=16, over=0):
    """Teeth at even x from row 0 to H-2, joined only by the last row: each tooth is its own run set until the
    last row merges them all."""
    m = background(H, W)
    v = (600 + max_diff * ((np.arange(H) // 3) % 2)).astype(np.int16)
    m[:H - 1, 0::2] = v[:H - 1, None]
    m[H - 1, :] = v[H - 2]
    size = len(range(0, W, 2)) * (H - 1) + W
    comp = components(m, new_val, max_diff)
    assert comp[0, 0] == size and comp[0, W - 1] == size, "the teeth are meant to join in the last row"
    assert components(m[:H - 1], new_val, max_diff)[0, 0] == H - 1, "and only there"
    return m, size - over, max_diff


def sp_checker(new_val, H=33, W=130, max_size=1):
    """Every other pixel is new_val: equal values that touch only diagonally, all components of size 1."""
    m = np.where((np.arange(H)[:, None] + np.arange(W)) % 2 == 0, 5, new_val).astype(np.int16)
    comp = components(m, new_val, 16)
    assert comp.max() == 1 and (m == new_val).sum() == (H * W) // 2
    return m, max_size, 16


RUN_LENGTHS, RUN_STARTS = (31, 32, 33, 65), (0, 31, 64, 95)


def sp_runs(new_val, W=200, max_size=32):
    """Row runs of 31, 32, 33 and 65 pixels starting at x % 32 == 0 and 31 (the carry of k_ccl_rows), one per row,
    between rows of isolated pixels; maxSize 32 removes the first two lengths and keeps the others."""
    rows = [(L, s) for L in RUN_LENGTHS for s in RUN_STARTS]
    H = 2 * len(rows) + 1
    m = background(H, W)
    for k, (L, s) in enumerate(rows):
        m[2 * k + 1, s:s + L] = 700 + 3 * (np.arange(L) % 2)       # steps of 3 inside the run
    comp = components(m, new_val, 16)
    for k, (L, s) in enumerate(rows):
        assert comp[2 * k + 1, s] == L and comp[2 * k + 1, s + L - 1] == L
    assert {s % 32 for _, s in rows} == {0, 31} and {max_size, max_size + 1} <= set(np.unique(comp).tolist())
    return m, max_size, 16


def shape_pixels(n, form):
    """n pixel offsets (y, x) of a connected shape: a horizontal or vertical line, a 7-wide block, a U whose arms
    meet only in the bottom row, an L."""
    if form == "hline":
        return [(0, i) for i in range(n)]
    if form == "vline":
        return [(i, 0) for i in range(n)]
    if form == "block":
        return [(i // 7, i % 7) for i in range(n)]
    if form == "U":
        h = (n - 7) // 2
        px = [(y, 0) for y in range(h)] + [(y, 6) for y in range(h)] + [(h, x) for x in range(7)]
        return px + [(h + 1, 3)] * (n - len(px))
    if form == "L":
        h = n // 2
        return [(y, 0) for y in range(h)] + [(h - 1, x) for x in range(1, n - h + 1)]
    raise ValueError(form)


def sp_sizes(new_val, max_size=20, max_diff=16):
    """Components of exactly maxSize and maxSize + 1 pixels in five shapes, placed across the 16-row strips and the
    128-column CTAs; the values inside each shape step by maxDiff."""
    forms = ("hline", "vline", "block", "U", "L")
    shapes = [shape_pixels(n, f) for f in forms for n in (max_size, max_size + 1)]
    H, W = max_size + 12, 2000
    m = background(H, W)
    x, expect = 5, []
    for k, px in enumerate(shapes):
        ys, xs = np.array(px).T
        m[3 + ys, x + xs] = 1000 + 100 * k + max_diff * ((ys + xs) % 2)
        expect.append((3 + ys[0], x + xs[0], len(set(px))))
        x += xs.max() + 3
    assert x < W
    comp = components(m, new_val, max_diff)
    for y, xx, n in expect:
        assert comp[y, xx] == n
    sizes = set(np.unique(comp).tolist())
    assert {max_size, max_size + 1} <= sizes, "this case is meant to hold components of maxSize and maxSize + 1"
    return m, max_size, max_diff


def sp_steps(new_val, max_diff, seed=0, H=60, W=210):
    """2 x 3 blocks whose neighbours differ by exactly maxDiff (joined) or maxDiff + 1 (apart), horizontally and
    vertically."""
    rng = np.random.default_rng(seed)
    s = rng.choice([max_diff, max_diff + 1], W // 3) * rng.choice([-1, 1], W // 3)
    t = rng.choice([max_diff, max_diff + 1], H // 2) * rng.choice([-1, 1], H // 2)
    a, b = np.cumsum(s), np.cumsum(t)
    m = (2000 + b[:, None] + a[None, :]).repeat(2, 0).repeat(3, 1).astype(np.int16)
    st = steps(m, new_val)
    assert {max_diff, max_diff + 1} <= st, "this case is meant to hold steps of maxDiff and maxDiff + 1"
    sizes = components(m, new_val, max_diff)
    max_size = int(np.median(sizes))
    assert sizes.min() <= max_size < sizes.max()
    return m, max_size, max_diff


def sp_newval_inside(new_val, seed=1, H=64, W=257):
    """Blobs whose values lie next to new_val, with new_val pixels scattered inside them: they split components and
    must not connect anything although |new_val - v| <= maxDiff."""
    rng = np.random.default_rng(seed)
    m = background(H, W)
    for _ in range(60):
        h, w = rng.integers(2, 20, 2)
        y, x = rng.integers(0, H - h), rng.integers(0, W - w)
        m[y:y + h, x:x + w] = new_val + rng.choice([-8, -4, 4, 8])
    holes = rng.random((H, W)) < 0.08
    m[holes] = new_val
    inner = holes[1:-1, 1:-1] & (m[1:-1, :-2] == m[1:-1, 2:]) & (m[1:-1, :-2] != new_val) & (m[1:-1, :-2] < FAR[0])
    assert inner.sum() > 20, "this case is meant to put new_val pixels inside components"
    return m, 12, 8


def sp_tiny(new_val, H, W, seed=2):
    rng = np.random.default_rng(seed)
    m = (rng.integers(0, 4, (H, W)) * 16 + 300).astype(np.int16)
    m[rng.random((H, W)) < 0.1] = new_val
    assert m.shape == (H, W)
    return m, 3, 16


def sp_diagonal(new_val, H=40, W=140):
    """2 x 2 motifs [[100, 116], [132, 124]] at maxDiff 16: the rows are linked at the right column only, while the
    left column's pixels are each linked to their own row (the case the 'left neighbours already link the rows' skip
    of k_ccl_vmerge must not take)."""
    m = background(H, W)
    for y in range(1, H - 2, 3):
        for x in range(1, W - 2, 3):
            m[y:y + 2, x:x + 2] = [[100, 116], [132, 124]]
    assert components(m, new_val, 16)[1, 1] == 4
    return m, 3, 16


def sp_wave(new_val, H=90, W=300):
    """A smooth surface whose neighbour differences range around maxDiff."""
    y, x = np.mgrid[0:H, 0:W]
    m = (2000 + 40 * np.sin(x / 5.3) + 40 * np.cos(y / 4.1) + 25 * np.sin((x + y) / 3.7)).astype(np.int16)
    st = steps(m, new_val)
    assert min(st) < 16 < max(st)
    return m, 40, 16


def speckle_cases():
    """(id, newVal, generator) of the crafted speckle maps; the generator is called lazily."""
    out = []
    for nv in NEWVALS:
        g = [("serpentine_kill", lambda nv=nv: sp_serpentine(nv, over=0)),
             ("serpentine_keep", lambda nv=nv: sp_serpentine(nv, over=1)),
             ("comb_kill", lambda nv=nv: sp_comb(nv, over=0)),
             ("comb_keep", lambda nv=nv: sp_comb(nv, over=1)),
             ("checker_kill", lambda nv=nv: sp_checker(nv, max_size=1)),
             ("checker_keep", lambda nv=nv: sp_checker(nv, max_size=0)),
             ("runs", lambda nv=nv: sp_runs(nv)),
             ("sizes20", lambda nv=nv: sp_sizes(nv, 20)),
             ("sizes150", lambda nv=nv: sp_sizes(nv, 150, 32)),
             ("newval_inside", lambda nv=nv: sp_newval_inside(nv)),
             ("h1", lambda nv=nv: sp_tiny(nv, 1, 300)),
             ("w2", lambda nv=nv: sp_tiny(nv, 100, 2)),
             ("h1w2", lambda nv=nv: sp_tiny(nv, 1, 2)),
             ("diagonal", lambda nv=nv: sp_diagonal(nv)),
             ("wave", lambda nv=nv: sp_wave(nv))]
        g += [("steps%d" % md, lambda nv=nv, md=md: sp_steps(nv, md)) for md in (0, 1, 16, 32)]
        out += [("%s_nv%d" % (name, nv), nv, gen) for name, gen in g]
    return out


SPECKLE_CASES = speckle_cases()


def sp_batch_boundary(new_val, B=3, H=20, W=150):
    """Frames whose last row equals the next frame's first row: a run of W pixels on each side of every frame
    boundary.  In one frame each run is one component of W pixels (removed with maxSize W + 5); joined across a
    boundary it would be kept."""
    m = np.stack([background(H, W) for _ in range(B)])
    for b in range(B):
        m[b, 0, :] = 900
        m[b, H - 1, :] = 900
    for b in range(B - 1):
        assert np.array_equal(m[b, -1], m[b + 1, 0])
    assert components(m.reshape(B * H, W), new_val, 16)[H - 1, 0] == 2 * W, "the rows are meant to join if stacked"
    return m, W + 5, 16


def blob_maps(B, H, W, new_val, vmax, seed):
    """Piecewise-constant blobs of many sizes (some with a gentle slope), over per-pixel noise, with new_val holes;
    values in [16, vmax] like a matcher's x16 disparities."""
    rng = np.random.default_rng(seed)
    m = rng.integers(16, vmax + 1, (B, H, W)).astype(np.int16)
    nb = H * W // 300
    for b in range(B):
        f = m[b]
        hs = np.minimum((2 ** rng.uniform(0, 7, (nb, 2))).astype(int), (H, W))
        ys = rng.integers(0, H - hs[:, 0] + 1)
        xs = rng.integers(0, W - hs[:, 1] + 1)
        vals = rng.integers(16, vmax + 1, nb)
        slope = rng.integers(0, 2, nb)
        for (h, w), y, x, v, s in zip(hs, ys, xs, vals, slope):
            if s:
                f[y:y + h, x:x + w] = np.minimum(v + np.arange(w) // 3, vmax)
            else:
                f[y:y + h, x:x + w] = v
    m[rng.random((B, H, W)) < 0.02] = new_val
    return m


# cv::StereoSGBM's filter settings of cfg 2 (minDisparity 1 -> newVal 0, speckle 150 / range 2 x 16) and cv::StereoBM's
# of OpenCV's stereo_match sample (newVal -16, window 100, range 32 as given)
SGBM_SPECKLE = dict(new_val=0, max_size=150, max_diff=32, vmax=16 * 65)
BM_SPECKLE = dict(new_val=-16, max_size=100, max_diff=32, vmax=16 * 64)


@functools.lru_cache(maxsize=None)
def blob_case(kind, B, H, W):
    s = SGBM_SPECKLE if kind == "sgbm" else BM_SPECKLE
    m = blob_maps(B, H, W, s["new_val"], s["vmax"], seed=B + H + W)
    want = ref_speckle(ref_median(m) if kind == "sgbm" else m, s["new_val"], s["max_size"], s["max_diff"])
    removed = np.mean((want == s["new_val"]) & (m != s["new_val"]))
    assert 0.05 < removed < 0.95, "this case is meant to remove some components and keep others (%.3f)" % removed
    return m, want, s


# ------------------------------------------------------------------------------------------------ median maps
MED_W = (2, 3, 4, 5, 8) + tuple(range(16, 24)) + tuple(range(119, 126)) + tuple(range(239, 245))
MED_H = (1, 2, 15, 16, 17, 33)


def med_random(B, H, W, seed):
    """Full-range int16 with both limits present."""
    rng = np.random.default_rng(seed)
    m = rng.integers(-32768, 32768, (B, H, W)).astype(np.int16)
    m.reshape(-1)[rng.integers(0, m.size, max(2, m.size // 8))] = rng.choice([-32768, 32767], max(2, m.size // 8))
    m.reshape(-1)[:2] = (-32768, 32767)
    assert m.min() == -32768 and m.max() == 32767
    return m


def med_values(kind, B, H, W, seed=3):
    rng = np.random.default_rng(seed)
    if kind == "fullrange":
        return med_random(B, H, W, seed)
    if kind == "around0":
        # alternating signs: a sign-extension or packed-compare error inverts medians
        m = rng.integers(1, 4, (B, H, W)) * np.where((np.arange(H)[:, None] + np.arange(W)) % 2 == 0, 1, -1)
        m[:, ::5] *= -1
        m = m.astype(np.int16)
        assert (m < 0).any() and (m > 0).any()
        return m
    if kind == "border":
        # constant except the last column and the last row: only the replicate border makes them the median there
        m = np.full((B, H, W), 7, np.int16)
        m[:, :, W - 1] = -30000
        m[:, H - 1, :] = 30000
        assert (ref_median(m)[:, :, W - 1] != 7).any()
        return m
    raise ValueError(kind)


# ------------------------------------------------------------------------------------------------ XYZ inputs
with open(os.path.join(cases.GOLDEN_DIR, "calibrations.json")) as _f:
    _RIG = json.load(_f)["rigs"]["baseline_small"]


def q_rectify(flags):
    r = _RIG
    out = cv2.stereoRectify(np.array(r["KL"]), np.array(r["DL"]), np.array(r["KR"]), np.array(r["DR"]), (752, 480),
                            np.array(r["R"]), np.array(r["T"]).reshape(3, 1), flags=flags, alpha=0)
    return out[4].astype(np.float32)


def q_matrices():
    qz, q0 = q_rectify(cv2.CALIB_ZERO_DISPARITY), q_rectify(0)
    assert qz[3, 3] == 0 and q0[3, 3] != 0
    qneg = cases.Q_REFERENCE.copy()
    qneg[3, 2] = -1.0 / 118.7                       # negative 1/Tx: every valid pixel has a negative divisor
    qzero = cases.Q_REFERENCE.copy()
    qzero[3, 2], qzero[3, 3] = 1.0 / 16, -1.0       # the divisor d/16 - 1 is exactly 0 at d = 16 (value 256)
    return {"reference": cases.Q_REFERENCE, "rectify_zero_disparity": qz, "rectify": q0, "neg_tx": qneg, "zero_div": qzero}


XYZ_SPECIAL = (-32768, -16, 0, 1, 16, 255, 256, 257, 32767)
# (W, H, B): W % 4 = 0..3, B * H * W % 4 != 0; 5 x 3 x 3 has a 4-pixel group across a row end and a frame end (pixels
# 12..15) and a one-pixel tail (pixel 44)
XYZ_SHAPES = ((8, 4, 3), (5, 3, 3), (10, 3, 3), (7, 5, 3), (11, 1, 3), (13, 7, 5), (752, 480, 2))


def xyz_map(W, H, B, seed=4):
    rng = np.random.default_rng(seed)
    m = rng.integers(-32768, 32768, (B, H, W)).astype(np.int16)
    pick = rng.random((B, H, W)) < 0.5
    m[pick] = rng.choice(XYZ_SPECIAL, int(pick.sum()))
    m.reshape(-1)[:len(XYZ_SPECIAL)] = XYZ_SPECIAL
    assert set(XYZ_SPECIAL) <= set(np.unique(m).tolist())
    return m


def assert_same_floats(got, want, what):
    """Bit for bit, with NaN (whatever its payload) in the same places."""
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), "%s: NaN at %d vs %d places" % (what, gn.sum(), wn.sum())
    g, w = got[~gn].view(np.uint32), want[~wn].view(np.uint32)
    bad = np.flatnonzero(g != w)
    assert bad.size == 0, "%s: %d differ, first %s vs %s" % (what, bad.size, got[~gn][bad[0]], want[~wn][bad[0]])


# ------------------------------------------------------------------------------------------------ ROI inputs
def roi_set(W, H, n, seed=5):
    """1 x 1, the full map, the last row and column, widths 1..17, then random ROIs up to n."""
    rng = np.random.default_rng(seed)
    r = [(0, 0, 1, 1), (W - 1, H - 1, 1, 1), (0, 0, W, H), (0, H - 1, W, 1), (W - 1, 0, 1, H)]
    r += [(W - w, int(rng.integers(0, H - 3)), w, 3) for w in range(1, 18)]
    while len(r) < n:
        w, h = int(rng.integers(1, min(W, 40) + 1)), int(rng.integers(1, min(H, 40) + 1))
        r.append((int(rng.integers(0, W - w + 1)), int(rng.integers(0, H - h + 1)), w, h))
    return r[:n]


def means_map(B, H, W, seed=6):
    """Values 1 and 2 (the v > 1 rule), negatives, and ordinary disparities."""
    rng = np.random.default_rng(seed)
    m = rng.choice([-16, -1, 0, 1, 2, 3, 17, 1024, 32767], (B, H, W)).astype(np.int16)
    assert {1, 2} <= set(np.unique(m).tolist()) and m.min() < 0
    return m


def cfg3_rois(W, H, num_disp):
    off = api.dmap_roi_offset(num_disp, W)
    return api.subimage_rois(W - off, H, off) + api.samplepoint_rois(W - off, H, off)


# ================================================================================================ CPU part
def test_median_reference_matches_oracle(oracle):
    for W in MED_W:
        for H in MED_H:
            m = med_random(1, H, W, seed=W * 100 + H)[0]
            want = ref_median(m)
            assert np.array_equal(want, oracle.median3(m)), (W, H)
            assert np.array_equal(want, ndimage.median_filter(m, 3, mode="nearest")), (W, H)
    for kind in ("fullrange", "around0", "border"):
        for H, W in ((33, 244), (17, 125), (2, 8), (1, 5)):
            m = med_values(kind, 1, H, W)[0]
            assert np.array_equal(ref_median(m), oracle.median3(m)), (kind, W, H)


@pytest.mark.parametrize("case", SPECKLE_CASES, ids=[c[0] for c in SPECKLE_CASES])
def test_speckle_reference_matches_oracle(oracle, case):
    _, nv, gen = case
    m, max_size, max_diff = gen()
    assert np.array_equal(ref_speckle(m, nv, max_size, max_diff), oracle.speckle(m, nv, max_size, max_diff))


@pytest.mark.parametrize("nv", NEWVALS)
def test_speckle_reference_batch_boundary(oracle, nv):
    m, max_size, max_diff = sp_batch_boundary(nv)
    want = ref_speckle(m, nv, max_size, max_diff)
    assert (want[:, 0] == nv).all() and (want[:, -1] == nv).all()
    for b in range(len(m)):
        assert np.array_equal(want[b], oracle.speckle(m[b], nv, max_size, max_diff))


@pytest.mark.parametrize("shape", [(148, 480, 752), (1, 1080, 1920)], ids=["cfg2", "1080p"])
@pytest.mark.parametrize("kind", ["sgbm", "bm"])
def test_speckle_reference_blobs(oracle, kind, shape):
    m, want, s = blob_case(kind, *shape)
    src = oracle_median(oracle, m) if kind == "sgbm" else m
    for b in range(len(m)):
        assert np.array_equal(want[b], oracle.speckle(src[b], s["new_val"], s["max_size"], s["max_diff"])), b


def oracle_median(oracle, m):
    return np.stack([oracle.median3(f) for f in m])


@pytest.mark.parametrize("qname", list(q_matrices()))
def test_xyz_reference_matches_oracle_and_cv2(oracle, qname):
    Q = q_matrices()[qname]
    for W, H, B in XYZ_SHAPES:
        m = xyz_map(W, H, B)
        want = ref_xyz(m, Q)
        for b in range(B):
            got, _ = oracle.reproject(m[b], Q)
            assert_same_floats(got, want[b], "%s %dx%d frame %d" % (qname, W, H, b))
            cv = cv2.reprojectImageTo3D(m[b].astype(np.float32) / 16, Q)
            ok = (m[b] > 0)[..., None] & np.isfinite(cv)
            np.testing.assert_allclose(want[b][ok], cv[ok], rtol=1e-5)
    if qname == "zero_div":
        w = ref_xyz(np.full((1, 1, 4), 256, np.int16), Q)
        assert np.isinf(w[..., 0]).all() and (w[..., 2] == 0).all(), "the divisor is meant to be 0 at d = 16"


def test_means_reference_matches_oracle(oracle):
    m = means_map(1, 120, 200)
    rois = roi_set(200, 120, 300)
    want = ref_means(m, rois)[0]
    for k, r in enumerate(rois):
        assert want[k] == oracle.mean(m[0], r), r
    for W, H, n, v, mean in ((752, 480, None, 32767, -2929.0), (512, 512, None, 16384, 0.0)):
        full = np.full((1, H, W), v, np.int16)
        assert int(full.astype(np.int64).sum()) >= 2 ** 31, "this case is meant to overflow the int sum"
        assert ref_means(full, [(0, 0, W, H)])[0, 0] == mean == oracle.mean(full[0], (0, 0, W, H))
    m = means_map(1, 480, 752)
    for W, H, nd, n in ((752, 480, 128, 5096), (752, 479, 64, 5243)):
        rois = cfg3_rois(W, H, nd)
        assert len(rois) == n
        want = ref_means(m[:, :H], rois)[0]
        assert all(want[k] == oracle.mean(m[0, :H], r) for k, r in enumerate(rois))


# ================================================================================================ GPU part
gpu = pytest.mark.gpu


def check(name, got, want):
    assert got.shape == want.shape, (name, got.shape, want.shape)
    if not np.array_equal(got, want):
        idx = np.argwhere(got != want)
        raise AssertionError("%s: %d mismatches, first at %s: got %s want %s" % (
            name, len(idx), tuple(idx[0]), got[tuple(idx[0])], want[tuple(idx[0])]))


def run_median(e, m, flags):
    e.debug_set_flags(flags)
    e.debug_postfilter(m, median=True)
    return e.download(len(m))["disp"]


@gpu
@pytest.mark.parametrize("W", MED_W)
def test_median_shapes(W):
    """Both median kernels (debug flag bit 2 forces the scalar one) at widths around the 30- and 120-column warp
    tiles and heights around the 16-row bands."""
    for H in MED_H:
        m = med_random(3, H, W, seed=W * 100 + H)
        want = ref_median(m)
        with api.Engine(W, H, max_batch=3) as e:
            for flags in (0, 4):
                check("W=%d H=%d flags=%d" % (W, H, flags), run_median(e, m, flags), want)


@gpu
def test_median_4k():
    m = med_random(1, 2160, 3840, seed=9)
    want = ref_median(m)
    with api.Engine(3840, 2160, max_batch=1) as e:
        for flags in (0, 4):
            check("4K flags=%d" % flags, run_median(e, m, flags), want)


@gpu
@pytest.mark.parametrize("kind", ["fullrange", "around0", "border"])
def test_median_values(kind):
    for H, W in ((33, 244), (17, 125), (16, 120), (2, 8), (1, 5), (15, 2)):
        m = med_values(kind, 3, H, W)
        with api.Engine(W, H, max_batch=3) as e:
            for flags in (0, 4):
                check("%s %dx%d flags=%d" % (kind, W, H, flags), run_median(e, m, flags), ref_median(m))


def run_speckle(m, nv, max_size, max_diff, median=False):
    m = m if m.ndim == 3 else m[None]
    B, H, W = m.shape
    with api.Engine(W, H, max_batch=B) as e:
        e.debug_postfilter(m, median=median, new_val=nv, speckle_size=max_size, speckle_diff=max_diff)
        check("raw", e.debug_read(2, B), m)
        return e.download(B)["disp"]


@gpu
@pytest.mark.parametrize("case", SPECKLE_CASES, ids=[c[0] for c in SPECKLE_CASES])
def test_speckle_crafted(case):
    _, nv, gen = case
    m, max_size, max_diff = gen()
    check("speckle", run_speckle(m, nv, max_size, max_diff)[0], ref_speckle(m, nv, max_size, max_diff))


@gpu
@pytest.mark.parametrize("nv", NEWVALS)
def test_speckle_batch_boundary(nv):
    """Nothing connects across the boundary of two frames of one batch."""
    m, max_size, max_diff = sp_batch_boundary(nv)
    check("batch", run_speckle(m, nv, max_size, max_diff), ref_speckle(m, nv, max_size, max_diff))


@gpu
@pytest.mark.parametrize("shape", [(148, 480, 752), (1, 1080, 1920)], ids=["cfg2", "1080p"])
@pytest.mark.parametrize("kind", ["sgbm", "bm"])
def test_speckle_blobs(kind, shape):
    """Random blob maps with cv::StereoSGBM's filters of cfg 2 (median, then speckle 150 / 2 x 16 with newVal 0) and
    cv::StereoBM's (speckle 100 / 32 with newVal -16)."""
    m, want, s = blob_case(kind, *shape)
    got = run_speckle(m, s["new_val"], s["max_size"], s["max_diff"], median=kind == "sgbm")
    check("%s %s" % (kind, shape), got, want)


@gpu
@pytest.mark.parametrize("shape", XYZ_SHAPES, ids=["%dx%dx%d" % s for s in XYZ_SHAPES])
@pytest.mark.parametrize("qname", list(q_matrices()))
def test_xyz(qname, shape):
    Q = q_matrices()[qname]
    W, H, B = shape
    m = xyz_map(W, H, B)
    with api.Engine(W, H, max_batch=B) as e:
        e.set_Q(Q)
        e.debug_postfilter(m, median=False, stages=api.STAGE_XYZ)
        got = e.download(B, xyz=True)["xyz"]
    assert_same_floats(got, ref_xyz(m, Q), "%s %s" % (qname, shape))


@gpu
@pytest.mark.parametrize("n", [1, 31, 32, 33, 300])
def test_means_roi_counts(n):
    """ROI counts around the 32 ROIs of a CTA; 1 x 1, full-map, last-row / last-column ROIs and widths 1..17 around the
    eight lanes of a ROI; values 1 and 2 and negatives."""
    B, H, W = 3, 120, 200
    m = means_map(B, H, W)
    rois = roi_set(W, H, n)
    with api.Engine(W, H, max_batch=B) as e:
        e.set_mean_rois(rois)
        e.debug_postfilter(m, median=False, stages=api.STAGE_MEANS)
        check("means n=%d" % n, e.download(B, disp=False, means=True)["means"], ref_means(m, rois))


@gpu
@pytest.mark.parametrize("geom", [(752, 480, 128, 5096), (752, 479, 64, 5243)], ids=["5096", "cfg3"])
def test_means_cfg3_rois(geom):
    W, H, nd, n = geom
    rois = cfg3_rois(W, H, nd)
    assert len(rois) == n
    m = means_map(4, H, W)
    with api.Engine(W, H, max_batch=4) as e:
        e.set_mean_rois(rois)
        e.debug_postfilter(m, median=False, stages=api.STAGE_MEANS)
        check("cfg3 means", e.download(4, disp=False, means=True)["means"], ref_means(m, rois))


@gpu
def test_means_wrapping_sums():
    """The reference's int sum wraps: 752 x 480 of 32767 gives -2929, 512 x 512 of 16384 wraps to exactly 0."""
    for W, H, v, mean in ((752, 480, 32767, -2929.0), (512, 512, 16384, 0.0)):
        m = np.full((2, H, W), v, np.int16)
        m[1, :, :W // 2] = -16            # half the map: a sum that does not wrap
        rois = [(0, 0, W, H), (0, 0, W, H // 2), (W // 2, 0, W - W // 2, H)]
        with api.Engine(W, H, max_batch=2) as e:
            e.set_mean_rois(rois)
            e.debug_postfilter(m, median=False, stages=api.STAGE_MEANS)
            got = e.download(2, disp=False, means=True)["means"]
        check("wrap %dx%d" % (W, H), got, ref_means(m, rois))
        assert got[0, 0] == mean


@gpu
def test_means_and_xyz_of_both_io_slots():
    """Two I/O slots: the results of the call before the last one stay readable with download(age=1)."""
    B, H, W = 2, 64, 96
    a, b = means_map(B, H, W, seed=7), xyz_map(W, H, B, seed=8)
    rois = roi_set(W, H, 40)
    with api.Engine(W, H, max_batch=B) as e:
        e.set_io_slots(2)
        e.set_Q(cases.Q_REFERENCE)
        e.set_mean_rois(rois)
        st = api.STAGE_XYZ | api.STAGE_MEANS
        e.debug_postfilter(a, median=False, stages=st)
        e.debug_postfilter(b, median=False, stages=st)
        for age, m in ((1, a), (0, b)):
            r = e.download(B, xyz=True, means=True, age=age)
            check("disp age %d" % age, r["disp"], m)
            check("means age %d" % age, r["means"], ref_means(m, rois))
            assert_same_floats(r["xyz"], ref_xyz(m, cases.Q_REFERENCE), "xyz age %d" % age)


def minmax_maps():
    rng = np.random.default_rng(10)
    out = {}
    m = rng.choice([-32768, -16, -1, 0], (1, 50, 70)).astype(np.int16)
    out["no_positive"] = m
    m = m.copy()
    m[0, -1, -1] = 5
    out["last_pixel"] = m
    m = rng.integers(-32768, 1, (2, 50, 70)).astype(np.int16)
    m[0, 3, 4], m[0, 40, 60], m[1, 10, 10] = 1, 32767, 1
    out["limits"] = m
    m = np.stack([rng.integers(1000 * b + 1, 1000 * b + 1000, (50, 70)) for b in range(4)]).astype(np.int16)
    m[rng.random(m.shape) < 0.2] = -16
    out["disjoint"] = m
    m = rng.integers(-64, 4000, (1, 2160, 3840)).astype(np.int16)
    out["4k"] = m
    assert (ref_minmax(out["no_positive"]) == 0).all() and tuple(ref_minmax(out["last_pixel"])[0]) == (5, 5)
    assert tuple(ref_minmax(out["limits"])[0]) == (1, 32767)
    return out


@gpu
@pytest.mark.parametrize("name", ["no_positive", "last_pixel", "limits", "disjoint", "4k"])
def test_minmax(name):
    m = minmax_maps()[name]
    B, H, W = m.shape
    with api.Engine(W, H, max_batch=B) as e:
        e.debug_postfilter(m, median=False)
        check("minmax " + name, e.download_minmax(B), ref_minmax(m))


@gpu
def test_postfilter_hook_row_stride_and_order():
    """A row stride above the width, and median then speckle in one call (cv::StereoSGBM's order)."""
    B, H, W = 2, 40, 100
    m = blob_maps(B, H, W, 0, 16 * 65, seed=11)
    padded = np.zeros((B, H, W + 12), np.int16)
    padded[:, :, :W] = m
    with api.Engine(W, H, max_batch=B) as e:
        e.debug_postfilter(padded[:, :, :W], median=True, new_val=0, speckle_size=20, speckle_diff=32)
        check("raw", e.debug_read(2, B), m)
        check("final", e.download(B)["disp"], ref_speckle(ref_median(m), 0, 20, 32))


@gpu
def test_postfilter_hook_rejections():
    """Rejected calls take no I/O slot; the results of the last two calls stay as they were."""
    B, H, W = 1, 16, 40
    a, b = means_map(B, H, W, seed=12), means_map(B, H, W, seed=13)
    with api.Engine(W, H, max_batch=B) as e:
        e.set_io_slots(2)
        e.debug_postfilter(a, median=False)
        e.debug_postfilter(b, median=False)
        bad = [dict(stages=api.STAGE_SGBM), dict(stages=api.STAGE_XYZ), dict(stages=api.STAGE_MEANS),
               dict(speckle_size=10, new_val=40000)]
        for kw in bad:
            with pytest.raises(api.MvsvError) as err:
                e.debug_postfilter(a if "stages" in kw else b, median=False, **kw)
            assert err.value.code in (-1, -4), kw
        with pytest.raises(api.MvsvError) as err:
            e.debug_postfilter(np.zeros((2, H, W), np.int16))
        assert err.value.code == -1
        check("age 0", e.download(B)["disp"], b)
        check("age 1", e.download(B, age=1)["disp"], a)
