"""Seeded stereo pairs on which block matchers tie: flat frames, exact matches, periodic structure, saturated and black
regions.  Real camera frames (walls, sky, highlights, shadows, fences, tiles) do this all the time; blurred noise
(mvstereovision3_b200.synth) almost never gives two disparities the same cost, a zero cost or a window without texture.

Every family is a function (H, W, D, seed) -> (left, right), uint8 H x W, deterministic in its arguments; D is the
number of disparities the pair is meant for (stripe periods divide it, flat regions are wider than it).  numpy only."""
import numpy as np

from mvstereovision3_b200 import synth


def _texture(rng, H, W):
    return synth._blur3(rng.integers(0, 256, size=(H, W), dtype=np.uint8))


def _shift(img, W, d):
    """right[y, x] = img[y, x + d] for a source at least W + d wide (the left image is img[:, :W])."""
    return np.ascontiguousarray(img[:, d:d + W])


def _disp(D, seed, lo=1):
    """A disparity inside [lo, D - 2], drawn from the seed."""
    return lo + seed % max(D - 2 - lo, 1)


def zeros(H, W, D, seed):
    z = np.zeros((H, W), np.uint8)
    return z, z.copy()


def whites(H, W, D, seed):
    z = np.full((H, W), 255, np.uint8)
    return z, z.copy()


def flat_levels(H, W, D, seed):
    """left flat at 100, right flat at 140: every disparity costs the same, and more than zero."""
    return np.full((H, W), 100, np.uint8), np.full((H, W), 140, np.uint8)


def same(H, W, D, seed):
    """a textured image paired with itself: zero cost at d = 0."""
    t = _texture(np.random.default_rng(seed), H, W)
    return t, t.copy()


def exact_shift(H, W, D, seed):
    """a textured image and its exact integer shift, no noise: zero cost at the true disparity."""
    d = _disp(D, seed, 2)
    t = _texture(np.random.default_rng(seed), H, W + d)
    return np.ascontiguousarray(t[:, :W]), _shift(t, W, d)


def _stripes(H, W, period, lo=0, hi=255):
    x = np.arange(W)
    row = np.where((x % period) < period // 2, hi, lo).astype(np.uint8)
    return np.ascontiguousarray(np.broadcast_to(row, (H, W)))


def stripes(H, W, D, seed):
    """vertical 0/255 stripes of period 8 (divides every D), shifted by exactly 3: ties every 8 disparities, at zero cost."""
    s = _stripes(H, W + 8, 8)
    return np.ascontiguousarray(s[:, :W]), _shift(s, W, 3)


def stripes_offset(H, W, D, seed):
    """stripes 30/220 left, 45/235 right (a brightness offset): the periodic ties stay, the minimum is above zero."""
    a, b = _stripes(H, W + 8, 8, 30, 220), _stripes(H, W + 8, 8, 45, 235)
    return np.ascontiguousarray(a[:, :W]), _shift(b, W, 3)


def stripes_noise(H, W, D, seed):
    """0/255 stripes with +-3 noise on the right: near-ties a few units apart, exact ties here and there."""
    s = _stripes(H, W + 8, 8)
    r = _shift(s, W, 3).astype(np.int16) + np.random.default_rng(seed).integers(-3, 4, size=(H, W))
    return np.ascontiguousarray(s[:, :W]), np.clip(r, 0, 255).astype(np.uint8)


def checker(H, W, D, seed):
    """a 3 x 3-pixel 0/255 checkerboard (period 6), shifted by exactly 2."""
    y, x = np.mgrid[0:H, 0:W + 6]
    c = np.where(((y // 3) + (x // 3)) % 2 == 0, 255, 0).astype(np.uint8)
    return np.ascontiguousarray(c[:, :W]), _shift(c, W, 2)


def quantised(H, W, D, seed):
    """texture quantised to three grey levels (0, 128, 255), shifted exactly: large plateaus, steps in between."""
    d = _disp(D, seed, 2)
    rng = np.random.default_rng(seed)
    t = synth._blur3(synth._blur3(rng.integers(0, 256, size=(H, W + d), dtype=np.uint8)))
    q = np.digitize(t, [112, 144]).astype(np.uint8) * 127
    q[q == 254] = 255
    return np.ascontiguousarray(q[:, :W]), _shift(q, W, d)


def dots(H, W, D, seed):
    """sparse binary dots (0/255, about 8 % lit), shifted exactly: the prefilter clips at 0 and 2 * cap."""
    d = _disp(D, seed, 2)
    rng = np.random.default_rng(seed)
    t = np.where(rng.random((H, W + d)) < 0.08, 255, 0).astype(np.uint8)
    return np.ascontiguousarray(t[:, :W]), _shift(t, W, d)


def hramp(H, W, D, seed):
    """a horizontal ramp of slope 1 (a constant non-zero x-Sobel response), repeating every 200 columns, shifted exactly."""
    d = _disp(D, seed, 2)
    x = np.arange(W + d)
    row = (28 + (x + 7 * seed) % 200).astype(np.uint8)
    t = np.ascontiguousarray(np.broadcast_to(row, (H, W + d)))
    return np.ascontiguousarray(t[:, :W]), _shift(t, W, d)


def vramp(H, W, D, seed):
    """a vertical ramp: zero x-Sobel response everywhere, the raw channel varies by row only."""
    y = np.arange(H)
    col = (20 + (2 * y + seed) % 216).astype(np.uint8)
    t = np.ascontiguousarray(np.broadcast_to(col[:, None], (H, W)))
    return t, t.copy()


def flat_patches(H, W, D, seed):
    """texture at an exact shift with a flat 90-grey rectangle wider than D, a 255 highlight and a 0 shadow, each at
    its own columns in the left image and shifted with the texture in the right one."""
    d = _disp(D, seed, 2)
    rng = np.random.default_rng(seed)
    t = _texture(rng, H, W + d)
    wf = min(D + 12, (W + d) // 2)
    x0 = int(rng.integers(0, max(W + d - wf, 1)))
    t[H // 6:H - H // 6, x0:x0 + wf] = 90
    for val in (255, 0):
        w = min(D // 2 + 6, (W + d) // 3)
        xx = int(rng.integers(0, max(W + d - w, 1)))
        yy = int(rng.integers(0, max(H - H // 3, 1)))
        t[yy:yy + H // 3, xx:xx + w] = val
    return np.ascontiguousarray(t[:, :W]), _shift(t, W, d)


FAMILIES = {f.__name__: f for f in (zeros, whites, flat_levels, same, exact_shift, stripes, stripes_offset, stripes_noise,
                                    checker, quantised, dots, hramp, vramp, flat_patches)}


def pair(name, H, W, D, seed=0):
    return FAMILIES[name](H, W, D, seed)


def scene(H, W, minD, D, seed, noise=2):
    """A full frame in the way a camera sees a room: a textured background plane at a small disparity, a textureless
    wall wider than D, a saturated highlight, a black region, a patch of vertical stripes (blinds) and a textured
    foreground plane at a larger disparity.  `noise` (+-) is added to the right image's textured planes only; flat,
    saturated, black and striped regions match exactly."""
    rng = np.random.default_rng(seed)
    maxd = minD + D
    dbg = max(minD + 2, minD + D // 8)
    dfg = max(dbg + 2, maxd - 6)
    pad = maxd + 8
    bg = _texture(rng, H, W + pad)
    fg = _texture(rng, H, W + pad)
    flat = np.zeros((H, W + pad), bool)
    # regions in scene coordinates (columns of the left image)
    wall = (H // 8, H // 2, W // 10, W // 10 + max(D + 24, W // 4))
    light = (H // 10, H // 4, W // 2, W // 2 + max(D // 2, 24))
    dark = (2 * H // 3, H - H // 12, W // 12, W // 12 + max(D // 2 + 8, 40))
    blind = (H // 2 + H // 12, 5 * H // 6, W // 2 + W // 8, min(W // 2 + W // 8 + max(D, 64), W + pad))
    for (y0, y1, x0, x1), v in ((wall, 110), (light, 255), (dark, 0)):
        bg[y0:y1, x0:x1] = v
        flat[y0:y1, x0:x1] = True
    y0, y1, x0, x1 = blind
    bg[y0:y1, x0:x1] = _stripes(y1 - y0, x1 - x0, 8, 20, 230)
    flat[y0:y1, x0:x1] = True
    left = bg[:, :W].copy()
    right = bg[:, dbg:dbg + W].copy()
    rflat = flat[:, dbg:dbg + W].copy()
    # the foreground plane, left of the image centre, at disparity dfg
    fy0, fy1, fx0, fx1 = H // 3, H - H // 5, maxd + W // 3, maxd + W // 3 + W // 6
    fx1 = min(fx1, W)
    left[fy0:fy1, fx0:fx1] = fg[fy0:fy1, fx0:fx1]
    right[fy0:fy1, fx0 - dfg:fx1 - dfg] = fg[fy0:fy1, fx0:fx1]
    rflat[fy0:fy1, fx0 - dfg:fx1 - dfg] = False
    if noise:
        n = rng.integers(-noise, noise + 1, size=(H, W))
        right = np.where(rflat, right, np.clip(right.astype(np.int16) + n, 0, 255)).astype(np.uint8)
    return np.ascontiguousarray(left), np.ascontiguousarray(right)
