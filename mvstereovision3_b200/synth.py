"""Synthetic random-dot stereograms with a known disparity ramp (SURVEY.md section 8d).

The reference ships no images (only calibration YAMLs), so every test and bench
input is made here, seeded and reproducible with numpy alone.
"""
import os

import numpy as np


def _blur3(a):
    """3x3 binomial blur ([1 2 1]/4 separable), replicate border, round-half-up, uint8."""
    a = a.astype(np.uint16)
    p = np.pad(a, ((0, 0), (1, 1)), mode="edge")
    a = (p[:, :-2] + 2 * p[:, 1:-1] + p[:, 2:] + 2) >> 2
    p = np.pad(a, ((1, 1), (0, 0)), mode="edge")
    a = (p[:-2] + 2 * p[1:-1] + p[2:] + 2) >> 2
    return a.astype(np.uint8)


def stereogram(height, width, min_disp, num_disp, seed=0, noise=4):
    """Return (left, right, true_disparity_per_row) uint8 H x W images.

    texture = blurred uniform noise; left = tex[:, :W]; right[y, x] = tex[y, x + d(y)] with
    d(y) = dmin + y*(dmax-dmin)//(H-1), dmin = 2, dmax = minD + D - 4; additive uniform noise on
    the right image in [-noise, +noise].
    """
    rng = np.random.default_rng(seed)
    max_d = min_disp + num_disp
    dmin, dmax = 2, max(max_d - 4, 2)
    tex = rng.integers(0, 256, size=(height, width + max(dmax, 0) + 8), dtype=np.uint8)
    tex = _blur3(tex)
    left = np.ascontiguousarray(tex[:, :width])
    d = dmin + (np.arange(height) * (dmax - dmin)) // max(height - 1, 1)
    cols = np.arange(width)[None, :] + d[:, None]
    right = np.take_along_axis(tex, cols, axis=1)
    if noise > 0:
        n = rng.integers(-noise, noise + 1, size=right.shape)
        right = np.clip(right.astype(np.int16) + n, 0, 255).astype(np.uint8)
    return left, np.ascontiguousarray(right), d


def random_pair(height, width, seed=0):
    """Unstructured pair (independent blurred noise) - exercises every code path, matches nothing."""
    rng = np.random.default_rng(seed)
    a = _blur3(rng.integers(0, 256, size=(height, width), dtype=np.uint8))
    b = _blur3(rng.integers(0, 256, size=(height, width), dtype=np.uint8))
    return a, b


def encode_map(m):
    """float32 map -> int32 second differences along rows of its bit patterns (wrapping).  The maps are smooth, so
    these deflate about six times smaller than the floats themselves; decode_map restores them bit for bit."""
    return np.diff(m.view(np.int32), n=2, axis=1, prepend=np.zeros((m.shape[0], 2), np.int32))


def decode_map(d):
    return np.cumsum(np.cumsum(d, axis=1, dtype=np.int32), axis=1, dtype=np.int32).view(np.float32)


def load_rectification(golden_dir):
    """The rectification fixture of the reference's parameters/baseline_small calibration (written by
    tests/golden/make_golden.py): cv2's float maps m1x, m1y, m2x, m2y, the display ROI `roi`, Q, and the seed-7 pair
    remapped and cropped by cv2 (rectL, rectR)."""
    g = dict(np.load(os.path.join(golden_dir, "rectify_baseline_small.npz")))
    with np.load(os.path.join(golden_dir, "rectify_baseline_small_maps.npz")) as maps:
        g.update((k, decode_map(maps[k])) for k in maps.files)
    return g
