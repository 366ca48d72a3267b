"""A geometry change the engine rejects leaves it as it was: the image size, the rectification maps and the buffers a
compute needs.  Each case installs a geometry, computes, makes the rejected call, and then finds the same size, the
same device maps and bit-identical disparities from the same compute."""
import numpy as np
import pytest

import cases
from mvstereovision3_b200 import api, synth

ERR_INVALID, ERR_UNSUPPORTED = -1, -5
SGBM = dict(minDisp=1, numDisp=64, blockSize=13, disp12MaxDiff=0, preFilterCap=0, uniquenessRatio=0,
            speckleWindowSize=150, speckleRange=2, disparityMode=0)


def _state(e, compute, cams, roi):
    """the image size, each camera's device map (or the error code reading it gives) and the disparities of `compute`"""
    compute()
    disp = e.download(1)["disp"]
    maps = []
    for cam in cams:
        try:
            maps.append(e.read_rectify_map(cam, roi))
        except api.MvsvError as x:
            maps.append(x.code)
    return (e.info.width, e.info.height), maps, disp


def _assert_same(before, after):
    assert after[0] == before[0]
    for a, b in zip(after[1], before[1]):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(after[2], before[2])


@pytest.mark.gpu
def test_rejected_map_upload_keeps_the_cameras_maps():
    """Frame 4100x8 resized by 8: camera 0's maps with a 100-wide ROI give 800x64 images.  The same camera's maps with a
    4000-wide ROI would give 32000-wide ones and are rejected; the 100-wide maps stay."""
    fw, fh = 4100, 8
    mx, my = cases.warp_maps(fh, fw, 1)
    roi = (0, 0, 100, fh)
    l, r = synth.random_pair(64, 800, seed=1)
    with api.Engine(fw, fh) as e:
        e.set_resize(8)
        e.upload_rectify_maps(0, mx, my, roi)
        e.set_sgbm_params(**SGBM)
        before = _state(e, lambda: e.compute(l, r, api.STAGE_SGBM), (0,), roi)
        assert before[0] == (800, 64)
        with pytest.raises(api.MvsvError) as x:
            e.upload_rectify_maps(0, mx, my, (0, 0, 4000, fh))
        assert x.value.code == ERR_INVALID
        _assert_same(before, _state(e, lambda: e.compute(l, r, api.STAGE_SGBM), (0,), roi))


@pytest.mark.gpu
def test_rejected_reset_rectification_keeps_the_maps():
    """Frame 8192x1100, ROI 1000x1000, numDisp 256: the SGBM parameters fit the ROI but not the frame (a frame's cost
    volume would exceed 2^31 cells), so dropping the maps is rejected and the maps stay."""
    fw, fh = 8192, 1100
    mx, my = cases.warp_maps(fh, fw, 2)
    roi = (100, 50, 1000, 1000)
    l, r = synth.random_pair(fh, fw, seed=2)
    with api.Engine(fw, fh) as e:
        for cam in (0, 1):
            e.upload_rectify_maps(cam, mx, my, roi)
        e.set_sgbm_params(**dict(SGBM, numDisp=256))

        def compute():
            e.compute(l, r, api.STAGE_RECTIFY | api.STAGE_SGBM)

        before = _state(e, compute, (0, 1), roi)
        with pytest.raises(api.MvsvError) as x:
            e.reset_rectification()
        assert x.value.code == ERR_UNSUPPORTED
        _assert_same(before, _state(e, compute, (0, 1), roi))


@pytest.mark.gpu
def test_rejected_image_size_keeps_the_buffers():
    """Frame 2048x2048, max_batch 8, resize by 8: a full-frame rectification would give 8 x 16384 x 16384 = 2^31 pixels
    per batch and is rejected; the engine keeps its 2048x2048 images and their buffers, and still has no map."""
    n = 2048
    mx, my = cases.warp_maps(n, n, 3)
    roi = (0, 0, n, n)
    l, r = synth.random_pair(n, n, seed=3)
    with api.Engine(n, n, max_batch=8) as e:
        e.set_bm_params(numDisp=16, blockSize=15, preFilterCap=31, textureThreshold=10, uniquenessRatio=15)
        e.set_resize(8)
        before = _state(e, lambda: e.compute(l, r, api.STAGE_BM), (0,), roi)
        with pytest.raises(api.MvsvError) as x:
            e.upload_rectify_maps(0, mx, my, roi)
        assert x.value.code == ERR_UNSUPPORTED
        _assert_same(before, _state(e, lambda: e.compute(l, r, api.STAGE_BM), (0,), roi))
