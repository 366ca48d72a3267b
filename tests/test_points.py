"""The point list of MVSV_STAGE_POINTS (Utility::dmap2pcl, reference src/utility.cpp:242-262) and mvsv_download_points:
over the batch, in (frame, row, column) order, the pixels with disparity > 0, reprojected exactly as MVSV_STAGE_XYZ does.

The oracle is exact: the dense XYZ of the same compute (points == xyz.reshape(-1, 3)[disp.ravel() > 0], compared as
uint32 so that NaN and inf of a Q with a zero divisor compare too) and ref_xyz of tests/test_postfilters.py.  The crafted
maps go through the test hook mvsv_debug_postfilter; their runs of valid pixels straddle the boundaries of the kernels'
tiles (PT_TILE pixels of one frame, 8 per thread, csrc/filters.cu), warps and frames.  The CPU part checks the numpy
reference against ref_xyz and the packed-float ply::write overload against the Vec4 one."""
import os
import subprocess

import numpy as np
import pytest

import cases
from mvstereovision3_b200 import api, synth
from test_postfilters import XYZ_SPECIAL, assert_same_floats, q_matrices, ref_xyz, xyz_map

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_INVALID, ERR_STATE = -1, -4
TILE = 2048                     # PT_TILE of csrc/filters.cu: 256 threads x 8 pixels
LIMITS = (-32768, -1, 0, 1, 32767)


# ------------------------------------------------------------------------------------------------ reference
def ref_points(disp, Qs):
    """dmap2pcl's list in numpy: disp [B, H, W] int16, Qs one Q or one per frame -> (offsets int64 [B + 1], points
    float32 [n, 3]).  Only the valid pixels are reprojected, with ref_xyz's arithmetic."""
    B = disp.shape[0]
    Qs = [Qs] * B if np.asarray(Qs).ndim == 2 else list(Qs)
    offsets = np.zeros(B + 1, np.int64)
    out = []
    for b in range(B):
        y, x = np.nonzero(disp[b] > 0)
        q = np.asarray(Qs[b], np.float32).astype(np.float64).reshape(4, 4)
        d = (disp[b][y, x].astype(np.float32) / np.float32(16)).astype(np.float64)
        x, y = x.astype(np.float64), y.astype(np.float64)
        cc = [(((q[r, 0] * x) + q[r, 1] * y) + q[r, 2] * d + q[r, 3]).astype(np.float32) for r in range(4)]
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            X, Y, Z = cc[0] / cc[3], cc[1] / cc[3], cc[2] / cc[3]
            Z = np.where(np.isinf(Z / np.float32(1000)), np.float32(0), Z)
        out.append(np.stack([X, Y, Z], -1).astype(np.float32).reshape(-1, 3))
        offsets[b + 1] = offsets[b] + len(y)
    return offsets, np.concatenate(out)


def dense_points(disp, xyz):
    """the list as a selection of the dense XYZ"""
    return xyz.reshape(-1, 3)[disp.ravel() > 0]


def counts(disp):
    return np.concatenate([[0], np.cumsum((disp > 0).reshape(len(disp), -1).sum(1))]).astype(np.int64)


def same_bits(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.flatnonzero(got.view(np.uint32).ravel() != want.view(np.uint32).ravel())
    assert bad.size == 0, "%s: %d floats differ, first at %d: %s vs %s" % (what, bad.size, bad[0], got.ravel()[bad[0]],
                                                                          want.ravel()[bad[0]])


# ------------------------------------------------------------------------------------------------ crafted maps
# (W, H, B): frames of exactly one tile, one tile +- 1 pixel, several tiles plus a remainder; widths not a multiple of 4,
# 16 or the tile; frames whose size is and is not a multiple of 8 pixels (16-byte aligned frame starts or not)
SHAPES = ((5, 3, 3), (7, 5, 3), (13, 7, 5), (64, 32, 3), (2047, 1, 3), (2049, 1, 3), (683, 3, 2), (100, 41, 2),
          (40, 103, 3), (752, 479, 2))
SHAPE_IDS = ["%dx%dx%d" % s for s in SHAPES]


def runs_map(W, H, B, seed):
    """Alternating runs of valid and invalid pixels over the batch's linear index, with lengths around 1, a thread's 8
    pixels, a warp's 256, the tile and a frame; every value of LIMITS and XYZ_SPECIAL occurs."""
    rng = np.random.default_rng(seed)
    n = B * H * W
    lens = [1, 2, 7, 8, 9, 31, 32, 33, 255, 256, 257, TILE - 1, TILE, TILE + 1, H * W - 1, H * W, H * W + 1]
    flat = np.zeros(n, np.int16)
    i, valid = int(rng.integers(0, 9)), True
    while i < n:
        k = int(rng.choice(lens))
        vals = [v for v in LIMITS + XYZ_SPECIAL if (v > 0) == valid]
        flat[i:i + k] = rng.choice(vals, min(k, n - i))
        i, valid = i + k, not valid
    m = flat.reshape(B, H, W)
    m.reshape(-1)[:len(LIMITS)] = LIMITS
    return m


def frame_kinds(W, H):
    """all-invalid frames between full ones, an all-valid frame, and one valid pixel at the batch's last pixel"""
    full = xyz_map(W, H, 1, seed=11)[0]
    empty = np.where(full > 0, -full, full).astype(np.int16)
    empty[empty == -32768] = 0
    allv = np.abs(full.astype(np.int32)).clip(1, 32767).astype(np.int16)
    last = np.zeros((H, W), np.int16)
    last[-1, -1] = 1
    return np.stack([full, empty, empty, allv, empty, full, last])


# ================================================================================================ CPU part
@pytest.mark.parametrize("qname", list(q_matrices()))
def test_ref_points_is_the_selection_of_ref_xyz(qname):
    Q = q_matrices()[qname]
    for k, (W, H, B) in enumerate(SHAPES[:-1]):
        for m in (runs_map(W, H, B, seed=k), frame_kinds(W, H)):
            offs, pts = ref_points(m, Q)
            assert np.array_equal(offs, counts(m))
            assert_same_floats(pts, dense_points(m, ref_xyz(m, Q)), "%s %dx%dx%d" % (qname, W, H, B))


def test_runs_map_covers_the_boundaries():
    m = runs_map(2049, 1, 3, seed=0)
    assert set(LIMITS) <= set(np.unique(m).tolist())
    k = frame_kinds(5, 3)
    assert counts(k)[1:].tolist() == np.cumsum([(f > 0).sum() for f in k]).tolist()
    assert (k[1] <= 0).all() and (k[3] > 0).all() and (k[6] > 0).sum() == 1 and k[6, -1, -1] > 0


def build_ply_points(tmp_path):
    exe = str(tmp_path / "ply_points")
    subprocess.check_call(["g++", "-std=c++11", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "ply_points.cpp"), "-o", exe])
    return exe


@pytest.mark.parametrize("mode", [0, 1], ids=["PLAIN", "WITH_COLOR"])
def test_ply_packed_floats_equal_vec4(tmp_path, mode):
    """ply::write(const float* xyz, size_t n) writes the bytes of the std::vector<Vec4> overload."""
    exe = build_ply_points(tmp_path)
    m = xyz_map(13, 7, 5)
    offs, pts = ref_points(m, cases.Q_REFERENCE)
    extra = np.array([[0, -0.0, 1e30], [np.inf, -np.inf, 12345.678], [1e-30, 3.5, -7.25]], np.float32)
    for name, p in (("points", pts), ("extra", extra), ("none", pts[:0])):
        src = tmp_path / (name + ".bin")
        src.write_bytes(np.ascontiguousarray(p, np.float32).tobytes())
        a, b = tmp_path / (name + "_vec4.ply"), tmp_path / (name + "_packed.ply")
        subprocess.check_call([exe, str(src), "17", "1009", str(mode), str(a), str(b)])
        got, want = b.read_bytes(), a.read_bytes()
        assert got == want, name
        assert ("element vertex %d\n" % len(p)).encode() in got and got.count(b"\n") == len(p) + 9 + 3 * mode


# ================================================================================================ GPU part
gpu = pytest.mark.gpu
SGBM = dict(minDisp=1, numDisp=64, blockSize=13, disp12MaxDiff=0, preFilterCap=0, uniquenessRatio=0,
            speckleWindowSize=150, speckleRange=2, disparityMode=0)          # configs/sgbm.yml at numDisp 64 (cfg 2)
BM = [p for name, p, _, _ in cases.BM_CASES if name == "bm_yml"][0]          # configs/bm.yml


def pairs(B, H, W, seed=0):
    g = [synth.stereogram(H, W, 1, 80, seed=seed + i)[:2] for i in range(B)]
    return np.stack([p[0] for p in g]), np.stack([p[1] for p in g])


def check_list(e, B, disp, xyz, what, age=0):
    """download_points against the dense XYZ of the same compute and the frame counts of its map"""
    offs, pts = e.download_points(B, age=age)
    assert np.array_equal(offs, counts(disp)), what
    same_bits(pts, dense_points(disp, xyz), what)
    return offs, pts


@gpu
@pytest.mark.parametrize("matcher", ["sgbm", "bm"])
def test_matchers(matcher):
    H, W, MB = 90, 260, 9
    with api.Engine(W, H, max_batch=MB) as e:
        if matcher == "sgbm":
            e.set_sgbm_params(**SGBM)
        else:
            e.set_bm_params(**BM)
        e.set_Q(cases.Q_REFERENCE)
        st = api.STAGE_SGBM if matcher == "sgbm" else api.STAGE_BM
        for B in (1, 4, MB):
            L, R = pairs(B, H, W, seed=B)
            e.compute(L, R, st | api.STAGE_XYZ | api.STAGE_POINTS)
            r = e.download(B, xyz=True)
            offs, pts = check_list(e, B, r["disp"], r["xyz"], "%s B=%d" % (matcher, B))
            assert 0 < offs[-1] < B * H * W
            e.compute(L, R, st | api.STAGE_POINTS)                # POINTS alone: the same list
            offs2, pts2 = e.download_points(B)
            assert np.array_equal(offs2, offs)
            same_bits(pts2, pts, "%s B=%d POINTS alone" % (matcher, B))


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=SHAPE_IDS)
def test_crafted_runs(shape):
    W, H, B = shape
    m = runs_map(W, H, B, seed=W + H)
    with api.Engine(W, H, max_batch=B) as e:
        e.set_Q(cases.Q_REFERENCE)
        for batch in sorted({1, B}):
            e.debug_postfilter(m[:batch], median=False, stages=api.STAGE_XYZ | api.STAGE_POINTS)
            xyz = e.download(batch, xyz=True)["xyz"]
            offs, pts = check_list(e, batch, m[:batch], xyz, "%s batch %d" % (SHAPE_IDS[SHAPES.index(shape)], batch))
            want_offs, want = ref_points(m[:batch], cases.Q_REFERENCE)
            assert np.array_equal(offs, want_offs)
            assert_same_floats(pts, want, "runs vs ref_points")


@gpu
@pytest.mark.parametrize("qname", list(q_matrices()))
@pytest.mark.parametrize("shape", [(13, 7), (64, 32), (2049, 1), (40, 103)], ids=["13x7", "64x32", "2049x1", "40x103"])
def test_crafted_frames(qname, shape):
    """all-invalid frames (count 0) between full ones, an all-valid frame, one valid pixel at the last pixel of the
    batch; the Q set, including a divisor that is exactly 0 (inf and NaN coordinates)"""
    W, H = shape
    Q = q_matrices()[qname]
    m = frame_kinds(W, H)
    with api.Engine(W, H, max_batch=len(m)) as e:
        e.set_Q(Q)
        e.debug_postfilter(m, median=False, stages=api.STAGE_XYZ | api.STAGE_POINTS)
        xyz = e.download(len(m), xyz=True)["xyz"]
        offs, pts = check_list(e, len(m), m, xyz, "%s %dx%d" % (qname, W, H))
        # frames 1, 2 and 4 hold no point, frame 3 one per pixel, frame 6 one
        assert offs[1] == offs[2] == offs[3] and offs[4] == offs[5]
        assert offs[4] - offs[3] == W * H and offs[-1] - offs[-2] == 1
        want_offs, want = ref_points(m, Q)
        assert np.array_equal(offs, want_offs)
        assert_same_floats(pts, want, "%s %dx%d vs ref_points" % (qname, W, H))
        e.debug_postfilter(m, median=False, stages=api.STAGE_POINTS)       # POINTS alone
        offs2, pts2 = e.download_points(len(m))
        assert np.array_equal(offs2, offs)
        same_bits(pts2, pts, "POINTS alone")


@gpu
def test_rigs():
    """frames of several rigs with different Q (mvsv_set_frame_rigs): each frame's points use its rig's Q"""
    W, H, B = 100, 41, 7
    qs = q_matrices()
    rig_q = {0: cases.Q_REFERENCE, 3: qs["rectify"], 9: qs["neg_tx"], 63: qs["zero_div"]}
    table = [3, 0, 63, 9, 3, 63]                              # frame 6: past the table, rig 0
    m = runs_map(W, H, B, seed=3)
    with api.Engine(W, H, max_batch=B) as e:
        for r, q in rig_q.items():
            e.set_Q(q, rig=r)
        e.set_frame_rigs(table)
        e.debug_postfilter(m, median=False, stages=api.STAGE_XYZ | api.STAGE_POINTS)
        xyz = e.download(B, xyz=True)["xyz"]
        offs, pts = check_list(e, B, m, xyz, "rigs")
        want_offs, want = ref_points(m, [rig_q[r] for r in table + [0]])
        assert np.array_equal(offs, want_offs)
        assert_same_floats(pts, want, "rigs vs ref_points")


@gpu
def test_two_io_slots():
    """download_points(age=1) after the next compute has been submitted returns the earlier compute's list"""
    H, W, B = 72, 200, 5
    (La, Ra), (Lb, Rb) = pairs(B, H, W, seed=20), pairs(B, H, W, seed=40)
    st = api.STAGE_SGBM | api.STAGE_XYZ | api.STAGE_POINTS
    want = []
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**SGBM)
        e.set_Q(cases.Q_REFERENCE)
        for L, R in ((La, Ra), (Lb, Rb)):
            e.compute(L, R, st)
            r = e.download(B, xyz=True)
            want.append((counts(r["disp"]), dense_points(r["disp"], r["xyz"])))
        e.set_io_slots(2)
        out = api.pinned((B * H * W, 3), np.float32)
        e.compute(La, Ra, st)
        e.compute(Lb, Rb, st)
        for age, (w_offs, w_pts) in ((1, want[0]), (0, want[1])):
            offs, pts = e.download_points(B, age=age, out=out.array)
            assert np.array_equal(offs, w_offs), age
            same_bits(pts, w_pts, "age %d" % age)
            assert pts.base is not None and np.shares_memory(pts, out.array)
        out.close()


def _device_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


DEVICE_LISTS = [[0, 0], [0, 0, 0]] + ([list(range(_device_count()))] if _device_count() >= 2 else [])


@gpu
@pytest.mark.parametrize("devs", DEVICE_LISTS, ids=["x".join(map(str, d)) for d in DEVICE_LISTS])
def test_devices(devs):
    """a multi-device ctx: the list and offsets of every batch size (fewer frames than parts too) are those of one
    engine; with two I/O slots, age 1 as well"""
    H, W = 72, 200
    n = len(devs)
    MB = 2 * n + 1
    st = api.STAGE_SGBM | api.STAGE_POINTS
    L, R = pairs(MB, H, W, seed=7)
    with api.Engine(W, H, max_batch=MB) as one, api.Engine(W, H, max_batch=MB, devices=devs) as many:
        for e in (one, many):
            e.set_sgbm_params(**SGBM)
            e.set_Q(cases.Q_REFERENCE)
        lists = {}
        for B in sorted({1, n - 1, n, n + 1, MB} - {0}):
            one.compute(L[:B], R[:B], st)
            many.compute(L[:B], R[:B], st)
            w_offs, w_pts = lists[B] = one.download_points(B)
            offs, pts = many.download_points(B)
            assert np.array_equal(offs, w_offs), B
            same_bits(pts, w_pts, "%s B=%d" % (devs, B))
        many.set_io_slots(2)
        many.compute(L[:1], R[:1], st)
        many.compute(L, R, st)
        offs, pts = many.download_points(1, age=1)
        assert np.array_equal(offs, lists[1][0])
        same_bits(pts, lists[1][1], "age 1")
        # the capacity check of the gathered list, and the size query
        total = int(lists[MB][0][-1])
        offs = np.full(MB + 1, -7, np.int64)
        sentinel = np.full((total, 3), 1.5, np.float32)
        rc = many._lib.mvsv_download_points(many._ctx, 0, offs.ctypes.data, sentinel.ctypes.data, total - 1)
        assert rc == ERR_INVALID
        assert np.array_equal(offs, lists[MB][0]) and (sentinel == 1.5).all()
        offs[:] = -7
        assert many._lib.mvsv_download_points(many._ctx, 0, offs.ctypes.data, None, 0) == 0
        assert np.array_equal(offs, lists[MB][0])


@gpu
def test_errors():
    H, W, B = 72, 200, 3
    L, R = pairs(B, H, W, seed=9)
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**SGBM)
        e.compute(L, R, api.STAGE_SGBM)
        disp = e.download(B)["disp"]
        # no Q: rejected before an I/O slot is taken, the earlier map stays downloadable
        with pytest.raises(api.MvsvError) as ei:
            e.compute(L, R, api.STAGE_SGBM | api.STAGE_POINTS)
        assert ei.value.code == ERR_STATE
        assert np.array_equal(e.download(B)["disp"], disp)
        # the compute did not run POINTS
        with pytest.raises(api.MvsvError) as ei:
            e.download_points(B)
        assert ei.value.code == ERR_STATE
        # a frame's rig without Q
        e.set_Q(cases.Q_REFERENCE)
        e.set_frame_rigs([0, 5])
        with pytest.raises(api.MvsvError) as ei:
            e.compute(L, R, api.STAGE_SGBM | api.STAGE_POINTS)
        assert ei.value.code == ERR_STATE
        e.set_frame_rigs([])
        e.compute(L, R, api.STAGE_SGBM | api.STAGE_XYZ | api.STAGE_POINTS)
        r = e.download(B, xyz=True)
        want_offs, want = counts(r["disp"]), dense_points(r["disp"], r["xyz"])
        total = int(want_offs[-1])
        assert total > 0
        # the size query: points == NULL writes the offsets only
        offs = np.full(B + 1, -7, np.int64)
        assert e._lib.mvsv_download_points(e._ctx, 0, offs.ctypes.data, None, 0) == 0
        assert np.array_equal(offs, want_offs)
        # capacity < total: the offsets are written, the points are not touched
        offs[:] = -7
        sentinel = np.full((total, 3), 2.5, np.float32)
        assert e._lib.mvsv_download_points(e._ctx, 0, offs.ctypes.data, sentinel.ctypes.data, total - 1) == ERR_INVALID
        assert np.array_equal(offs, want_offs) and (sentinel == 2.5).all()
        with pytest.raises(api.MvsvError) as ei:
            e.download_points(B, out=np.empty((total - 1, 3), np.float32))
        assert ei.value.code == ERR_INVALID
        # exactly enough
        assert e._lib.mvsv_download_points(e._ctx, 0, offs.ctypes.data, sentinel.ctypes.data, total) == 0
        same_bits(sentinel, want, "capacity == total")
        # ages past the I/O slots
        with pytest.raises(api.MvsvError) as ei:
            e.download_points(B, age=1)
        assert ei.value.code == ERR_INVALID
