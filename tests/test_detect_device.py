"""Obstacle detection on the device: MVSV_STAGE_DETECT, mvsv_set_detection, mvsv_download_obstacles(_stream).

The authority is include/mvsv_detection.hpp: tests/cpp/detect_records.cpp runs both host detectors frame by frame and
prints the records they find.  On the CPU that driver is checked against a numpy restatement of the contract in
include/mvsv.h; on the GPU the engine's records must equal the driver's, bit for bit, on the engine's own means, and the
restatement's on crafted maps (debug_postfilter) whose means sit on the edges of the ranges."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import cases
import test_devices as td
from mvstereovision3_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_INVALID, ERR_STATE = -1, -4
f32, f64 = np.float32, np.float64
SENT = -7.0


# ---- the restatement ---------------------------------------------------------------------------------------------------
def dvalue(dist, Q):
    """Utility::calcDMapValues({0, 0, dist * 1000}, Q).dValue in float arithmetic"""
    z = f32(dist) * f32(1000)
    with np.errstate(all="ignore"):
        return f32(f32(f32(Q[2, 3]) - z * f32(Q[3, 3])) / f32(z * f32(Q[3, 2]))) * f32(16)


def coordinate(x, y, value, Q):
    """Utility::calcCoordinate: double accumulation k = 0..3 from 0, float components, times the double reciprocal"""
    v = [f64(f32(x)), f64(f32(y)), f64(f32(value) / f32(16)), f64(1.0)]
    c = []
    for r in range(4):
        acc = f64(0.0)
        for k in range(4):
            acc = acc + f64(Q[r, k]) * v[k]
        c.append(f32(acc))
    with np.errstate(all="ignore"):
        inv = f64(1.0) / f64(c[3])
        out = [f32(f64(cr) * inv) for cr in c]
        if np.isinf(out[2] / f32(1000)):
            out[2] = f32(0)
    return out


def restate(means, det, centers, dists, Qs):
    """records of every frame: means [F, n], det [n], centers [n, 2], dists [ndet, 2], Qs [F, 4, 4] (each frame's Q)"""
    offs, recs = [0], []
    for f in range(len(means)):
        Q = Qs[f]
        rng = [(dvalue(a, Q), dvalue(b, Q)) for a, b in dists]
        for i in range(len(det)):
            d = int(det[i])
            v = f32(means[f, i])
            if d >= 0 and v < rng[d][0] and v > rng[d][1]:
                recs.append((i, v, coordinate(centers[i][0], centers[i][1], v, Q)))
        offs.append(len(recs))
    out = np.zeros(len(recs), api.OBSTACLE_DTYPE)
    for k, (i, v, xyzw) in enumerate(recs):
        out[k] = (i, v, xyzw)
    return np.array(offs, np.int64), out


def same_records(got, want, what):
    """roi equal; value and xyzw equal bit for bit, except that any NaN matches any NaN (host and device NaN payloads
    differ)"""
    assert got.shape == want.shape, (what, got.shape, want.shape)
    assert np.array_equal(got["roi"], want["roi"]), what
    for key in ("value", "xyzw"):
        a, b = got[key], want[key]
        nan = np.isnan(a) & np.isnan(b)
        bad = (a.view(np.uint32) != b.view(np.uint32)) & ~nan
        assert not bad.any(), "%s: %s differs at %s: %s vs %s" % (what, key, np.argwhere(bad)[0], a[bad][:3], b[bad][:3])


# ---- the C++ driver ----------------------------------------------------------------------------------------------------
def build_driver(tmp_path):
    exe = str(tmp_path / "detect_records")
    subprocess.check_call(["g++", "-std=c++11", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "detect_records.cpp"), "-o", exe])
    return exe


def run_driver(exe, tmp_path, cols, rows, xoff, dists, Qs, means, device=None):
    """(table det, centers, offsets, records, counters [F, 2], build-same flags [F]) of the host detectors; `device`:
    (offsets, records) of a download for buildFromObstacles"""
    (tmp_path / "q.bin").write_bytes(np.ascontiguousarray(Qs, f32).tobytes())
    (tmp_path / "m.bin").write_bytes(np.ascontiguousarray(means, f32).tobytes())
    args = [exe, str(cols), str(rows), str(xoff)] + [repr(float(v)) for v in np.ravel(dists)] + \
        [str(tmp_path / "q.bin"), str(tmp_path / "m.bin")]
    if device is not None:
        (tmp_path / "o.bin").write_bytes(np.ascontiguousarray(device[0], np.int64).tobytes())
        (tmp_path / "r.bin").write_bytes(np.ascontiguousarray(device[1]).tobytes())
        args += [str(tmp_path / "o.bin"), str(tmp_path / "r.bin")]
    lines = subprocess.check_output(args).decode().split("\n")
    det, centers, recs, offs, counters, same = [], [], [], [0], [], []
    for l in lines:
        t = l.split()
        if not t:
            continue
        if t[0] == "T":
            det.append(int(t[1]))
            centers.append((float(t[2]), float(t[3])))
        elif t[0] == "F":
            counters.append((int(t[3]), int(t[4])))
        elif t[0] == "R":
            recs.append((int(t[1]), f32(float.fromhex(t[2])), [f32(float.fromhex(v)) for v in t[3:7]]))
        elif t[0] == "B":
            same.append(int(t[2]))
            offs.append(len(recs))
    out = np.zeros(len(recs), api.OBSTACLE_DTYPE)
    for k, r in enumerate(recs):
        out[k] = r
    return np.array(det), np.array(centers, f32), np.array(offs, np.int64), out, np.array(counters), np.array(same)


def table(cols, rows):
    """both reference detectors over a dMapWork view of cols x rows: detector 0 the 81 Subimages, 1 the Samplepoints;
    centers as MeanDisparityDetection / SamplepointDetection hand them to calcCoordinate"""
    subs = api.subimage_rois(cols, rows)
    sps = api.samplepoint_rois(cols, rows)
    centers = [(x + w // 2, y + h // 2) for x, y, w, h in subs] + [(x + 2, y + 2) for x, y, _, _ in sps]
    return np.array([0] * len(subs) + [1] * len(sps), np.int32), np.array(centers, f32)


def qs_of(Q, F):
    return np.repeat(np.asarray(Q, f32)[None], F, axis=0)


# ---- CPU: the driver (the header) against the restatement ---------------------------------------------------------------
def test_driver_matches_restatement(tmp_path):
    exe = build_driver(tmp_path)
    cols, rows, xoff = 200, 96, 32
    det, centers = table(cols, rows)
    n = len(det)
    F = 5
    Qs = qs_of(cases.Q_REFERENCE, F)
    Qs[1, 0, 3] -= 7.0
    Qs[2, 3, 2] *= 1.3
    Qs[3, 1, 3] += 2.5
    dists = np.array([[0.4, 2.0], [0.6, 3.0]], f32)
    rng = np.random.default_rng(3)
    means = np.floor(rng.uniform(100, 1700, (F, n))).astype(f32)
    means[:, ::6] = 0
    for f in range(F):                 # the edges: exactly first / second, one float step inside and outside
        for d in range(2):
            lo, hi = dvalue(dists[d][0], Qs[f]), dvalue(dists[d][1], Qs[f])
            idx = np.flatnonzero(det == d)[:6]
            means[f, idx] = [lo, hi, np.nextafter(lo, f32(0)), np.nextafter(hi, f32(1e9)), np.nextafter(lo, f32(1e9)),
                             np.nextafter(hi, f32(0))]
    means[4] = 0                       # a frame without hits
    tdet, tcent, offs, recs, counters, same = run_driver(exe, tmp_path, cols, rows, xoff, dists, Qs, means)
    assert np.array_equal(tdet, det) and np.array_equal(tcent, centers)
    w_offs, w_recs = restate(means, det, centers, dists, Qs)
    assert np.array_equal(offs, w_offs)
    same_records(recs, w_recs, "driver")
    assert (same == 1).all()
    assert all(offs[f + 1] - offs[f] > 0 for f in range(4)) and offs[5] == offs[4]
    # the edges: first and second are never hits, the steps inside always are
    for f in range(4):
        got = set(recs["roi"][offs[f]:offs[f + 1]])
        for d in range(2):
            idx = np.flatnonzero(det == d)[:6]
            assert idx[0] not in got and idx[1] not in got and idx[2] in got and idx[3] in got
            assert idx[4] not in got and idx[5] not in got
    assert counters[-1].tolist() == [4, 4]


def test_binding_and_header():
    lib = api.load_library()
    vp, sz, ci = C.c_void_p, C.c_size_t, C.c_int
    assert lib.mvsv_set_detection.argtypes == [vp, vp, vp, ci, vp, ci]
    assert lib.mvsv_download_obstacles.argtypes == [vp, ci, vp, vp, sz]
    assert lib.mvsv_download_obstacles_stream.argtypes == [vp, ci, vp, vp, sz, vp]
    assert api.STAGE_DETECT == 64 and api.OBSTACLE_DTYPE.itemsize == 24
    with open(os.path.join(ROOT, "include", "mvsv.h")) as f:
        header = f.read()
    assert "MVSV_STAGE_DETECT = 64" in header
    for name in ("mvsv_set_detection", "mvsv_download_obstacles", "mvsv_download_obstacles_stream"):
        assert "int %s(" % name in header


# ---- GPU helpers ---------------------------------------------------------------------------------------------------------
def _torch():
    return pytest.importorskip("torch")


def dists_for(means, Q):
    """distances whose disparity range holds the middle of the positive means (Q[3, 3] == 0: dValue = 16 Q23 / (z Q32)),
    so that some ROIs hit and some do not"""
    pos = means[means > 0]
    lo, hi = np.quantile(pos, 0.3), np.quantile(pos, 0.8)
    k = 16 * float(Q[2, 3]) / float(Q[3, 2]) / 1000
    return np.array([[k / hi, k / lo], [k / hi * 1.05, k / lo * 0.95]], f32)


def check_against_driver(e, exe, tmp_path, B, cols, rows, Qs, dists):
    offs, recs = e.download_obstacles(B)
    means = e.download(B, disp=False, means=True)["means"]
    _, _, w_offs, w_recs, _, same = run_driver(exe, tmp_path, cols, rows, 0, dists, Qs, means, device=(offs, recs))
    assert np.array_equal(offs, w_offs)
    same_records(recs, w_recs, "engine vs host detectors")
    assert (same == 1).all()                         # buildFromObstacles on the device's records
    assert 0 < offs[-1] < B * len(means[0])
    return offs, recs


# ---- GPU: the engine's own means against the host detectors --------------------------------------------------------------
@pytest.mark.gpu
def test_cfg3_pipeline(tmp_path):
    """rectify + SGBM + MEANS + DETECT with both detectors on the reference grids of the dMapWork view"""
    exe = build_driver(tmp_path)
    B, FW, FH = 6, 320, 120
    L, R = np.stack([cases.synth.stereogram(FH, FW, 1, 64, seed=60 + i)[0] for i in range(B)]), None
    R = np.stack([cases.synth.stereogram(FH, FW, 1, 64, seed=60 + i)[1] for i in range(B)])
    Q = cases.Q_REFERENCE
    with api.Engine(FW, FH, max_batch=B) as e:
        for cam in range(2):
            mx, my = cases.warp_maps(FH, FW, seed=cam)
            e.upload_rectify_maps(cam, mx, my, (8, 4, 300, 110))
        e.set_sgbm_params(**td.SGBM)
        e.set_Q(Q)
        W, H = e.info.width, e.info.height
        off = api.dmap_roi_offset(64, W)
        cols = W - off
        e.set_mean_rois(api.subimage_rois(cols, H, off) + api.samplepoint_rois(cols, H, off))
        e.compute(L, R, api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_MEANS)
        dists = dists_for(e.download(B, disp=False, means=True)["means"], Q)
        det, centers = table(cols, H)
        e.set_detection(det, centers, dists)
        n0 = e.launch_count
        e.compute(L, R, api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_MEANS)
        n1 = e.launch_count
        e.compute(L, R, api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_MEANS | api.STAGE_DETECT)
        assert e.launch_count - n1 - (n1 - n0) == 3        # count, scan, emit
        e.profile_enable(True)
        e.compute(L, R, api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_MEANS | api.STAGE_DETECT)
        assert e.profile_read()["detect"][1] == 3
        e.profile_enable(False)
        check_against_driver(e, exe, tmp_path, B, cols, H, qs_of(Q, B), dists)


@pytest.mark.gpu
def test_bm_with_filters(tmp_path):
    exe = build_driver(tmp_path)
    B, W, H = 5, 260, 90
    g = [cases.synth.stereogram(H, W, 1, 80, seed=30 + i)[:2] for i in range(B)]
    L, R = np.stack([p[0] for p in g]), np.stack([p[1] for p in g])
    Q = cases.Q_REFERENCE
    with api.Engine(W, H, max_batch=B) as e:
        e.set_bm_params(**td.BM)
        e.set_bm_filters(0, 40, 16)
        e.set_Q(Q)
        det, centers = table(W, H)
        e.set_mean_rois(api.subimage_rois(W, H) + api.samplepoint_rois(W, H))
        e.compute(L, R, api.STAGE_BM | api.STAGE_MEANS)
        dists = dists_for(e.download(B, disp=False, means=True)["means"], Q)
        e.set_detection(det, centers, dists)
        e.compute(L, R, api.STAGE_BM | api.STAGE_MEANS | api.STAGE_DETECT)
        check_against_driver(e, exe, tmp_path, B, W, H, qs_of(Q, B), dists)


@pytest.mark.gpu
def test_three_rigs(tmp_path):
    """three rigs with different Q (td.setup's pipeline): ranges and coordinates differ per rig"""
    exe = build_driver(tmp_path)
    B = 10
    L, R = td.frames(B, seed=3)
    with api.Engine(td.FW, td.FH, max_batch=B) as e:
        stages, _ = td.setup(e, "pipeline", B)
        W, H = e.info.width, e.info.height
        rigs = td.rig_table(B)
        Qs = []
        for rig in rigs:
            k = td.RIGS.index(rig)
            q = cases.Q_REFERENCE.copy()
            q[0, 3] -= 3 * k
            q[3, 2] *= 1 + 0.1 * k
            Qs.append(q)
        Qs = np.array(Qs, f32)
        e.compute(L, R, stages)
        dists = dists_for(e.download(B, disp=False, means=True)["means"], cases.Q_REFERENCE)
        det, centers = table(W, H)
        e.set_detection(det, centers, dists)
        e.compute(L, R, stages | api.STAGE_DETECT)
        check_against_driver(e, exe, tmp_path, B, W, H, Qs, dists)
        assert len(set(rigs)) == 3


# ---- GPU: crafted means through debug_postfilter ----------------------------------------------------------------------
# one-pixel ROIs: the mean of ROI i is pixel i of the map when it is > 1, else 0 (an empty ROI)
CW, CH = 64, 5                    # 320 ROIs: more than one CTA-wide chunk of the kernels
Q_EDGE = np.array([[1, 0, 0, -10.5], [0, 1, 0, -1.25], [0, 0, 0, 64], [0, 0, 0.5, 0]], f32)     # first 32, second 16
DIST_EDGE = np.array([[0.064, 0.128], [0.064, 0.128]], f32)
# c[3] = -0.25 x + 0.5 d: zero at x = 64, value 512 (d = 32), which DIST_W's range (2048 / z: 1024 to 256) holds
Q_ZERO_W = np.array([[1, 0, 0, -10.5], [0, 1, 0, -1.25], [0, 0, 0, 64], [-0.25, 0, 0.5, 0]], f32)
# the same plus a tiny Q[3][3]: c[3] = 1e-38, z = 64 / 1e-38 overflows the float, so z := 0
Q_TINY_W = Q_ZERO_W.copy()
Q_TINY_W[3, 3] = 1e-38
DIST_W = np.array([[0.002, 0.008], [0.0, 0.0]], f32)


def crafted_means(maps):
    m = maps.reshape(len(maps), -1).astype(f32)
    m[m <= 1] = 0
    return m


def one_pixel_rois():
    return [(i % CW, i // CW, 1, 1) for i in range(CW * CH)]


def run_crafted(e, maps, det, centers, dists, Q):
    e.set_Q(Q)
    e.set_detection(det, centers, dists)
    e.debug_postfilter(maps, median=False, stages=api.STAGE_MEANS | api.STAGE_DETECT)
    B = len(maps)
    offs, recs = e.download_obstacles(B)
    w_offs, w_recs = restate(crafted_means(maps), det, centers, dists, qs_of(Q, B))
    assert np.array_equal(offs, w_offs)
    same_records(recs, w_recs, "crafted")
    return offs, recs


@pytest.mark.gpu
def test_crafted_edges():
    assert (dvalue(0.064, Q_EDGE), dvalue(0.128, Q_EDGE)) == (32, 16)
    assert np.isinf(dvalue(0.0, Q_EDGE))               # a detector at distance 0 has an empty range
    n = CW * CH
    rng = np.random.default_rng(9)
    det = rng.integers(-1, 2, n).astype(np.int32)          # detectors interleaved, with untested ROIs
    centers = np.stack([rng.integers(0, 300, n), rng.integers(0, 200, n)], 1).astype(f32)
    maps = np.zeros((4, CH, CW), np.int16)
    maps[0].flat[:] = rng.choice([0, 1, 15, 16, 17, 24, 31, 32, 33, 500], n)   # on, inside and outside the edges
    maps[1] = 40                                                              # no hit
    maps[2] = 24                                                              # every tested ROI hits
    maps[3].flat[:] = rng.choice([0, 1, 17, 31], n)                           # empty ROIs among hits
    with api.Engine(CW, CH, max_batch=4) as e:
        e.set_mean_rois(one_pixel_rois())
        offs, recs = run_crafted(e, maps, det, centers, DIST_EDGE, Q_EDGE)
        assert offs[2] - offs[1] == 0 and offs[3] - offs[2] == (det >= 0).sum()
        f0 = recs[offs[0]:offs[1]]
        assert set(f0["value"]) == {17, 24, 31}
        assert np.all(det[recs["roi"]] >= 0)
        # detector 1 with an empty range (distances 0): only detector 0's ROIs hit
        offs, recs = run_crafted(e, maps, det, centers, np.array([[0.064, 0.128], [0.0, 0.0]], f32), Q_EDGE)
        assert offs[3] - offs[2] == (det == 0).sum() and np.all(det[recs["roi"]] == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("Q", [Q_ZERO_W, Q_TINY_W], ids=["w_zero", "z_overflow"])
def test_crafted_degenerate_w(Q):
    n = CW * CH
    det = np.zeros(n, np.int32)
    centers = np.stack([np.arange(n) % 128, np.arange(n) // 128], 1).astype(f32)
    centers[5] = (64, 3)
    maps = np.full((2, CH, CW), 512, np.int16)
    maps[1].flat[::3] = 300
    with api.Engine(CW, CH, max_batch=2) as e:
        e.set_mean_rois(one_pixel_rois())
        offs, recs = run_crafted(e, maps, det, centers, DIST_W, Q)
        r5 = recs[recs["roi"] == 5][0]
        assert r5["xyzw"][2] == 0                                   # z := 0 where z / 1000 is infinite
        if Q is Q_ZERO_W:
            assert np.isnan(r5["xyzw"][3]) and np.isinf(r5["xyzw"][0])


# ---- downloads -------------------------------------------------------------------------------------------------------
def stream_records(e, B, cap=None, stream=None):
    torch = _torch()
    out = None
    if cap is not None:
        out = (torch.full((B + 1,), -1, dtype=torch.int64, device="cuda:0"),
               torch.full((cap, 6), SENT, dtype=torch.float32, device="cuda:0"))
    offs, rec = e.download_obstacles_stream(B, out=out, stream=stream)
    if stream is not None:
        stream.synchronize()
    torch.cuda.synchronize()
    return offs.cpu().numpy(), rec.cpu().numpy()


def as_records(a):
    return np.ascontiguousarray(a, f32).view(api.OBSTACLE_DTYPE).reshape(-1)


def crafted_engine(e, B, seed):
    n = CW * CH
    rng = np.random.default_rng(seed)
    e.set_Q(Q_EDGE)
    e.set_mean_rois(one_pixel_rois())
    e.set_detection(rng.integers(-1, 2, n).astype(np.int32), rng.uniform(0, 100, (n, 2)).astype(f32), DIST_EDGE)
    maps = rng.choice(np.array([0, 17, 24, 31, 40], np.int16), (B, CH, CW))
    maps[1] = 0
    return maps


@pytest.mark.gpu
def test_host_and_stream_downloads():
    torch = _torch()
    B = 4
    with api.Engine(CW, CH, max_batch=B) as e:
        e.set_io_slots(2)
        m0 = crafted_engine(e, B, 1)
        m1 = np.flip(m0, 2).copy()
        e.debug_postfilter(m0, median=False, stages=api.STAGE_MEANS | api.STAGE_DETECT)
        e.debug_postfilter(m1, median=False, stages=api.STAGE_MEANS | api.STAGE_DETECT)
        for age, m in ((1, m0), (0, m1)):
            offs, recs = e.download_obstacles(B, age=age)
            s = torch.cuda.Stream()
            for st in (None, s):
                o_d, r_d = stream_records(e, B, stream=st) if age == 0 else (None, None)
                if age == 1:
                    o, r = e.download_obstacles_stream(B, age=1, stream=st)
                    torch.cuda.synchronize()
                    o_d, r_d = o.cpu().numpy(), r.cpu().numpy()
                assert np.array_equal(o_d, offs)
                same_records(as_records(r_d)[:offs[-1]], recs, "stream age %d" % age)
            assert offs[2] == offs[1]                          # frame 1: all zero, no hit
            # size query: NULL records give the offsets only
            o = np.full(B + 1, -1, np.int64)
            assert e._lib.mvsv_download_obstacles(e._ctx, age, o.ctypes.data, None, 0) == 0 and np.array_equal(o, offs)
            # a short host buffer: MVSV_ERR_INVALID with the offsets written
            short = np.zeros(max(int(offs[-1]) - 1, 0), api.OBSTACLE_DTYPE)
            o[:] = -1
            assert e._lib.mvsv_download_obstacles(e._ctx, age, o.ctypes.data, short.ctypes.data or 8, short.size) == ERR_INVALID
            assert np.array_equal(o, offs)


@pytest.mark.gpu
def test_stream_truncation():
    B = 4
    with api.Engine(CW, CH, max_batch=B) as e:
        maps = crafted_engine(e, B, 2)
        e.debug_postfilter(maps, median=False, stages=api.STAGE_MEANS | api.STAGE_DETECT)
        offs, recs = e.download_obstacles(B)
        total = int(offs[-1])
        assert total > 10
        for cap in (1, int(offs[1]), int(offs[1]) + 1, total - 1, total, total + 5):
            o, r = stream_records(e, B, cap=cap)
            assert np.array_equal(o, offs), cap                   # the offsets are always complete
            k = min(cap, total)
            same_records(as_records(r[:k]), recs[:k], "cap %d" % cap)
            assert (r[k:] == SENT).all(), cap                       # nothing past the capacity
        # NULL records: the offsets only
        torch = _torch()
        o = torch.full((B + 1,), -1, dtype=torch.int64, device="cuda:0")
        assert e._lib.mvsv_download_obstacles_stream(e._ctx, 0, o.data_ptr(), None, 0, None) == 0
        assert np.array_equal(o.cpu().numpy(), offs)


# ---- state and contract ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_state_and_contract():
    B = 2
    n = CW * CH
    det = np.zeros(n, np.int32)
    centers = np.zeros((n, 2), f32)
    maps = np.full((B, CH, CW), 24, np.int16)
    with api.Engine(CW, CH, max_batch=B) as e:
        lib, ctx = e._lib, e._ctx
        e.set_Q(Q_EDGE)
        e.set_mean_rois(one_pixel_rois())

        def post(stages):
            return lib.mvsv_debug_postfilter(ctx, maps.ctypes.data, maps.strides[1], B, 0, 0, 0, 0, stages)

        def obst():
            o = np.zeros(B + 1, np.int64)
            return lib.mvsv_download_obstacles(ctx, 0, o.ctypes.data, None, 0)

        assert post(api.STAGE_MEANS) == 0
        assert obst() == ERR_STATE                               # a compute without DETECT
        means0 = e.download(B, disp=False, means=True)["means"]
        assert post(api.STAGE_MEANS | api.STAGE_DETECT) == ERR_STATE       # no table
        e.set_detection(det, centers, DIST_EDGE)
        assert post(api.STAGE_DETECT) == ERR_INVALID                       # DETECT without MEANS
        # a table of the wrong length is refused and the one set before stays
        assert lib.mvsv_set_detection(ctx, det.ctypes.data, centers.ctypes.data, n - 1, DIST_EDGE.ctypes.data, 2) == ERR_STATE
        bad = det.copy()
        bad[3] = 2
        assert lib.mvsv_set_detection(ctx, bad.ctypes.data, centers.ctypes.data, n, DIST_EDGE.ctypes.data, 2) == ERR_INVALID
        assert lib.mvsv_set_detection(ctx, det.ctypes.data, centers.ctypes.data, n, DIST_EDGE.ctypes.data, 9) == ERR_INVALID
        # a rig without Q
        e.set_frame_rigs([0, 5])
        assert post(api.STAGE_MEANS | api.STAGE_DETECT) == ERR_STATE
        e.set_frame_rigs([])
        # every rejection left the first results downloadable
        assert np.array_equal(e.download(B, disp=False, means=True)["means"], means0)
        assert obst() == ERR_STATE
        assert post(api.STAGE_MEANS | api.STAGE_DETECT) == 0
        offs, _ = e.download_obstacles(B)
        assert offs[-1] == B * n
        # ROIs set again: the table and the obstacle lists are dropped
        e.set_mean_rois(one_pixel_rois())
        assert obst() == ERR_STATE
        assert post(api.STAGE_MEANS | api.STAGE_DETECT) == ERR_STATE
        assert e.download(B)["disp"].shape == (B, CH, CW)
        e.set_detection(det, centers, DIST_EDGE)
        assert post(api.STAGE_MEANS | api.STAGE_DETECT) == 0
        # a geometry change (rectification maps with a 60 x 4 display ROI) drops them too
        for cam in range(2):
            mx, my = cases.warp_maps(CH, CW, seed=cam)
            e.upload_rectify_maps(cam, mx, my, (0, 0, 60, 4))
        assert (e.info.width, e.info.height) == (60, 4)
        assert obst() == ERR_STATE
        e.set_mean_rois([(i % 60, i // 60, 1, 1) for i in range(240)])
        maps = np.full((B, 4, 60), 24, np.int16)
        assert post(api.STAGE_MEANS | api.STAGE_DETECT) == ERR_STATE
        e.set_detection(np.zeros(240, np.int32), np.zeros((240, 2), f32), DIST_EDGE)
        assert post(api.STAGE_MEANS | api.STAGE_DETECT) == 0
        assert e.download_obstacles(B)[0][-1] == B * 240


# ---- several engines ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("parts", [2, 3])
def test_multi_device(parts):
    """a ctx over two or three engines on one GPU gives the records and offsets of one engine, host and stream paths"""
    torch = _torch()
    B = 7
    L, R = td.frames(B, seed=8)
    got = []
    dists = None
    for devs in ([0], [0] * parts):
        with api.Engine(td.FW, td.FH, max_batch=B, devices=devs) as e:
            stages, _ = td.setup(e, "pipeline", B)
            W, H = e.info.width, e.info.height
            if dists is None:
                e.compute(L, R, stages)
                dists = dists_for(e.download(B, disp=False, means=True)["means"], cases.Q_REFERENCE)
            det, centers = table(W, H)
            e.set_detection(det, centers, dists)
            e.compute(L, R, stages | api.STAGE_DETECT)
            offs, recs = e.download_obstacles(B)
            s = torch.cuda.Stream()
            o_d, r_d = e.download_obstacles_stream(B, stream=s)
            s.synchronize()
            assert np.array_equal(o_d.cpu().numpy(), offs)
            same_records(as_records(r_d.cpu().numpy())[:offs[-1]], recs, "stream, %d parts" % len(devs))
            got.append((offs, recs))
    assert 0 < got[0][0][-1]
    assert np.array_equal(got[1][0], got[0][0])
    same_records(got[1][1], got[0][1], "%d parts against one" % parts)
