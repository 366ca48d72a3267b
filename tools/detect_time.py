"""Obstacle detection on the device (MVSV_STAGE_DETECT) at cfg 3: remap + crop of 752x480 raw frames
(parameters/baseline_small maps) + configs/sgbm.yml SGBM with numDisp 64 + XYZ + the means of the 81 sub-images and the
sample points, batch 148, inputs resident in device memory, two I/O slots, one torch stream.  Three loops, alternated
`reps` times in one run, each timed with the host clock between two device synchronisations for about `seconds` seconds:
  (a) compute:      compute_device_stream with MEANS, nothing fetched;
  (b) host_detect:  the same plus the host path of the previous compute: its means to host memory (mvsv_download_age,
                    which waits for that compute), then the range test and calcCoordinate of the hits on the host (a
                    vectorised numpy restatement of the two host detectors);
  (c) device_detect: compute with MEANS + DETECT plus download_obstacles_stream(age=1), no host wait.
For (b) and (c) also the host time per step spent in the fetch.  In a separate pass the per-kernel CUDA-event timing of the
engine (mvsv_profile_read) gives the stage's three kernels ("detect") against the means kernel.  Checks that (c)'s last
records equal mvsv_download_obstacles of the same compute.  Writes one JSON document, with the GPU name and power limit, to
`out` (default profiles/r10_detect_time.json) and prints it.
usage: python tools/detect_time.py [seconds] [reps] [out]"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import bench  # noqa: E402
from mvstereovision3_b200 import api  # noqa: E402

seconds = float(sys.argv[1]) if len(sys.argv) > 1 else 3.0
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 2
out_path = sys.argv[3] if len(sys.argv) > 3 else os.path.join(ROOT, "profiles", "r10_detect_time.json")
spec = bench.CONFIGS["cfg3_pipeline"]
p, FH, FW, B = spec["params"], spec["H"], spec["W"], 148
BASE = api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_XYZ | api.STAGE_MEANS
DISTS = np.array([[0.3, 1.5], [0.3, 1.5]], np.float32)     # min / max distance of both detectors, metres


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "nvidia-smi unavailable (%s)" % type(e).__name__
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


if not torch.cuda.is_available():
    sys.exit("detect_time.py measures on a CUDA device; none is visible")

gen, uniq = bench.make_inputs(spec, list(range(B)), B)
hl, hr = np.empty((B, FH, FW), np.uint8), np.empty((B, FH, FW), np.uint8)
for i in range(B):
    hl[i], hr[i] = gen[i % uniq]
dl, dr = torch.from_numpy(hl).cuda(), torch.from_numpy(hr).cuda()

e = api.Engine(FW, FH, max_batch=B)
g, roi = bench.load_rectification()
e.upload_rectify_maps(0, g["m1x"], g["m1y"], roi)
e.upload_rectify_maps(1, g["m2x"], g["m2y"], roi)
e.set_sgbm_params(**p)
Q = np.asarray(g["Q"], np.float32).reshape(4, 4)
e.set_Q(Q)
W, H = e.info.width, e.info.height
off = api.dmap_roi_offset(p["numDisp"], W)
subs, sps = api.subimage_rois(W - off, H, off), api.samplepoint_rois(W - off, H, off)
e.set_mean_rois(subs + sps)
n = len(subs) + len(sps)
det = np.array([0] * len(subs) + [1] * len(sps), np.int32)
centers = np.array([(x - off + w // 2, y + h // 2) for x, y, w, h in subs] + [(x - off + 2, y + 2) for x, y, _, _ in sps],
                   np.float32)
e.set_detection(det, centers, DISTS)
e.set_io_slots(2)
s = torch.cuda.Stream()

# the host path's detectors, vectorised: ranges of calcDMapValues, then calcCoordinate of the hits
z = DISTS.astype(np.float32) * np.float32(1000)
rng = (np.float32(Q[2, 3]) - z * np.float32(Q[3, 3])) / (z * np.float32(Q[3, 2])) * np.float32(16)
first, second = rng[det, 0], rng[det, 1]
Q64 = Q.astype(np.float64)
means_pinned = api.pinned((B, n), np.float32)      # kept alive: the buffer is freed with it
means_h = means_pinned.array


def host_detect(means):
    hit = (means < first) & (means > second)
    f, i = np.nonzero(hit)
    v = means[f, i]
    inp = np.stack([centers[i, 0], centers[i, 1], v / np.float32(16), np.ones_like(v)], 1).astype(np.float64)
    c = (inp @ Q64.T).astype(np.float32)
    xyzw = (c.astype(np.float64) * (1.0 / c[:, 3:4].astype(np.float64))).astype(np.float32)
    return f, i, xyzw


offs = [torch.empty(B + 1, dtype=torch.int64, device="cuda:0") for _ in range(2)]
recs = [torch.empty((B * n, 6), dtype=torch.float32, device="cuda:0") for _ in range(2)]
torch.cuda.synchronize()
host_s = {"compute": 0.0, "host_detect": 0.0, "device_detect": 0.0}


def fetch(name, age, k):
    if name == "host_detect":
        e._ck(e._lib.mvsv_download_age(e._ctx, age, None, 0, None, None, 0, None, means_h.ctypes.data))
        host_detect(means_h)
    elif name == "device_detect":
        e.download_obstacles_stream(B, age=age, out=(offs[k & 1], recs[k & 1]), stream=s)


def loop(name, steps):
    stages = BASE | (api.STAGE_DETECT if name == "device_detect" else 0)
    with torch.cuda.stream(s):
        e.compute_tensors(dl, dr, stages, stream=s)
        for k in range(1, steps + 1):
            if k < steps:
                e.compute_tensors(dl, dr, stages, stream=s)
            t0 = time.perf_counter()
            fetch(name, 1 if k < steps else 0, k - 1)
            host_s[name] += time.perf_counter() - t0
    s.synchronize()


names = list(host_s)
steps = {}
for name in names:                                   # warm-up, then a short pass sizes the timed window
    loop(name, 5)
    t0 = time.perf_counter()
    loop(name, 10)
    steps[name] = max(10, int(seconds / ((time.perf_counter() - t0) / 10)))
runs = {name: [] for name in names}
for _ in range(reps):
    for name in names:
        torch.cuda.synchronize()
        host_s[name] = 0.0
        t0 = time.perf_counter()
        loop(name, steps[name])
        dt = time.perf_counter() - t0
        runs[name].append({"steps": steps[name], "seconds": round(dt, 3), "ms_per_step": round(dt * 1e3 / steps[name], 4),
                           "frames_per_s": round(B * steps[name] / dt, 1),
                           "host_us_in_fetch_per_step": round(host_s[name] * 1e6 / steps[name], 1)})

# (c)'s last step (age 0 of the last compute) against the host download of the same compute
last = (steps["device_detect"] - 1) & 1
ho, hrec = e.download_obstacles(B)
total = int(ho[-1])
got = recs[last][:total].cpu().numpy()
exact = bool(np.array_equal(offs[last].cpu().numpy(), ho)
             and np.array_equal(np.ascontiguousarray(got).view(np.uint8).ravel(), hrec.view(np.uint8).ravel()))
# the host path finds the same hits
e._ck(e._lib.mvsv_download_age(e._ctx, 0, None, 0, None, None, 0, None, means_h.ctypes.data))
hf, hi, _ = host_detect(means_h)
same_hits = bool(np.array_equal(hi, hrec["roi"]) and np.array_equal(np.bincount(hf, minlength=B), np.diff(ho)))

# per-kernel CUDA events of the engine: the stage's three kernels against the means kernel
n_prof = 50
e.set_io_slots(1)
e.profile_enable(True)
with torch.cuda.stream(s):
    for _ in range(5):
        e.compute_tensors(dl, dr, BASE | api.STAGE_DETECT, stream=s)
    e.profile_read()
    for _ in range(n_prof):
        e.compute_tensors(dl, dr, BASE | api.STAGE_DETECT, stream=s)
prof = e.profile_read()
e.profile_enable(False)
e.close()

best = {name: max(r["frames_per_s"] for r in v) for name, v in runs.items()}
kern = {k: {"ms_per_compute": round(v[0] / n_prof, 4), "launches_per_compute": v[1] // n_prof}
        for k, v in prof.items() if k in ("detect", "means")}
res = {"gpu": gpu_info(),
       "workload": "cfg3_pipeline (rectify, SGBM, XYZ, means of %d ROIs: 81 sub-images + %d sample points) %dx%d raw "
                   "frames, batch %d, device-resident inputs, two I/O slots, one torch stream; both detectors at "
                   "%.1f-%.1f m" % (n, len(sps), FW, FH, B, DISTS[0, 0], DISTS[0, 1]),
       "seconds_per_timed_loop": seconds, "reps": reps,
       "timing": "host clock between two device synchronisations; loops alternate (compute, host_detect, device_detect) "
                 "x reps; host_us_in_fetch_per_step: host clock around the fetch only (host_detect: means download, "
                 "which waits for the compute, plus the numpy detectors; device_detect: download_obstacles_stream)",
       "obstacles_per_step": total, "runs": runs, "best_frames_per_s": best,
       "host_detect_over_compute": round(best["host_detect"] / best["compute"], 4),
       "device_detect_over_compute": round(best["device_detect"] / best["compute"], 4),
       "kernels_cuda_events": kern,
       "kernels_note": "mvsv_profile_read over %d computes with per-kernel timing on (kernels serialised); 'detect' is "
                       "k_detect_count + k_points_scan + k_detect_emit" % n_prof,
       "device_records_equal_host_download": exact, "host_detectors_find_the_same_hits": same_hits}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    json.dump(res, f, indent=1)
print(json.dumps(res, indent=1))
