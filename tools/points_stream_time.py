"""Point lists and min/max in device memory with no host wait, at cfg 3 with MVSV_STAGE_POINTS: remap + crop of 752x480
raw frames (parameters/baseline_small maps) + configs/sgbm.yml SGBM with numDisp 64 + 81 sub-image and sample-point
means + the point list, batch 148, inputs resident in device memory, two I/O slots, one torch stream.  Three loops,
alternated `reps` times in one run, each timed with the host clock between two device synchronisations for about
`seconds` seconds:
  (a) compute:  compute_device_stream only;
  (b) points_device: the same plus download_points_device(age=1) of the previous compute (offsets to the host first,
      which waits for that compute, then the point copy on the stream);
  (c) points_stream: the same plus download_points_stream(age=1) and download_minmax_device(age=1), no host wait.
For (b) and (c) also the host time spent inside the download calls per step.  In separate passes: k_points_out's time
from CUDA events around repeated download_points_stream calls on a finished compute, and from torch.profiler.  Checks
that (c)'s last results equal the host calls of the same compute.  Writes one JSON document, which includes the GPU name
and power limit, to `out` (default profiles/r09_points_stream_time.json) and prints it.
usage: python tools/points_stream_time.py [seconds] [reps] [out]"""
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
out_path = sys.argv[3] if len(sys.argv) > 3 else os.path.join(ROOT, "profiles", "r09_points_stream_time.json")
spec = bench.CONFIGS["cfg3_pipeline"]
p, FH, FW, B = spec["params"], spec["H"], spec["W"], 148
STAGES = api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_MEANS | api.STAGE_POINTS


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "nvidia-smi unavailable (%s)" % type(e).__name__
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


if not torch.cuda.is_available():
    sys.exit("points_stream_time.py measures on a CUDA device; none is visible")

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
e.set_Q(g["Q"])
W, H = e.info.width, e.info.height
off = api.dmap_roi_offset(p["numDisp"], W)
e.set_mean_rois(api.subimage_rois(W - off, H, off) + api.samplepoint_rois(W - off, H, off))
e.set_io_slots(2)
npx = B * H * W
s = torch.cuda.Stream()
# the outputs of every loop, allocated once: two of each, alternating between steps
pts = [torch.empty((npx, 3), dtype=torch.float32, device="cuda:0") for _ in range(2)]
offs = [torch.empty(B + 1, dtype=torch.int64, device="cuda:0") for _ in range(2)]
mms = [torch.empty((B, 2), dtype=torch.int16, device="cuda:0") for _ in range(2)]
torch.cuda.synchronize()
host_s = {"compute": 0.0, "points_device": 0.0, "points_stream": 0.0}


def fetch(name, age, k):
    if name == "points_device":
        e.download_points_device(B, age=age, out=pts[k & 1], stream=s)
    elif name == "points_stream":
        e.download_points_stream(B, age=age, out=(offs[k & 1], pts[k & 1]), stream=s)
        e.download_minmax_device(B, age=age, out=mms[k & 1], stream=s)


def loop(name, n):
    with torch.cuda.stream(s):
        e.compute_tensors(dl, dr, STAGES, stream=s)
        for k in range(1, n + 1):
            if k < n:
                e.compute_tensors(dl, dr, STAGES, stream=s)
            t0 = time.perf_counter()
            fetch(name, 1 if k < n else 0, k - 1)
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
                           "host_us_in_download_calls_per_step": round(host_s[name] * 1e6 / steps[name], 1)})

# (c)'s last step (age 0 of the last compute) against the host calls of the same compute
last = (steps["points_stream"] - 1) & 1
ho, hp = e.download_points(B)
total = int(ho[-1])
exact = bool(np.array_equal(offs[last].cpu().numpy(), ho)
             and np.array_equal(pts[last][:total].cpu().numpy().view(np.uint32), hp.view(np.uint32))
             and np.array_equal(mms[last].cpu().numpy(), e.download_minmax(B)))

# k_points_out alone: the compute has finished, so the calls queue nothing but the kernel behind the stream's events
ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
n_ev = 200
with torch.cuda.stream(s):
    for _ in range(10):
        e.download_points_stream(B, out=(offs[0], pts[0]), stream=s)
    ev[0].record(s)
    for _ in range(n_ev):
        e.download_points_stream(B, out=(offs[0], pts[0]), stream=s)
    ev[1].record(s)
s.synchronize()
events_ms = ev[0].elapsed_time(ev[1]) / n_ev
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    with torch.cuda.stream(s):
        for _ in range(50):
            e.download_points_stream(B, out=(offs[0], pts[0]), stream=s)
    s.synchronize()
kern = {}
for a in prof.key_averages():
    for kname in ("k_points_out", "k_minmax_fold"):
        if kname in a.key:
            t = getattr(a, "device_time_total", None) or getattr(a, "cuda_time_total", 0)
            kern[kname] = {"ms_per_call": round(t / 1e3 / max(a.count, 1), 4), "calls": a.count}
e.close()

best = {name: max(r["frames_per_s"] for r in v) for name, v in runs.items()}
moved = 2 * 12 * total + 2 * 8 * (B + 1)             # k_points_out reads and writes the list and the offsets
res = {"gpu": gpu_info(), "workload": "cfg3_pipeline + MVSV_STAGE_POINTS (rectify, SGBM, means, points; no XYZ), "
       "%dx%d raw frames, batch %d, device-resident inputs, two I/O slots, one torch stream" % (FW, FH, B),
       "seconds_per_timed_loop": seconds, "reps": reps,
       "timing": "host clock between two device synchronisations; loops alternate (compute, points_device, "
                 "points_stream) x reps; host_us_in_download_calls_per_step: host clock around the download calls only",
       "points_per_step": total, "valid_fraction": round(total / npx, 4), "runs": runs, "best_frames_per_s": best,
       "points_device_over_compute": round(best["points_device"] / best["compute"], 4),
       "points_stream_over_compute": round(best["points_stream"] / best["compute"], 4),
       "k_points_out_ms_cuda_events": round(events_ms, 4),
       "k_points_out_cuda_events_note": "events on the caller's stream around %d download_points_stream calls on a "
                                        "finished compute; includes the stream-to-stream event waits" % n_ev,
       "profiler_kernels": kern,
       "k_points_out_bytes": moved,
       "k_points_out_GB_per_s_from_events": round(moved / (events_ms * 1e-3) / 1e9, 1) if events_ms > 0 else None,
       "points_stream_equals_host_calls": exact}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    json.dump(res, f, indent=1)
print(json.dumps(res, indent=1))
