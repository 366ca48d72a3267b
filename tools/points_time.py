"""Cost of the point list (MVSV_STAGE_POINTS + mvsv_download_points) at cfg 3: remap + crop of 752x480 raw frames
(parameters/baseline_small maps) + configs/sgbm.yml SGBM with numDisp 64 + 81 sub-image and sample-point means, batch
148, against the dense XYZ a caller otherwise downloads and scans.  Measures, in one run:
  1. device-resident ms per step (inputs in device memory, CUDA events on the engine's stream) of the pipeline with
     XYZ, with POINTS, with both and with neither, alternated in `rounds` rounds of `steps` steps; then, in a separate
     profiled pass (torch.profiler, CUDA activities), the kernel times of k_points_count, k_points_scan and
     k_points_emit against k_xyz, with the bytes each kernel must move (from the shapes and the valid count) over its
     time;
  2. end to end with two I/O slots, host inputs in pinned memory, host clock around `steps` pipelined steps that end in
     a synchronise: (a) compute with XYZ, download disp + dense XYZ of the previous step into pinned buffers; the host
     selection xyz[disp > 0] timed separately; (b) compute with POINTS, mvsv_download_points of the previous step into
     a pinned buffer;
  3. the fraction of valid pixels (disparity > 0) of the frames used, overall and per frame (min / max).
Also checks that (a)'s selection and (b)'s list are identical.  Writes one JSON document, which includes the GPU name
and power limit, to `out` (default profiles/r06_points_time.json) and prints it.
usage: python tools/points_time.py [steps] [rounds] [out]"""
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

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 50
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 5
out_path = sys.argv[3] if len(sys.argv) > 3 else os.path.join(ROOT, "profiles", "r06_points_time.json")
spec = bench.CONFIGS["cfg3_pipeline"]
p, FH, FW, B = spec["params"], spec["H"], spec["W"], 148
BASE = api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_MEANS
VARIANTS = {"neither": BASE, "xyz": BASE | api.STAGE_XYZ, "points": BASE | api.STAGE_POINTS,
            "both": BASE | api.STAGE_XYZ | api.STAGE_POINTS}
PT_TILE = 2048                                        # csrc/filters.cu


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "nvidia-smi unavailable (%s)" % type(e).__name__
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


if not torch.cuda.is_available():
    sys.exit("points_time.py measures on a CUDA device; none is visible")

gen, uniq = bench.make_inputs(spec, list(range(B)), B)
hl, hr = api.pinned((B, FH, FW), np.uint8), api.pinned((B, FH, FW), np.uint8)
for i in range(B):
    hl.array[i], hr.array[i] = gen[i % uniq]
dl, dr = torch.from_numpy(hl.array).cuda(), torch.from_numpy(hr.array).cuda()

e = api.Engine(FW, FH, max_batch=B)
g, roi = bench.load_rectification()
e.upload_rectify_maps(0, g["m1x"], g["m1y"], roi)
e.upload_rectify_maps(1, g["m2x"], g["m2y"], roi)
e.set_sgbm_params(**p)
e.set_Q(g["Q"])
W, H = e.info.width, e.info.height
off = api.dmap_roi_offset(p["numDisp"], W)
e.set_mean_rois(api.subimage_rois(W - off, H, off) + api.samplepoint_rois(W - off, H, off))
npx = B * H * W


def step_device(stages):
    e.compute_device(dl.data_ptr(), FW, dr.data_ptr(), FW, FH * FW, B, stages)


# ---- 1. device-resident ms per step --------------------------------------------------------------------------------
for st in VARIANTS.values():
    for _ in range(3):
        step_device(st)
e.sync()
dev_ms = {k: [] for k in VARIANTS}
for _ in range(rounds):
    for k, st in VARIANTS.items():
        e.timer_start()
        for _ in range(steps):
            step_device(st)
        dev_ms[k].append(e.timer_stop() / steps)
offs, _ = e.download_points(B)
total = int(offs[-1])
per_frame = np.diff(offs) / (H * W)

# kernel times, profiled in a pass of their own
prof_steps = 10
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    for _ in range(prof_steps):
        step_device(VARIANTS["both"])
    e.sync()
    torch.cuda.synchronize()
kern = {}
for ev in prof.key_averages():
    for name in ("k_points_count", "k_points_scan", "k_points_emit", "k_xyz"):
        if name in ev.key and "rigs" not in ev.key:
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
            kern[name] = {"ms_per_step": round(t / 1e3 / prof_steps, 4), "launches_per_step": ev.count / prof_steps}
ntiles = B * -(-H * W // PT_TILE)
bytes_moved = {                                      # what each kernel must read and write at this valid count
    "k_points_count": 2 * npx + 8 * ntiles,
    "k_points_scan": 2 * 8 * ntiles + 8 * (B + 1),
    "k_points_emit": 2 * npx + 8 * ntiles + 12 * total,
    "k_xyz": 2 * npx + 12 * npx,
}
for k, v in kern.items():
    v["bytes"] = int(bytes_moved[k])
    v["GB_per_s"] = round(bytes_moved[k] / (v["ms_per_step"] * 1e-3) / 1e9, 1) if v["ms_per_step"] > 0 else None

# ---- 2. end to end, two I/O slots ----------------------------------------------------------------------------------
e.set_io_slots(2)
hd = api.pinned((B, H, W), np.int16)
hx = api.pinned((B, H, W, 3), np.float32)
hp = api.pinned((npx, 3), np.float32)
lib, ctx = e._lib, e._ctx


def dl_dense(age):
    rc = lib.mvsv_download_age(ctx, age, hd.ptr, W * 2, None, None, 0, hx.ptr, None)
    assert rc == 0, rc


def run_e2e(stages, fetch):
    e.compute(hl.array, hr.array, stages)
    for _ in range(2):
        e.compute(hl.array, hr.array, stages)
        fetch(1)
    e.sync()
    ms = []
    for _ in range(rounds):
        t0 = time.perf_counter()
        for _ in range(steps):
            e.compute(hl.array, hr.array, stages)
            fetch(1)
        e.sync()
        ms.append((time.perf_counter() - t0) * 1e3 / steps)
    return ms


e2e = {}
e2e["a_dense_disp_xyz"] = run_e2e(VARIANTS["xyz"], dl_dense)
sel_ms = []
for _ in range(5):
    t0 = time.perf_counter()
    sel = hx.array.reshape(-1, 3)[hd.array.ravel() > 0]
    sel_ms.append((time.perf_counter() - t0) * 1e3)
e2e["b_download_points"] = run_e2e(VARIANTS["points"], lambda age: e.download_points(B, age=age, out=hp.array))
b_offs, b_pts = e.download_points(B, age=1, out=hp.array)
same = bool(np.array_equal(b_pts.view(np.uint32), sel.view(np.uint32))) and int(b_offs[-1]) == total

med = lambda v: round(float(np.median(v)), 4)
rng = lambda v: [round(min(v), 4), round(max(v), 4)]
res = {
    "workload": "cfg3: remap + crop to %dx%d + SGBM numDisp 64 + %d ROI means, %dx%d raw frames, batch %d" % (
        W, H, e.info.num_rois, FW, FH, B),
    "gpu": gpu_info(), "steps_per_round": steps, "rounds": rounds,
    "device_resident_ms_per_step": {k: {"median": med(v), "min_max": rng(v)} for k, v in dev_ms.items()},
    "kernels_profiled": kern,
    "end_to_end_two_io_slots_ms_per_step": {k: {"median": med(v), "min_max": rng(v)} for k, v in e2e.items()},
    "host_selection_xyz_disp_gt_0_ms": {"median": med(sel_ms), "min_max": rng(sel_ms)},
    "download_bytes_per_step": {"a_dense_disp_xyz": 14 * npx, "b_points": 12 * total + 8 * (B + 1)},
    "valid_pixels": {"total": total, "pixels": npx, "fraction": round(total / npx, 4),
                     "per_frame_min": round(float(per_frame.min()), 4), "per_frame_max": round(float(per_frame.max()), 4)},
    "points_equal_host_selection": same,
}
txt = json.dumps(res, indent=1)
print(txt)
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    f.write(txt + "\n")
e.close()
for b in (hl, hr, hd, hx, hp):
    b.close()
