"""Eight stereo rigs at cfg 3 (remap + crop + configs/sgbm.yml SGBM with numDisp 64 + XYZ + sub-image and sample-point
means, 752x480 raw frames, inputs resident in device memory), three ways:
  (a) one engine, 8 rigs x 18 frames per step (mvsv_set_frame_rigs);
  (b) 8 engines of 18 frames, one per rig, submitted round-robin, each on its own stream;
  (c) one engine, one rig, 144 frames per step.
Reports ms per step, frames/s and the device memory each setup holds after its warm-up (the drop of cudaMemGetInfo's
free memory while it was created: on a shared card, another process's allocations would show up there too).  Each setup is timed with a host clock around
`steps` steps that end in a synchronise of every engine.  The setups alternate in `rounds` rounds.  Also checks that
(a) and (b) give the same disparities, XYZ and means.  The rigs are the three calibrations of tests/golden/calibrations.json,
used in turn, each with its display ROI cropped to 736x464 at a different offset.  Prints one JSON document that
includes the GPU name and power limit.
usage: python tools/rigs_time.py [steps] [rounds]"""
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
from mvstereovision3_b200 import api, synth  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 50
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 5
NRIGS, PER_RIG = 8, 18
B = NRIGS * PER_RIG
FW, FH = 752, 480
ROI_W, ROI_H = 736, 464
P = dict(bench.SGBM_YML, numDisp=64)
STAGES = api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_XYZ | api.STAGE_MEANS

with open(os.path.join(ROOT, "tests", "golden", "calibrations.json")) as f:
    CAL = json.load(f)["rigs"]
NAMES = sorted(CAL)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "nvidia-smi unavailable (%s)" % type(e).__name__
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def install(e, rig, k):
    """calibration k % 3 at ROI offset (2k, k) mod the room its display ROI leaves"""
    r = CAL[NAMES[k % len(NAMES)]]
    m = r["modes"]["full"]
    dx, dy, dw, dh = m["display_roi"]
    roi = (dx + (2 * k) % (dw - ROI_W + 1), dy + k % (dh - ROI_H + 1), ROI_W, ROI_H)
    for cam, (K, D, R, Pm) in enumerate(((r["KL"], r["DL"], m["R0"], m["P0"]), (r["KR"], r["DR"], m["R1"], m["P1"]))):
        e.set_rectification(cam, np.array(K), np.array(D), np.array(R), np.array(Pm), roi, rig=rig)
    e.set_Q(np.array(m["Q"], np.float32), rig=rig)


def engine(batch, rigs):
    """an engine for `batch` frames holding calibrations `rigs` as rigs 0.."""
    e = api.Engine(FW, FH, max_batch=batch)
    for rig, k in enumerate(rigs):
        install(e, rig, k)
    e.set_sgbm_params(**P)
    oW, oH = e.info.width, e.info.height
    off = api.dmap_roi_offset(P["numDisp"], oW)
    e.set_mean_rois(api.subimage_rois(oW - off, oH, off) + api.samplepoint_rois(oW - off, oH, off))
    return e


def used_bytes():
    torch.cuda.synchronize()
    free, total = torch.cuda.mem_get_info()
    return total - free


pairs = [synth.stereogram(FH, FW, P["minDisp"], P["numDisp"], seed=s)[:2] for s in range(16)]
dl = torch.from_numpy(np.stack([pairs[i % 16][0] for i in range(B)])).cuda()
dr = torch.from_numpy(np.stack([pairs[i % 16][1] for i in range(B)])).cuda()
fs = FH * FW


def step(engines):
    for eng, first, n in engines:            # round-robin submission: each engine's kernels run on its own stream
        eng.compute_device(dl.data_ptr() + first * fs, FW, dr.data_ptr() + first * fs, FW, fs, n, STAGES)


def sync(engines):
    for eng, _, _ in engines:
        eng.sync()


def add(name, engines, m0):
    """warm the setup up (the first compute allocates the XYZ buffers) and note the device memory it added"""
    for _ in range(3):
        step(engines)
    sync(engines)
    setups[name] = engines
    mem[name] = used_bytes() - m0


setups, mem = {}, {}
m0 = used_bytes()
ea = engine(B, range(NRIGS))
ea.set_frame_rigs([i // PER_RIG for i in range(B)])        # rig r holds frames 18r .. 18r+17
add("a_one_engine_8_rigs", [(ea, 0, B)], m0)
m0 = used_bytes()
add("b_8_engines", [(engine(PER_RIG, [r]), r * PER_RIG, PER_RIG) for r in range(NRIGS)], m0)   # engine r: rig r's frames
m0 = used_bytes()
add("c_one_engine_1_rig", [(engine(B, [0]), 0, B)], m0)

times = {k: [] for k in setups}
for _ in range(rounds):
    for k, engines in setups.items():
        sync(engines)
        t0 = time.perf_counter()
        for _ in range(steps):
            step(engines)
        sync(engines)
        times[k].append((time.perf_counter() - t0) * 1e3 / steps)

# (a) and (b) compute the same frames with the same calibrations
step(setups["a_one_engine_8_rigs"])
got_a = ea.download(B, xyz=True, means=True)
same = True
for eng, first, n in setups["b_8_engines"]:
    step([(eng, first, n)])
    got_b = eng.download(n, xyz=True, means=True)
    for key in ("disp", "xyz", "means"):
        same &= bool(np.array_equal(got_a[key][first:first + n].view(np.uint8), got_b[key].view(np.uint8)))

res = {"workload": "cfg3 with %d rigs: remap + crop to %dx%d + SGBM numDisp 64 + XYZ + %d ROI means, %dx%d raw frames, "
                   "device-resident inputs" % (NRIGS, ROI_W, ROI_H, ea.info.num_rois, FW, FH),
       "frames_per_step": B, "steps_per_round": steps, "rounds": rounds, "gpu": gpu_info(),
       "a_equals_b": same, "setups": {}}
for k in setups:
    med = float(np.median(times[k]))
    res["setups"][k] = {"ms_per_step": {"median": round(med, 4), "min": round(min(times[k]), 4), "max": round(max(times[k]), 4)},
                        "frames_per_s": round(B / (med * 1e-3), 1),
                        "device_bytes_held": int(mem[k]), "device_GB_held": round(mem[k] / 1e9, 2)}
print(json.dumps(res, indent=1))
for engines in setups.values():
    for eng, _, _ in engines:
        eng.close()
