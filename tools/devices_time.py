"""One engine over several devices (mvsv_init_devices) against one engine per device, at cfg 2 (SGBM, configs/sgbm.yml with
numDisp 64, 752x480) and cfg 3 (remap + crop to 736x464 + the same SGBM + XYZ + sub-image and sample-point means, two
rigs: the first two calibrations of tests/golden/calibrations.json, each rig holding half of the frames), 148 frames per
engine of one device:
  (a) one mvsv_init engine, batch 148;
  (b) mvsv_init_devices over every device, batch 148 x n; on a box of one GPU, over [0, 0] (two engines on device 0);
  (c) with n > 1 devices, one mvsv_init engine per device driven from one thread in a loop.
Each setup is timed two ways with a host clock around `steps` steps that end in a synchronise:
  device: compute_device on inputs resident on device 0 (other devices copy their share peer to peer);
  e2e: pinned host inputs and results, two I/O slots, compute k+1 submitted before the results of compute k are
       downloaded (age 1), as bench.py's end-to-end figure does.
The setups alternate in `rounds` rounds; the median is reported with the spread.  Also checks that (b) and (c) give
(a)'s disparities and means.  Prints one JSON document with the GPU name, power limit and device count.
usage: python tools/devices_time.py [steps] [rounds]"""
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

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 30
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
PER_GPU = 148
FW, FH = 752, 480
ROI_W, ROI_H = 736, 464
P = dict(bench.SGBM_YML, numDisp=64)
NDEV = torch.cuda.device_count()
if NDEV < 1:
    raise SystemExit("devices_time.py: no CUDA device")

with open(os.path.join(ROOT, "tests", "golden", "calibrations.json")) as f:
    CAL = json.load(f)["rigs"]
NAMES = sorted(CAL)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        q = ["nvidia-smi unavailable (%s)" % type(e).__name__]
    return {"device_count": NDEV, "torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def make_engine(cfg, batch, device=0, devices=None):
    e = api.Engine(FW, FH, max_batch=batch, device=device, devices=devices)
    stages, want = api.STAGE_SGBM, {}
    if cfg == "cfg3":
        for rig in range(2):
            r = CAL[NAMES[rig]]
            m = r["modes"]["full"]
            dx, dy, dw, dh = m["display_roi"]
            roi = (dx + (2 * rig) % (dw - ROI_W + 1), dy + rig % (dh - ROI_H + 1), ROI_W, ROI_H)
            for cam, (K, D, R, Pm) in enumerate(((r["KL"], r["DL"], m["R0"], m["P0"]), (r["KR"], r["DR"], m["R1"], m["P1"]))):
                e.set_rectification(cam, np.array(K), np.array(D), np.array(R), np.array(Pm), roi, rig=rig)
            e.set_Q(np.array(m["Q"], np.float32), rig=rig)
        stages = api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_XYZ | api.STAGE_MEANS
        want = dict(means=True)          # bench.py's e2e downloads: disparities and means (XYZ stays on the device)
    e.set_sgbm_params(**P)
    if cfg == "cfg3":
        oW, oH = e.info.width, e.info.height
        off = api.dmap_roi_offset(P["numDisp"], oW)
        e.set_mean_rois(api.subimage_rois(oW - off, oH, off) + api.samplepoint_rois(oW - off, oH, off))
    return e, stages, want


def rig_table(batch):
    """rig 0 holds the first half of every engine's frames, rig 1 the second"""
    return [(i % PER_GPU) * 2 // PER_GPU for i in range(batch)]


class Setup:
    """engines (engine, first frame, frames) driven together on one batch of `total` frames"""

    def __init__(self, cfg, total, engines):
        self.cfg, self.total, self.engines = cfg, total, engines
        for e, first, n in engines:
            if cfg == "cfg3":
                e[0].set_frame_rigs(rig_table(total)[first:first + n])

    def step_device(self, dl, dr):
        fs = FH * FW
        for (e, stages, _), first, n in self.engines:
            e.compute_device(dl.data_ptr() + first * fs, FW, dr.data_ptr() + first * fs, FW, fs, n, stages)

    def sync(self):
        for (e, _, _), _, _ in self.engines:
            e.sync()

    def e2e(self, hl, hr, out, nsteps):
        """the two-slot loop: submit k, then download k - 1 (age 1) into out[(k - 1) & 1]"""
        def submit():
            for (e, stages, _), first, n in self.engines:
                e.compute(hl.array[first:first + n], hr.array[first:first + n], stages)

        def collect(k, age):
            for (e, _, want), first, n in self.engines:
                o = out[k & 1]
                r = e.download(n, out={"disp": o["disp"].array[first:first + n]}, age=age, **want)
                for key in want:
                    o[key].array[first:first + n] = r[key]
        for (e, _, _), _, _ in self.engines:
            e.set_io_slots(2)
        submit()
        for k in range(1, nsteps):
            submit()
            collect(k - 1, 1)
        collect(nsteps - 1, 0)

    def close(self):
        for (e, _, _), _, _ in self.engines:
            e.close()


def measure(cfg, report):
    n_b = max(NDEV, 2)
    devs_b = list(range(NDEV)) if NDEV > 1 else [0, 0]
    total = PER_GPU * n_b
    pairs = [synth.stereogram(FH, FW, P["minDisp"], P["numDisp"], seed=s)[:2] for s in range(16)]
    hl, hr = api.pinned((total, FH, FW), np.uint8), api.pinned((total, FH, FW), np.uint8)
    for i in range(total):
        hl.array[i], hr.array[i] = pairs[i % 16]
    dl, dr = torch.from_numpy(hl.array).cuda(0), torch.from_numpy(hr.array).cuda(0)
    setups = {"a_one_engine": Setup(cfg, PER_GPU, [(make_engine(cfg, PER_GPU), 0, PER_GPU)]),
              "b_init_devices_%s" % "x".join(map(str, devs_b)):
                  Setup(cfg, total, [(make_engine(cfg, total, devices=devs_b), 0, total)])}
    if NDEV > 1:
        setups["c_engine_per_device_loop"] = Setup(cfg, total, [(make_engine(cfg, PER_GPU, device=d), d * PER_GPU, PER_GPU)
                                                                for d in range(NDEV)])
    e0 = setups["a_one_engine"].engines[0][0][0]
    oH, oW, nr = e0.info.height, e0.info.width, e0.info.num_rois
    outs = {}
    for name, s in setups.items():
        outs[name] = [dict(disp=api.pinned((s.total, oH, oW), np.int16),
                           **({"means": api.pinned((s.total, nr), np.float32)} if cfg == "cfg3" else {}))
                      for _ in range(2)]
        s.step_device(dl, dr)
        s.e2e(hl, hr, outs[name], 3)
        s.sync()
    times = {name: {"device": [], "e2e": []} for name in setups}
    for _ in range(rounds):
        for name, s in setups.items():
            s.sync()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                s.step_device(dl, dr)
            s.sync()
            times[name]["device"].append((time.perf_counter() - t0) * 1e3 / steps)
            t0 = time.perf_counter()
            s.e2e(hl, hr, outs[name], steps)
            s.sync()
            times[name]["e2e"].append((time.perf_counter() - t0) * 1e3 / steps)
    # every setup computed the same frames (frame i of a batch is pair i % 16): compare with (a) frame by frame
    ref = {k: v.array for k, v in outs["a_one_engine"][(steps - 1) & 1].items()}
    same = {}
    for name in setups:
        got = {k: v.array for k, v in outs[name][(steps - 1) & 1].items()}
        same[name] = all(np.array_equal(got[k][i].view(np.uint8), ref[k][i % PER_GPU].view(np.uint8))
                         for k in ref for i in range(got[k].shape[0]) if (i % PER_GPU) % 16 == i % 16)
    res = {"frames_per_engine_of_one_device": PER_GPU, "equal_to_a": same, "setups": {}}
    for name, s in setups.items():
        r = res["setups"][name] = {"frames_per_step": s.total}
        for how in ("device", "e2e"):
            t = times[name][how]
            med = float(np.median(t))
            r[how] = {"ms_per_step": {"median": round(med, 3), "min": round(min(t), 3), "max": round(max(t), 3)},
                      "frames_per_s": round(s.total / (med * 1e-3), 1)}
    report[cfg] = res
    for s in setups.values():
        s.close()
    for o in outs.values():
        for d in o:
            for b in d.values():
                b.close()
    hl.close()
    hr.close()
    del dl, dr
    torch.cuda.empty_cache()


report = {"gpu": gpu_info(), "steps_per_round": steps, "rounds": rounds,
          "not_measured": [] if NDEV > 1 else ["scaling over several physical GPUs (one GPU here: (b) runs over [0, 0], "
                                               "(c) needs two devices)", "device inputs copied peer to peer across GPUs"],
          "workloads": {"cfg2": "SGBM configs/sgbm.yml numDisp 64, 752x480",
                        "cfg3": "remap + crop to %dx%d (2 rigs) + cfg-2 SGBM + XYZ + ROI means, 752x480 raw" % (ROI_W, ROI_H)}}
for cfg in ("cfg2", "cfg3"):
    measure(cfg, report)
print(json.dumps(report, indent=1))
