"""Throughput of SGBM at disparity ranges above 256 (numDisp in (256, 512]) against D = 256 at the same size, with
device-resident inputs (CUDA events on the engine's stream around `steps` steps, after `warmup` steps):
  - 1920x1080 MODE_HH with the cfg 4 parameters (blockSize 5, P1 200, P2 800, LR check, speckle), D = 256 / 384 / 512,
    batch 14 as cfg 4;
  - 1280x720 MODE_SGBM with the configs/sgbm.yml wiring (minDisp 1, blockSize 13, speckle 150 / 2), D = 384 (S kept as
    bytes), batch 32.
For each: frames/s, evaluated cells/s (W1 * H * D * frames/s), the sweep's strip count and whether S was kept as bytes,
and the per-kernel split of one step (mvsv_profile_*, the kernels one after the other) in a separate pass.  Writes one
JSON document, which includes the GPU name and power limit, to `out` (default profiles/r07_wide_disp_time.json).
usage: python tools/wide_disp_time.py [steps] [warmup] [out]"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from mvstereovision3_b200 import api, synth  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
warmup = int(sys.argv[2]) if len(sys.argv) > 2 else 3
out_path = sys.argv[3] if len(sys.argv) > 3 else os.path.join(ROOT, "profiles", "r07_wide_disp_time.json")

CFG4 = dict(minDisp=0, blockSize=5, P1=200, P2=800, disp12MaxDiff=1, preFilterCap=0, uniquenessRatio=10,
            speckleWindowSize=150, speckleRange=2, disparityMode=1)
SGBM_YML = dict(minDisp=1, blockSize=13, P1=0, P2=0, disp12MaxDiff=0, preFilterCap=0, uniquenessRatio=0,
                speckleWindowSize=150, speckleRange=2, disparityMode=0)
RUNS = [("1080p_hh_d256", 1920, 1080, 14, dict(CFG4, numDisp=256)),
        ("1080p_hh_d384", 1920, 1080, 14, dict(CFG4, numDisp=384)),
        ("1080p_hh_d512", 1920, 1080, 14, dict(CFG4, numDisp=512)),
        ("720p_sgbm_yml_d384", 1280, 720, 32, dict(SGBM_YML, numDisp=384))]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "nvidia-smi unavailable (%s)" % type(e).__name__
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def measure(W, H, B, p):
    uniq = 4
    gen = [synth.stereogram(H, W, max(p["minDisp"], 0), p["numDisp"], seed=s)[:2] for s in range(uniq)]
    dl = torch.from_numpy(np.stack([gen[b % uniq][0] for b in range(B)])).cuda()
    dr = torch.from_numpy(np.stack([gen[b % uniq][1] for b in range(B)])).cuda()
    torch.cuda.synchronize()
    with api.Engine(W, H, max_batch=B) as e:
        e.set_sgbm_params(**p)

        def step():
            e.compute_device(dl.data_ptr(), W, dr.data_ptr(), W, H * W, B, api.STAGE_SGBM)

        for _ in range(warmup):
            step()
        e.sync()
        e.timer_start()
        for _ in range(steps):
            step()
        ms = e.timer_stop() / steps
        i = e.info
        # per-kernel split: a pass of its own (profiling runs the kernels one after the other)
        e.profile_enable(True)
        step()
        e.sync()
        e.profile_read()
        nprof = 2
        for _ in range(nprof):
            step()
        e.sync()
        split = {k: {"ms_per_step": round(v[0] / nprof, 3), "launches_per_step": v[1] / nprof}
                 for k, v in e.profile_read().items()}
        e.profile_enable(False)
        fps = B * 1e3 / ms
        return {"W": W, "H": H, "batch": B, "params": p, "W1": i.sgbm_W1, "D": i.sgbm_D, "Dpad": i.sgbm_Dpad,
                "sweep_strips": i.sgbm_td_cluster, "s8": i.sgbm_s8, "ms_per_step": round(ms, 3),
                "frames_per_s": round(fps, 1), "cells_per_s": float("%.4g" % (i.sgbm_W1 * H * i.sgbm_D * fps)),
                "kernels": split}


if not torch.cuda.is_available():
    sys.exit("wide_disp_time.py measures on a CUDA device; none is visible")
res = {"gpu": gpu_info(), "steps": steps, "warmup": warmup, "inputs": "device-resident", "runs": {}}
for name, W, H, B, p in RUNS:
    res["runs"][name] = measure(W, H, B, p)
    print(name, res["runs"][name]["frames_per_s"], "frames/s", res["runs"][name]["cells_per_s"], "cells/s", flush=True)
r = res["runs"]
res["cells_per_s_d512_over_d256_1080p"] = round(r["1080p_hh_d512"]["cells_per_s"] / r["1080p_hh_d256"]["cells_per_s"], 3)
res["cells_per_s_d384_over_d256_1080p"] = round(r["1080p_hh_d384"]["cells_per_s"] / r["1080p_hh_d256"]["cells_per_s"], 3)
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    json.dump(res, f, indent=1)
print(json.dumps(res, indent=1))
