"""Cost of StereoBM's post-filters at cfg 1 (configs/bm.yml, 752x480, batch 148, bench.py's cfg1_bm inputs resident in
device memory): ms per step with the filters off and with OpenCV's stereo_match filters (disp12MaxDiff 1, speckle
window 100, range 32), measured with CUDA events on the engine's stream, the two settings alternating in rounds; then
one profiled step of each for the per-kernel times.  Prints one JSON document (GPU name and power limit included).
usage: python tools/bm_filters_time.py [steps] [rounds]"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import bench  # noqa: E402
from mvstereovision3_b200 import api  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 50
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 5
spec = bench.CONFIGS["cfg1_bm"]
p, H, W, B = spec["params"], spec["H"], spec["W"], spec["batch"]
gen, uniq = bench.make_inputs(spec, list(range(B)), B)
dl = torch.from_numpy(np.stack([gen[i % uniq][0] for i in range(B)])).cuda()
dr = torch.from_numpy(np.stack([gen[i % uniq][1] for i in range(B)])).cuda()
SETTINGS = {"off": (-1, 0, 0), "stereo_match": (1, 100, 32)}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "nvidia-smi unavailable (%s)" % type(e).__name__
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


with api.Engine(W, H, max_batch=B) as e:
    e.set_bm_params(**p)

    def step():
        e.compute_device(dl.data_ptr(), W, dr.data_ptr(), W, H * W, B, api.STAGE_BM)

    times = {k: [] for k in SETTINGS}
    for k, f in SETTINGS.items():              # warm-up of both settings
        e.set_bm_filters(*f)
        for _ in range(3):
            step()
        e.sync()
    for _ in range(rounds):
        for k, f in SETTINGS.items():
            e.set_bm_filters(*f)
            step()
            e.sync()
            e.timer_start()
            for _ in range(steps):
                step()
            times[k].append(e.timer_stop() / steps)
    kernels = {}
    for k, f in SETTINGS.items():
        e.set_bm_filters(*f)
        step()
        e.sync()
        e.profile_enable(True)
        step()
        e.sync()
        kernels[k] = {n: round(v[0], 4) for n, v in sorted(e.profile_read().items(), key=lambda kv: -kv[1][0])}
        e.profile_enable(False)

res = {"config": spec["name"], "batch": B, "steps_per_round": steps, "rounds": rounds, "gpu": gpu_info(),
       "filters": {k: dict(zip(("disp12MaxDiff", "speckleWindowSize", "speckleRange"), f)) for k, f in SETTINGS.items()},
       "ms_per_step": {k: {"median": round(float(np.median(v)), 4), "min": round(min(v), 4), "max": round(max(v), 4)}
                       for k, v in times.items()},
       "kernel_ms_one_profiled_step": kernels}
res["filter_cost_ms_per_step"] = round(res["ms_per_step"]["stereo_match"]["median"] - res["ms_per_step"]["off"]["median"], 4)
print(json.dumps(res, indent=1))
