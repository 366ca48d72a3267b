"""Throughput of three loops over the bench.py configurations cfg 1 (StereoBM, configs/bm.yml) and cfg 2 (StereoSGBM,
configs/sgbm.yml at numDisp 64), 752x480 at batch 148, all measured in one run:
  (a) device:   compute_device only, the inputs resident in device memory (bench.py's HBM-resident figure);
  (b) device_io: compute_device_stream plus download_device of the disparities into torch tensors, two I/O slots, one
      torch stream, no host wait inside the loop (compute k+1, then the age-1 download of compute k);
  (c) host:     pinned host inputs and a host download of the disparities, two I/O slots (bench.py's end to end).
Every loop is warmed up, then timed with the host clock between two device synchronisations for about `seconds`
seconds; the three loops alternate, `reps` times each.  Also checks that the last step of (b) equals the host download.
Writes one JSON document, which includes the GPU name and power limit, to `out` (default
profiles/r08_device_io_time.json).
usage: python tools/device_io_time.py [seconds] [reps] [out]"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from mvstereovision3_b200 import api, synth  # noqa: E402

seconds = float(sys.argv[1]) if len(sys.argv) > 1 else 3.0
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 2
out_path = sys.argv[3] if len(sys.argv) > 3 else os.path.join(ROOT, "profiles", "r08_device_io_time.json")

SGBM_YML = dict(minDisp=1, blockSize=13, disp12MaxDiff=0, preFilterCap=0, uniquenessRatio=0, speckleWindowSize=150,
                speckleRange=2, disparityMode=0, P1=0, P2=0)
CONFIGS = [("cfg1_bm", "bm", dict(numDisp=80, blockSize=21, preFilterCap=2, textureThreshold=30, uniquenessRatio=0)),
           ("cfg2", "sgbm", dict(SGBM_YML, numDisp=64))]
W, H, B = 752, 480, 148


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = "nvidia-smi unavailable (%s)" % type(e).__name__
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def measure(kind, p):
    uniq = 16
    gen = [synth.stereogram(H, W, p.get("minDisp", 0), p["numDisp"], seed=s)[:2] for s in range(uniq)]
    hl, hr = api.pinned((B, H, W), np.uint8), api.pinned((B, H, W), np.uint8)
    for i in range(B):
        hl.array[i], hr.array[i] = gen[i % uniq]
    dl, dr = torch.from_numpy(hl.array).cuda(), torch.from_numpy(hr.array).cuda()
    hd = [api.pinned((B, H, W), np.int16) for _ in range(2)]
    td = [torch.empty((B, H, W), dtype=torch.int16, device="cuda:0") for _ in range(2)]
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    e = api.Engine(W, H, max_batch=B)
    if kind == "bm":
        e.set_bm_params(**p)
        stages = api.STAGE_BM
    else:
        e.set_sgbm_params(**p)
        stages = api.STAGE_SGBM
    e.set_io_slots(2)

    def loop_device(n):
        for _ in range(n):
            e.compute_device(dl.data_ptr(), W, dr.data_ptr(), W, H * W, B, stages)
        e.sync()

    def loop_device_io(n):
        with torch.cuda.stream(s):
            e.compute_tensors(dl, dr, stages, stream=s)
            for k in range(1, n):
                e.compute_tensors(dl, dr, stages, stream=s)
                e.download_device(B, age=1, out={"disp": td[(k - 1) & 1]}, stream=s)
            e.download_device(B, age=0, out={"disp": td[(n - 1) & 1]}, stream=s)
        s.synchronize()

    def loop_host(n):
        e.compute(hl.array, hr.array, stages)
        for k in range(1, n):
            e.compute(hl.array, hr.array, stages)
            e.download(B, age=1, out={"disp": hd[(k - 1) & 1].array})
        e.download(B, age=0, out={"disp": hd[(n - 1) & 1].array})

    loops = {"device": loop_device, "device_io": loop_device_io, "host": loop_host}
    steps = {}
    for name, f in loops.items():                    # warm-up, then a short pass sizes the timed window
        f(5)
        t0 = time.perf_counter()
        f(10)
        steps[name] = max(10, int(seconds / ((time.perf_counter() - t0) / 10)))
    runs = {name: [] for name in loops}
    for _ in range(reps):
        for name, f in loops.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f(steps[name])
            dt = time.perf_counter() - t0
            runs[name].append({"steps": steps[name], "seconds": round(dt, 3), "ms_per_step": round(dt * 1e3 / steps[name], 4),
                               "frames_per_s": round(B * steps[name] / dt, 1)})
    # the device download of the last step equals the host download of the same compute
    loop_device_io(2)
    ref = e.download(B, age=0)["disp"]
    exact = bool(np.array_equal(td[1].cpu().numpy(), ref))
    e.close()
    for b in (hl, hr, hd[0], hd[1]):
        b.close()
    best = {name: max(r["frames_per_s"] for r in v) for name, v in runs.items()}
    return {"W": W, "H": H, "batch": B, "kind": kind, "params": p, "runs": runs, "best_frames_per_s": best,
            "device_io_over_device": round(best["device_io"] / best["device"], 4),
            "host_over_device": round(best["host"] / best["device"], 4),
            "device_download_bytes_per_step": 2 * B * H * W, "device_io_equals_host_download": exact}


if not torch.cuda.is_available():
    sys.exit("device_io_time.py measures on a CUDA device; none is visible")
res = {"gpu": gpu_info(), "seconds_per_timed_loop": seconds, "reps": reps,
       "timing": "host clock between two device synchronisations; loops alternate (device, device_io, host) x reps",
       "configs": {}}
for name, kind, p in CONFIGS:
    res["configs"][name] = measure(kind, p)
    r = res["configs"][name]
    print(name, r["best_frames_per_s"], "device_io/device", r["device_io_over_device"], flush=True)
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w") as f:
    json.dump(res, f, indent=1)
print(json.dumps(res, indent=1))
