#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric (SGBM frames/s and Gdisp-evals/s) on BASELINE.json's config 2:
StereoSGBM MODE_SGBM (5 paths), reference configs/sgbm.yml wiring with numDisp 64, 752x480, synthetic random-dot
stereograms with a disparity ramp.  The other BASELINE.json configurations (cfg 1 StereoBM, sgbm.yml as shipped,
cfg 3 full pipeline, cfg 4 MODE_HH 1080p D=256, cfg 5 4K D=256) are measured in the same run and reported in the
`configs` block of the same JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--configs LIST|none]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path (mvsv_compute: prefilter -> BT cost -> box sums -> 5 path scans -> WTA/LR ->
median -> speckle) over one batch of B stereo pairs per GPU; every configuration runs K timed steps.  With
--dump-outputs, rank 0 writes what the last HBM-resident step of each configuration returns to a caller (disparities;
for cfg 3 also the ROI means) as DIR/<config>_<array>.npy in float32, so that two builds can be compared output for
output: the inputs are seeded, the same from run to run.  `value` times K steps with inputs resident in HBM
(CUDA events on the engine's stream); `e2e` times the same K steps through the host-facing C-ABI call with pinned
HOST buffers, host->device and device->host copies inside the timed region, pipelined inside ONE engine over two
I/O slots (mvsv_set_io_slots).  For N > 1 the script runs under torchrun, one rank per GPU; frames are
round-robined over ranks (no data-path collective) and the time is the max over ranks.  `--impl reference` times
the reference's own CPU implementation of the path (OpenCV's StereoSGBM through cv2 4.13.0 -- the library call
reference src/disparity.cpp:8 makes) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from mvstereovision3_b200 import shard, synth  # noqa: E402

SGBM_YML = dict(minDisp=1, blockSize=13, disp12MaxDiff=0, preFilterCap=0, uniquenessRatio=0, speckleWindowSize=150,
                speckleRange=2, disparityMode=0, P1=0, P2=0)      # reference configs/sgbm.yml, P1/P2 never set
CFG4_PARAMS = dict(minDisp=0, numDisp=256, blockSize=5, disp12MaxDiff=1, preFilterCap=0, uniquenessRatio=10,
                   speckleWindowSize=150, speckleRange=2, disparityMode=1, P1=200, P2=800)

# BASELINE.json configs; `model_bpc` = algorithmic HBM bytes per evaluated cell of SURVEY.md 8(d)'s roofline model
CONFIGS = {
    "cfg2": dict(name="cfg2: StereoSGBM MODE_SGBM 5-path, configs/sgbm.yml (numDisp=64), 752x480", kind="sgbm",
                 H=480, W=752, params=dict(SGBM_YML, numDisp=64), batch=148, model_bpc=8.0),
    "cfg1_bm": dict(name="cfg1: StereoBM configs/bm.yml (numDisp=80, blockSize=21), 752x480", kind="bm", H=480, W=752,
                    params=dict(numDisp=80, blockSize=21, preFilterCap=2, textureThreshold=30, uniquenessRatio=0),
                    batch=148, model_bpc=4.0),
    "sgbm_yml_d128": dict(name="configs/sgbm.yml as shipped (numDisp=128), 752x480", kind="sgbm", H=480, W=752,
                          params=dict(SGBM_YML, numDisp=128), batch=74, model_bpc=8.0),
    "cfg3_pipeline": dict(name="cfg3: remap (parameters/baseline_small maps) + crop + cfg-2 SGBM + XYZ + 81 sub-image and "
                               "5x5 sample-point means, 752x480 raw frames", kind="pipeline", H=480, W=752,
                          params=dict(SGBM_YML, numDisp=64), batch=148, model_bpc=8.0),
    "cfg4_hh_1080p_d256": dict(name="cfg4: StereoSGBM MODE_HH 8-path 1920x1080 numDisp=256 blockSize=5 P1=200 P2=800, "
                                    "LR check + speckle", kind="sgbm", H=1080, W=1920, params=CFG4_PARAMS, batch=14,
                               model_bpc=14.0),
    "cfg5_4k_d256": dict(name="cfg5: StereoSGBM MODE_SGBM 3840x2160 numDisp=256 blockSize=5 P1=200 P2=800", kind="sgbm",
                         H=2160, W=3840, params=dict(CFG4_PARAMS, disparityMode=0, uniquenessRatio=0, disp12MaxDiff=0,
                                                     speckleWindowSize=0, speckleRange=0), batch=9, model_bpc=8.0),
}
HEADLINE = "cfg2"

# algorithmic HBM bytes per evaluated cell (x, y, d) of each aggregation-stage kernel in the current pipeline
# (int16 volumes; images, maps and per-pixel outputs are < 1 % and ignored) -- see DESIGN.md "Kernels"
KERNEL_BYTES_PER_CELL = {"sgbm_vsum": 2.0, "sgbm_h1": 6.0, "sgbm_td": 6.0, "sgbm_vdir": 6.0, "sgbm_h2_wta": 4.0,
                         "bm_colsum": 2.0, "bm_wta": 2.0}
# the same when the aggregated volume S is kept as one byte per cell (mvsv_info.sgbm_s8: npaths * P2 <= 255)
KERNEL_BYTES_PER_CELL_S8 = dict(KERNEL_BYTES_PER_CELL, sgbm_h1=5.0, sgbm_td=4.0, sgbm_h2_wta=3.0)
NCU_SUMMARY = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
# --dump-outputs: at most this many values per array (8 MiB of float32), so that the seven arrays of a run with every
# configuration stay under 64 MB
DUMP_VALUES_PER_ARRAY = 1 << 21


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_summary():
    """Per-kernel figures of the committed `ncu --set full` capture of the headline workload: DRAM bytes and
    ALU-pipe lane operations per evaluated cell ({} when the summary is absent)."""
    try:
        with open(NCU_SUMMARY) as f:
            return json.load(f)
    except Exception:
        return {}


def int_pipe_peak():
    """Measured issue peak of the packed 16x2 integer instructions the path is made of (tools/dpx_peak.cu,
    profiles/r01_dpx_issue_peak.txt): 2.0 warp instructions per clock per SM = 18.2 T lane-ops/s at 1965 MHz."""
    return 2.0 * 32 * 148 * 1.965e9, "measured (profiles/r01_dpx_issue_peak.txt: 2.0 warp-instr/clk/SM at 1965 MHz)"


def bind_to_gpu_numa_node(local_rank):
    """Run this rank (and allocate its pinned host buffers) on the CPUs next to its GPU, so that host<->device copies
    of different ranks do not cross sockets.  Sources, in order: the GPU's sysfs numa_node; `nvidia-smi topo -m`'s CPU
    affinity column.  Returns a description of what was done (it is reported in the JSON line)."""
    def apply(cpus, how):
        allowed = set(cpus) & os.sched_getaffinity(0)
        if not allowed:
            return "not bound: %s lists no allowed cpu" % how
        os.sched_setaffinity(0, allowed)
        return "bound to %d cpus (%s)" % (len(allowed), how)

    def parse_cpulist(txt):
        cpus = set()
        for part in txt.strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        return cpus

    tried = []
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id,
                                                                   getattr(pr, "pci_device_id", 0))
        node = int(open(path).read().strip())
        if node >= 0:
            return apply(parse_cpulist(open("/sys/devices/system/node/node%d/cpulist" % node).read()), "sysfs numa node %d" % node)
        tried.append("sysfs numa_node=-1")
    except Exception as e:
        tried.append("sysfs: %s" % type(e).__name__)
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        lines = [ln for ln in out.splitlines() if ln.strip()]
        hdr = lines[0].split("\t")
        col = next(i for i, h in enumerate(hdr) if "CPU Affinity" in h)
        row = next(ln for ln in lines[1:] if ln.split("\t")[0].strip() == "GPU%d" % local_rank).split("\t")
        aff = row[col].strip()
        if aff and aff[0].isdigit():
            return apply(parse_cpulist(aff), "nvidia-smi topo CPU affinity %s" % aff)
        tried.append("nvidia-smi topo: no affinity column value")
    except Exception as e:
        tried.append("nvidia-smi topo: %s" % type(e).__name__)
    return "not bound (" + "; ".join(tried) + ")"


def w1_of(W, p):
    maxD = p["minDisp"] + p["numDisp"]
    return (W + min(p["minDisp"], 0)) - max(maxD, 0)


def cells_per_frame(spec, W=None):
    W = W or spec["W"]
    p = spec["params"]
    if spec["kind"] == "bm":
        return (W - p["numDisp"] + 1) * spec["H"] * p["numDisp"]
    return w1_of(W, p) * spec["H"] * p["numDisp"]


def dump_sample(a):
    """`a` as float32; above DUMP_VALUES_PER_ARRAY values, the values at a fixed seeded sample of its flat indices
    (ascending), the same sample for every run at the same shape."""
    if a.size > DUMP_VALUES_PER_ARRAY:
        idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_VALUES_PER_ARRAY, replace=False))
        a = a.reshape(-1)[idx]
    return a.astype(np.float32)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU reference: OpenCV through cv2 (frame-parallel, one matcher per worker, cv2.setNumThreads(1))
# ---------------------------------------------------------------------------------------------------------------
def _cv2_or_none():
    try:
        import cv2
        return cv2
    except Exception:
        return None


def _make_cv_matcher(cv2, spec):
    p = spec["params"]
    if spec["kind"] == "bm":
        m = cv2.StereoBM_create(numDisparities=p["numDisp"], blockSize=p["blockSize"])
        m.setPreFilterCap(p["preFilterCap"]); m.setUniquenessRatio(p["uniquenessRatio"]); m.setTextureThreshold(p["textureThreshold"])
        return m
    return cv2.StereoSGBM_create(minDisparity=p["minDisp"], numDisparities=p["numDisp"], blockSize=p["blockSize"],
                                 P1=p["P1"], P2=p["P2"], disp12MaxDiff=p["disp12MaxDiff"], preFilterCap=p["preFilterCap"],
                                 uniquenessRatio=p["uniquenessRatio"], speckleWindowSize=p["speckleWindowSize"],
                                 speckleRange=p["speckleRange"],
                                 mode=cv2.STEREO_SGBM_MODE_HH if p["disparityMode"] == 1 else cv2.STEREO_SGBM_MODE_SGBM)


def load_rectification():
    """Maps cv2 derives from the reference's parameters/baseline_small calibration (committed fixture, generated by
    tests/golden/make_golden.py)."""
    g = synth.load_rectification(os.path.join(ROOT, "tests", "golden"))
    return g, tuple(int(v) for v in g["roi"])


def cv_reference_frame(cv2, spec, left, right):
    """The reference's CPU path for one frame of `spec` (what the GPU result must equal bit for bit)."""
    if spec["kind"] == "pipeline":
        g, roi = load_rectification()
        x, y, w, h = roi
        left = np.ascontiguousarray(cv2.remap(left, g["m1x"], g["m1y"], cv2.INTER_LINEAR)[y:y + h, x:x + w])
        right = np.ascontiguousarray(cv2.remap(right, g["m2x"], g["m2y"], cv2.INTER_LINEAR)[y:y + h, x:x + w])
    return _make_cv_matcher(cv2, spec).compute(left, right)


class CpuReference:
    """Times the reference's CPU path.  kind = "reference": cv2's StereoSGBM (the OpenCV call the reference makes);
    kind = "port": the C oracle (only if cv2 cannot be imported)."""

    def __init__(self, spec, frames):
        self.spec, self.frames = spec, frames
        self.cv2 = _cv2_or_none()
        self.cores = max(1, os.cpu_count() or 1)
        if self.cv2 is not None:
            self.cv2.setNumThreads(1)
            self.kind = "reference"
            from concurrent.futures import ThreadPoolExecutor
            self.pool = ThreadPoolExecutor(self.cores)
            self.matchers = [_make_cv_matcher(self.cv2, spec) for _ in range(self.cores)]
        else:
            import oracle
            self.oracle = oracle
            self.kind = "port"
            self.cores = 1

    def run(self, frames_per_worker):
        """Every worker processes frames_per_worker frames; returns (seconds, frames, outputs of worker 0)."""
        if self.kind == "reference":
            def work(wi):
                outs = []
                for j in range(frames_per_worker):
                    l, r = self.frames[(wi + j * self.cores) % len(self.frames)]
                    outs.append(self.matchers[wi].compute(l, r))
                return outs
            t0 = time.perf_counter()
            res = list(self.pool.map(work, range(self.cores)))
            dt = time.perf_counter() - t0
            return dt, frames_per_worker * self.cores, res[0]
        p = dict(self.spec["params"])
        p["mode"] = p.pop("disparityMode")
        t0 = time.perf_counter()
        outs = [self.oracle.sgbm(*self.frames[j % len(self.frames)], p) for j in range(frames_per_worker)]
        return time.perf_counter() - t0, frames_per_worker, outs

    def describe(self):
        if self.kind == "reference":
            return "cv2 %s StereoSGBM.compute, %d frame-parallel workers (cv2.setNumThreads(1) each)" % (
                self.cv2.__version__, self.cores)
        return "C oracle port (oracle/mvsv_oracle.c), single thread"


def run_reference_arm(args, rank):
    if rank != 0:
        return 0
    spec = CONFIGS[HEADLINE]
    p = spec["params"]
    frames = [synth.stereogram(spec["H"], spec["W"], p["minDisp"], p["numDisp"], seed=s)[:2] for s in range(16)]
    ref = CpuReference(spec, frames)
    fpw = 2 if ref.kind == "reference" else 1
    for _ in range(max(args.warmup, 1)):
        ref.run(1)
    t_total, n_total = 0.0, 0
    for _ in range(args.steps):
        dt, n, _ = ref.run(fpw)
        t_total += dt; n_total += n
    fps = n_total / t_total
    gd = spec["W"] * spec["H"] * p["numDisp"] * fps / 1e9
    sample = "%d steps x %d frames of the cfg-2 workload (%s)" % (args.steps, fpw * ref.cores, ref.describe())
    line = {"impl": "reference", "metric": "sgbm_frames_per_s", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16", "data": "synthetic",
            "gdisp_evals_per_s": gd,
            "config": {"workload": spec["name"], "frames_per_step": fpw * ref.cores, "host_cores": ref.cores},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": ref.cores, "kind": ref.kind, "sample": sample},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------------------
# One configuration on this rank's GPU
# ---------------------------------------------------------------------------------------------------------------
class Ctx:
    """torch / distributed plumbing shared by all configurations of a run."""

    def __init__(self, torch, api, dist, dev, rank, world, local_rank):
        self.torch, self.api, self.dist, self.dev = torch, api, dist, dev
        self.rank, self.world, self.local_rank = rank, world, local_rank


def make_inputs(spec, ids, B):
    """B stereo pairs of the configuration for frame ids `ids` (at most 16 distinct seeded pairs; the batch repeats
    them -- the matcher's work does not depend on the content, the speckle filter's labelling does slightly)."""
    p, H, W = spec["params"], spec["H"], spec["W"]
    uniq = min(B, 16)
    minD = p.get("minDisp", 0)
    gen = [synth.stereogram(H, W, minD, p["numDisp"], seed=ids[i])[:2] for i in range(uniq)]
    return gen, uniq


def run_config(cx, key, batch, steps, warmup, detail=False, dump=False):
    """Device-resident and end-to-end throughput of one configuration (this rank's share of the frames), plus a
    one-frame bit-exactness check against cv2 on rank 0.  Returns a dict; `detail` adds per-kernel times, `dump` the
    outputs of the last device-resident step under "_dump" (dump_sample of each)."""
    torch, api = cx.torch, cx.api
    spec = CONFIGS[key]
    p, H, W, B = spec["params"], spec["H"], spec["W"], batch
    ids = shard.frames_for_rank(B * cx.world, cx.rank, cx.world)
    gen, uniq = make_inputs(spec, ids, B)
    hl, hr = api.pinned((B, H, W), np.uint8), api.pinned((B, H, W), np.uint8)
    for i in range(B):
        hl.array[i], hr.array[i] = gen[i % uniq]
    dl = torch.from_numpy(hl.array).to(cx.dev)
    dr = torch.from_numpy(hr.array).to(cx.dev)

    eng = api.Engine(W, H, max_batch=B, device=cx.local_rank)
    stages, extra_out = api.STAGE_SGBM, {}
    if spec["kind"] == "bm":
        eng.set_bm_params(**p)
        stages = api.STAGE_BM
    else:
        if spec["kind"] == "pipeline":
            g, roi = load_rectification()
            eng.upload_rectify_maps(0, g["m1x"], g["m1y"], roi)
            eng.upload_rectify_maps(1, g["m2x"], g["m2y"], roi)
            stages = api.STAGE_RECTIFY | api.STAGE_SGBM | api.STAGE_XYZ | api.STAGE_MEANS
        eng.set_sgbm_params(**p)
        if spec["kind"] == "pipeline":
            eng.set_Q(g["Q"])
            oW, oH = eng.info.width, eng.info.height
            off = api.dmap_roi_offset(p["numDisp"], oW)
            rois = api.subimage_rois(oW - off, oH, off) + api.samplepoint_rois(oW - off, oH, off)
            eng.set_mean_rois(rois)
            extra_out = {"means": True}
    oW, oH = eng.info.width, eng.info.height
    cells = cells_per_frame(spec, oW) if spec["kind"] == "pipeline" else cells_per_frame(spec)
    if spec["kind"] == "pipeline":
        cells = w1_of(oW, p) * oH * p["numDisp"]
    hd = [api.pinned((B, oH, oW), np.int16) for _ in range(2)]

    def fence():
        eng.sync()
        torch.cuda.synchronize()
        if cx.dist is not None:
            cx.dist.barrier()

    # ---- HBM-resident figure: CUDA events on the engine's stream ------------------------------------------------
    def step_device():
        eng.compute_device(dl.data_ptr(), W, dr.data_ptr(), W, H * W, B, stages)

    for _ in range(warmup):
        step_device()
    fence()
    sampler = ClockSampler(cx.local_rank) if (detail and cx.rank == 0) else None
    if sampler:
        sampler.start()
    l0 = eng.launch_count
    eng.timer_start()
    for _ in range(steps):
        step_device()
    ms = eng.timer_stop()
    launches = eng.launch_count - l0
    fence()
    dumped = {k: dump_sample(v) for k, v in eng.download(B, **extra_out).items()} if dump else None
    # Per-kernel CUDA-event durations come from a second pass over the same K steps: with per-kernel timing enabled the
    # engine runs its kernels one after the other (mvsv_profile_enable), while in the timed pass above the cost kernel
    # and the first row scan of different chunks of frames overlap on two streams -- a kernel's duration only means
    # something when it runs alone, so the kernel times add up to a little more than ms_per_step.
    eng.profile_enable(True)
    for _ in range(steps):
        step_device()
    eng.sync()
    prof = eng.profile_read()
    eng.profile_enable(False)
    fence()
    clocks = sampler.stop() if sampler else None
    ms_max, frames_total = shard.reduce_max_and_sum(cx.dist, cx.dev, ms, B * steps)
    fps = frames_total / (ms_max * 1e-3)

    # ---- end to end through the host-facing call ---------------------------------------------------------------
    # One engine, two I/O slots: compute k+1 is submitted (pinned H2D on the copy stream + kernels on the engine's
    # stream) before the results of compute k are fetched (D2H on the download stream), so both copies overlap
    # kernels while the cost volumes exist once.  Every step does its own H2D of both images and D2H of its results.
    eng.set_io_slots(2)

    def submit(k):
        eng.compute(hl.array, hr.array, stages)

    def collect(k, age):
        return eng.download(B, out={"disp": hd[k & 1].array}, age=age, **extra_out)

    def e2e_loop(n):
        submit(0)
        for k in range(1, n):
            submit(k)
            collect(k - 1, 1)
        return collect(n - 1, 0)

    e2e_loop(3)
    fence()
    t0 = time.perf_counter()
    last = e2e_loop(steps)
    eng.sync()
    ms_e2e = (time.perf_counter() - t0) * 1e3          # host clock between two device synchronisations
    fence()
    if os.environ.get("MVSV_BENCH_DEBUG"):
        print("[rank %d] %s: device %.3f ms/step, e2e %.3f ms/step" % (cx.rank, key, ms / steps, ms_e2e / steps), file=sys.stderr, flush=True)
    ms_e2e_max, frames_e2e = shard.reduce_max_and_sum(cx.dist, cx.dev, ms_e2e, B * steps)
    fps_e2e = frames_e2e / (ms_e2e_max * 1e-3)
    gpu_disp = hd[(steps - 1) & 1].array[:uniq].copy()
    if steps > 1:
        assert np.array_equal(hd[0].array, hd[1].array), "consecutive pipelined steps disagree"
    d2h = 2 * B * oH * oW + (4 * B * eng.info.num_rois if extra_out else 0)

    # ---- bit-exactness of frame 0 against the reference's CPU path, computed in this run -------------------------
    parity = None
    cv2 = _cv2_or_none() if cx.rank == 0 else None
    if cv2 is not None:
        cv2.setNumThreads(max(1, os.cpu_count() or 1))
        t0 = time.perf_counter()
        want = cv_reference_frame(cv2, spec, gen[0][0], gen[0][1])
        parity = {"frames_checked": 1, "bit_exact_vs_cv2": bool(np.array_equal(want, gpu_disp[0])),
                  "cv2_seconds_per_frame_one_thread_pool": time.perf_counter() - t0}
        cv2.setNumThreads(1)
    peak, _ = hbm_peak()
    out = {"workload": spec["name"], "batch_per_gpu": B, "steps": steps, "value": fps, "unit": "frames/s",
           "ms_per_step": ms_max / steps,
           "e2e": {"value": fps_e2e, "unit": "frames/s", "ms_per_step": ms_e2e_max / steps,
                   "h2d_bytes_per_step": 2 * B * H * W, "d2h_bytes_per_step": d2h},
           "evaluated_gcells_per_s": cells * fps / 1e9,
           "gdisp_evals_per_s": W * H * p["numDisp"] * fps / 1e9,
           "roofline_path": {"model_bytes_per_cell": spec["model_bpc"],
                             "achieved": spec["model_bpc"] * cells * fps / cx.world / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": spec["model_bpc"] * cells * fps / cx.world / 1e9 / peak},
           "kernel_ms_per_step": {k: v[0] / steps for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])},
           "sweep_strips_per_frame": eng.info.sgbm_td_cluster if spec["kind"] != "bm" else None,
           "s_volume": None if spec["kind"] == "bm" else ("u8 excess over npaths*C" if eng.info.sgbm_s8 else "u16"),
           "bm_column_sums": None if spec["kind"] != "bm" else ("u8 (blockSize*2*cap <= 255)" if eng.info.bm_col8 else "u16"),
           "parity": parity}
    if spec["kind"] == "bm":
        # bytes the two volume kernels actually move per cell: the column sums written once and read once
        out["roofline_path"]["step_bytes_per_cell"] = 2.0 if eng.info.bm_col8 else 4.0
    if dump:
        out["_dump"] = dumped
    if detail:
        out["_detail"] = dict(s8=bool(eng.info.sgbm_s8), prof=prof, launches=launches, clocks=clocks, gen=gen, uniq=uniq, gpu_disp=gpu_disp,
                              cells=cells, fps=fps, fps_e2e=fps_e2e, ms_max=ms_max, ms_e2e_max=ms_e2e_max, d2h=d2h)
    eng.close()
    for b in (hl, hr, hd[0], hd[1]):
        b.close()
    del dl, dr
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=CONFIGS[HEADLINE]["batch"],
                    help="stereo pairs per GPU per step of the headline workload (148 = one frame slot per SM pair)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--configs", default="all",
                    help="comma separated keys of the other BASELINE configurations to add to the line (%s), "
                         "'all' or 'none'" % ", ".join(k for k in CONFIGS if k != HEADLINE))
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of each configuration's last timed step to DIR/<config>_<array>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference_arm(args, rank)

    import torch
    from mvstereovision3_b200 import api
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback (use --impl reference for the CPU arm)")
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else "single process, not bound"
    cx = Ctx(torch, api, dist, dev, rank, world, local_rank)

    spec = CONFIGS[HEADLINE]
    p, H, W, B = spec["params"], spec["H"], spec["W"], args.batch
    dump = args.dump_outputs is not None and rank == 0
    head = run_config(cx, HEADLINE, B, args.steps, args.warmup, detail=True, dump=dump)
    det = head.pop("_detail")
    dumped = {HEADLINE: head.pop("_dump", None)}

    # ---- the other BASELINE configurations (same measurement, same parity gate) ----------------------------------
    others = {}
    want = [k for k in CONFIGS if k != HEADLINE] if args.configs == "all" else (
        [] if args.configs == "none" else [k.strip() for k in args.configs.split(",") if k.strip()])
    for key in want:
        try:
            others[key] = run_config(cx, key, CONFIGS[key]["batch"], args.steps, args.warmup, dump=dump)
            dumped[key] = others[key].pop("_dump", None)
        except Exception as e:       # a configuration that cannot run must not take the headline down with it
            others[key] = {"workload": CONFIGS[key]["name"], "error": "%s: %s" % (type(e).__name__, e)}

    if dump:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for key, arrays in dumped.items():
            for name, a in (arrays or {}).items():
                np.save(os.path.join(args.dump_outputs, "%s_%s.npy" % (key, name)), a)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel (live CUDA-event durations from the timed region) ----------------------
    peak, peak_src = hbm_peak()
    ncu = ncu_summary()
    cells = det["cells"]
    cells_per_launch = cells * B
    prof = det["prof"]
    kbytes = KERNEL_BYTES_PER_CELL_S8 if det["s8"] else KERNEL_BYTES_PER_CELL
    kern = {k: {"ms_total": v[0], "launches": v[1], "ms_per_launch": v[0] / v[1]} for k, v in prof.items()}
    total_kernel_ms = sum(v["ms_total"] for v in kern.values())
    for k, v in kern.items():
        v["share"] = v["ms_total"] / total_kernel_ms if total_kernel_ms else 0.0
        if k in kbytes:
            v["algorithmic_GBps"] = kbytes[k] * cells_per_launch / (v["ms_per_launch"] * 1e-3) / 1e9
    dom = max(kern, key=lambda k: kern[k]["ms_total"])
    tpc = (ncu.get("dram_bytes_per_cell") or {}).get(dom)
    if dom in kbytes:
        ach = kern[dom]["algorithmic_GBps"]
        roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": (tpc * cells_per_launch if tpc is not None else None), "peak_source": peak_src,
                    "bytes_per_cell": kbytes[dom], "cells_per_launch": cells_per_launch,
                    "ms_per_launch": kern[dom]["ms_per_launch"], "share_of_step": kern[dom]["share"]}
    else:
        roofline = {"bound": "hbm", "kernel": dom, "achieved": None, "peak": peak, "unit": "GB/s", "frac": None,
                    "traffic": None, "peak_source": peak_src}
    # integer / DPX pipe: packed 16x2 lane operations of the dominant kernel (ncu: ALU-pipe instructions x 32 lanes
    # per evaluated cell, from the committed capture) over its live duration, against the measured issue peak
    ipeak, ipeak_src = int_pipe_peak()
    ops_pc = (ncu.get("alu_pipe_lane_ops_per_cell") or {}).get(dom)
    roofline_int = {"bound": "int-pipe", "kernel": dom, "unit": "lane-ops/s", "peak": ipeak, "peak_source": ipeak_src,
                    "lane_ops_per_cell": ops_pc,
                    "achieved": (ops_pc * cells_per_launch / (kern[dom]["ms_per_launch"] * 1e-3) if ops_pc else None)}
    roofline_int["frac"] = roofline_int["achieved"] / ipeak if roofline_int["achieved"] else None
    # whole-path figure against the 8 B/cell aggregation model of SURVEY.md 8(d)
    roofline_path = dict(head["roofline_path"], note="per GPU; whole step (all kernels) against the 8 B/cell model",
                         step_bytes_per_cell=sum(kbytes.get(k, 0.0) * v["launches"] / args.steps for k, v in kern.items()))

    # ---- CPU baseline on this box's host cores (bounded sample) + parity gate on the frames it computed ---------
    cpu = None
    parity = head["parity"]
    if world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(spec, det["gen"])
        ref.run(1)
        fpw = 16 if ref.kind == "reference" else 2          # ~14 s of CPU work on 16 cores (cv2), bounded for the port
        dt, n, outs = ref.run(fpw)
        cpu = {"value": n / dt, "unit": "frames/s", "cores": ref.cores, "kind": ref.kind,
               "sample": "%d frames of the same workload, %s, %.1f s wall" % (n, ref.describe(), dt),
               "gdisp_evals_per_s": W * H * p["numDisp"] * (n / dt) / 1e9}
        ok, checked = True, 0
        for j, o in enumerate(outs):
            fi = (0 + j * ref.cores) % det["uniq"]
            ok &= bool(np.array_equal(o, det["gpu_disp"][fi]))
            checked += 1
        parity = {"frames_checked": checked, "bit_exact_vs_cpu_reference": ok}

    line = {"metric": "sgbm_frames_per_s", "value": det["fps"], "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": det["ms_max"] / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int16", "data": "synthetic",
            "gdisp_evals_per_s": W * H * p["numDisp"] * det["fps"] / 1e9,
            "evaluated_gcells_per_s": cells * det["fps"] / 1e9,
            "config": {"workload": spec["name"], "batch_per_gpu": B, "frames_per_step": B * world,
                       "sharding": "frame i -> rank i mod N, no collective", "host_binding_rank0": numa,
                       "inputs": "16 distinct seeded stereograms repeated over the batch (the matcher's work is content "
                                 "independent; the connected-components labelling of the speckle filter is not)",
                       "l2": "working set per step (3 int16 volumes x %d frames = %.1f GB) exceeds the 126 MB L2"
                             % (B, 3 * 2 * cells * B / 1e9)},
            "e2e": {"value": det["fps_e2e"], "unit": "frames/s", "h2d_bytes_per_step": 2 * B * H * W,
                    "d2h_bytes_per_step": det["d2h"], "ms_per_step": det["ms_e2e_max"] / args.steps,
                    "pipeline": "one engine, two I/O slots (mvsv_set_io_slots): H2D of step k+1 and D2H of step k-1 "
                                "overlap the kernels of step k; pinned host buffers; host clock between device syncs",
                    "gdisp_evals_per_s": W * H * p["numDisp"] * det["fps_e2e"] / 1e9},
            "gpu_launches": det["launches"], "clocks": det["clocks"], "roofline": roofline, "roofline_int": roofline_int,
            "roofline_path": roofline_path, "kernels": kern, "cpu_baseline": cpu, "parity": parity, "configs": others}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
