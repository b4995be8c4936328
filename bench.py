#!/usr/bin/env python3
"""Benchmark of the AprilTag detection hot path (BASELINE.json metric: frames/s per GPU and box at
1280x800 tag36h11, plus p50 latency).

  python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA engine
  python bench.py --impl reference ...                            the CPU implementation of the same path

A "step" is one pass of the hot path over one batch of synthetic frames of BASELINE config 2
(Arducam-style 1280x800 YUYV stream, tag36h11, quad_decimate=2) on each of `--device-lanes` detectors.
  value      frames/s with the frames already resident in HBM when the timed region starts
  e2e        frames/s through the public API with HOST (pinned) frame buffers: H2D copies, all kernels
             and the result read-back inside the timed region
  p50/p99    host frame in -> detections out, one frame at a time
  roofline   the slowest FRONT-END kernel: algorithmic bytes per launch / measured launch duration vs the measured HBM
             peak; the front end as a whole (per-kernel bytes and compulsory bytes); per kernel the CUDA-event time and,
             from the committed ncu table (profiles/traffic.json), DRAM bytes and issue-slot utilisation
  step_stats min / median / max of the step time
  cpu_baseline  the classic CPU detector (libapriltag's apriltag_detector_detect restated in oracle/classic_detector.c,
             kind "port") on a bounded sample of the same frames: one thread and all threads, CPU model printed
  e2e_mjpg   the same scenes as JPEG bitstreams in host memory (the camera wire format), at every N
  extra      BASELINE configs 4 (one 1600x1200 stream per GPU) and 5 (4K clutter scene, batch 16 per GPU), at every N
Multi-GPU (torchrun): frames shard by rank, no collective on the data path (SURVEY.md section 8e);
time = max over ranks, value = total frames / that time.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, FMT, DECIMATE, SIGMA = 1280, 800, "yuyv", 2, 0.0
WORKLOAD = "config2: 1280x800 YUYV stream, tag36h11, quad_decimate=2, 1-6 tags per frame, noise N(0,4)"
UNIQUE_FRAMES = 16     # distinct synthetic frames (seeds 2000..2015), tiled to fill a batch
BATCH = 128            # frames per step: 262 MB of input + ~3 GB of intermediates, far beyond the 126 MB L2
CONFIG = 2
SMALL_CAP, MEDIUM_CAP = 192, 768   # blob tiers of the fit kernels (dev_types.h kSmallBlobPoints, kernels_blobs.cu kMediumCap)

# the other BASELINE.json configs (parity-test cases; `--config N` measures them for DESIGN.md, the default
# bench line is always config 2): (W, H, fmt, decimate, sigma, workload, distinct frames, default batch)
OTHER_CONFIGS = {
    1: (640, 480, "gray", 2, 0.0, "config1: 640x480 gray, 4 tags", 8, 256),
    3: (1920, 1080, "bgr", 1, 0.8, "config3: 1920x1080 BGR, 30 small tags, quad_decimate=1, quad_sigma=0.8", 4, 16),
    4: (1600, 1200, "yuyv", 2, 0.0, "config4: 1600x1200 YUYV camera stream, 2-8 tags", 8, 64),
    5: (3840, 2160, "yuyv", 2, 0.0, "config5: 3840x2160 YUYV cluttered scene, 100 tags, batch 16", 2, 16),
}


def select_config(cfg: int):
    global W, H, FMT, DECIMATE, SIGMA, WORKLOAD, UNIQUE_FRAMES, BATCH, CONFIG
    if cfg == 2:
        return
    W, H, FMT, DECIMATE, SIGMA, WORKLOAD, UNIQUE_FRAMES, BATCH = OTHER_CONFIGS[cfg]
    CONFIG = cfg


def make_frames(n_unique=None):
    from ros_vision_b200 import synth
    out = []
    for i in range(n_unique or UNIQUE_FRAMES):
        frame, fmt, w, h, dec, sigma, sc = synth.config_frame(CONFIG, i)
        if fmt != FMT:  # --format: the same scene in another pixel format (e.g. the node's bgr8 frames)
            frame = {"gray": lambda g: g, "yuyv": synth.gray_to_yuyv, "bgr": synth.gray_to_bgr}[FMT](sc.gray)
        out.append(np.ascontiguousarray(frame).reshape(-1))
    return out


def algorithmic_bytes_per_frame(points_per_frame: float) -> float:
    """B_frame of SURVEY.md section 8(d): input + gray + quad + thresholded + labels + 8 B per boundary point."""
    N, n = W * H, (W // DECIMATE) * (H // DECIMATE)
    bpp = {"gray": 1, "yuyv": 2, "bgr": 3}[FMT]
    return bpp * N + (N if FMT != "gray" else 0) + (n if (DECIMATE > 1 or SIGMA != 0) else 0) + n + 4 * n + 8.0 * points_per_frame


# per-kernel algorithmic bytes per frame (SURVEY.md section 8(d), "Per-kernel algorithmic bytes", for the kernels as
# they are fused here; DESIGN.md section 2 lists them).  Per-blob kernels (fit_*, quads, decode) are latency / issue
# bound: their only compulsory HBM traffic is the 4-byte segment point each of them reads once.
FRONT_END = ("pre_yuyv_dec2", "pre_gray_dec2", "pre_bgr_dec1", "pre_bgr_dec2", "pre_generic", "blur", "tile_minmax",
             "ccl_local", "ccl_merge", "ccl_handoff", "ccl_final", "boundary", "select", "scatter")


def kernel_bytes(name: str, P: float, tiers: dict) -> float:
    N, n = W * H, (W // DECIMATE) * (H // DECIMATE)
    Pseg = tiers["small"] + tiers["medium"] + tiers["large"]
    bpp = {"gray": 1, "yuyv": 2, "bgr": 3}[FMT]
    table = {
        "pre_yuyv_dec2": 2 * N + N + n + n / 8,
        "pre_gray_dec2": N / 2 + n + n / 8,
        "pre_generic": bpp * N + (N if FMT != "gray" else 0) + n + n / 8,
        "pre_bgr_dec1": 3 * N + N + n,
        "pre_bgr_dec2": 3 * N + N + n + n / 8,
        "blur": n + n,
        "tile_minmax": n + n / 8,
        "ccl_local": n + n / 8 + n + 4 * n + 4 * n,   # quad image + raw tile min/max in; thresholded, labels, sizes out
        "ccl_merge": 0.0,                             # tile borders only
        "ccl_handoff": 0.0,                           # border-touching tile roots only
        "ccl_final": 4 * n + 4 * n,                   # label words in, label words out
        "boundary": 4 * n + 8 * P,                    # label words in, point records out
        "select": 0.0,
        "scatter": 8 * P + 4 * Pseg,
        "fit_small": 4 * tiers["small"],
        "fit_medium": 4 * tiers["medium"],
        "fit_large": 4 * tiers["large"],
        "decode": 0.0,
    }
    return table.get(name, 0.0)


class ClockSampler:
    """Samples SM clocks and throttle reasons while a timed region runs: NVML every 10 ms (nvidia_ml_py), or
    nvidia-smi every 200 ms when NVML is not importable.  Several regions can be sampled into one summary."""

    _NVML_REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        try:
            self.index = int(vis.split(",")[index]) if vis else index
        except ValueError:
            self.index = index
        self.samples = []   # (sm_mhz, sm_max_mhz, [reasons])
        self._stop = threading.Event()
        self._t = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        nv = self._nvml
        sm = nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)
        mx = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
        try:
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        self.samples.append((int(sm), int(mx), [n for bit, n in self._NVML_REASONS.items() if mask & bit]))

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
            f = [x.strip() for x in out.split(",")]
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            self.samples.append((int(f[0]), int(f[1]), [n for n, v in zip(names, f[2:6]) if v.lower().startswith("active")]))

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.01 if self._nvml else 0.2)

    def __enter__(self):
        self._stop.clear()
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(s[0] for s in self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(s[1] for s in self.samples),
                "reasons": sorted({r for s in self.samples for r in s[2]}), "samples": len(self.samples),
                "source": "nvml" if self._nvml else "nvidia-smi", "regions": "device-resident and end-to-end timed regions"}


def pin_to_gpu_numa_node(local: int):
    """Runs this rank on the CPU cores next to its GPU (NVML's ideal CPU set), so that the pinned frame buffers it
    allocates are on the GPU's NUMA node: with 8 ranks pulling ~50 GB/s each over PCIe, frames that sit on the other
    socket would have to cross the inter-socket link first.  Returns the core list (or None)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        idx = int(vis.split(",")[local]) if vis else local
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        words = (max(os.cpu_count() or 1, 1024) + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {i * 64 + b for i, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)
    except Exception:
        pass
    return None


def dist_setup(n_gpus: int):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ----------------------------------------------------------------------------------------------
def cpu_model() -> str:
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def gray_planes(frames):
    """The luma plane of every frame: what the reference's CPU path is handed (cv::COLOR_BGR2GRAY of the frame,
    gpu_detector_test.cu:106) -- the colour conversion itself is left out of the CPU figure, in its favour."""
    out = []
    for f in frames:
        if FMT == "gray":
            out.append(np.ascontiguousarray(f.reshape(H, W)))
        elif FMT == "yuyv":
            out.append(np.ascontiguousarray(f.reshape(H, W, 2)[:, :, 0]))
        else:
            from ros_vision_b200 import synth
            out.append(synth.bgr_to_luma(f.reshape(H, W, 3)))
    return out


def cpu_timed(fn, work, threads):
    from concurrent.futures import ThreadPoolExecutor
    t0 = time.perf_counter()
    if threads == 1:
        for f in work:
            fn(f)
    else:
        with ThreadPoolExecutor(threads) as ex:  # ctypes releases the GIL inside the C call
            list(ex.map(fn, work))
    return time.perf_counter() - t0


def cpu_baseline(frames, seconds_budget=14.0, threads=None):
    """The reference's CPU path for this workload: the classic AprilTag 3 detector (libapriltag
    apriltag_detector_detect as gpu_detector_test.cu:104-120 runs it; upstream is not vendored, so this is the
    restatement in oracle/classic_detector.c, kind "port"), compiled -O3, on a bounded sample of the bench frames.
    Timed with ONE thread and with every host thread (frames in parallel: a frame is independent work, which favours
    the CPU more than upstream's intra-frame worker pool); `value` is the all-threads figure.  The GPU-semantics
    oracle (the restatement of GpuDetector's arithmetic the parity tests use) is timed beside it."""
    from oracle import pyoracle
    pyoracle.build()
    cfg = pyoracle.make_config(W, H, "gray", DECIMATE, SIGMA)
    grays = gray_planes(frames)
    threads = threads or (os.cpu_count() or 1)
    classic = lambda g: pyoracle.classic_detect_raw(cfg, g)  # noqa: E731
    t0 = time.perf_counter()
    classic(grays[0])
    one = max(time.perf_counter() - t0, 1e-3)
    n1 = max(4, min(256, int(0.25 * seconds_budget / one)))
    dt1 = cpu_timed(classic, [grays[i % len(grays)] for i in range(n1)], 1)
    nt = max(threads, min(4096, int(0.5 * seconds_budget / one) * threads))
    dtn = cpu_timed(classic, [grays[i % len(grays)] for i in range(nt)], threads)
    ocfg = pyoracle.make_config(W, H, FMT, DECIMATE, SIGMA)
    no = max(threads, min(2048, int(0.25 * seconds_budget / (3 * one)) * threads))
    dto = cpu_timed(lambda f: pyoracle.detect_raw(ocfg, f), [frames[i % len(frames)] for i in range(no)], threads)
    return {"value": nt / dtn, "unit": "frames/s", "cores": threads, "kind": "port",
            "what": "classic CPU detector (libapriltag apriltag_detector_detect restated in oracle/classic_detector.c), gcc -O3",
            "one_thread": {"value": n1 / dt1, "unit": "frames/s", "frames": n1, "seconds": dt1},
            "all_threads": {"value": nt / dtn, "unit": "frames/s", "threads": threads, "frames": nt, "seconds": dtn},
            "gpu_semantics_oracle": {"value": no / dto, "unit": "frames/s", "threads": threads, "frames": no, "seconds": dto,
                                     "what": "oracle/apriltag_oracle.c (GpuDetector's arithmetic, the parity checker), built for parity not speed"},
            "cpu_model": cpu_model(), "host_threads": os.cpu_count(),
            "sample": f"{nt} luma frames of the bench workload ({len(frames)} distinct), oracle/liboracle.so classic detector, "
                      f"{threads} threads, {dtn:.1f} s (+ {n1} frames on 1 thread, {dt1:.1f} s)"}


def reference_gpu_leg(frames, iters=300):
    """The reference's own GpuDetector (its kernels recompiled for sm_100a into oracle/_ref by
    oracle/build_ref.sh), one synchronous Detect per frame exactly as the node calls it (pageable H2D
    included).  libapriltag is absent, so quad decode is stubbed: the figure EXCLUDES decode and is
    therefore an upper bound on the reference's frame rate.  Reported beside the headline, never as it."""
    try:
        from oracle import pyrefgpu
        if not pyrefgpu.available():
            return None
        ref = pyrefgpu.ReferenceGpuDetector(W, H)
        ms = ref.time_detect([f.reshape(H, W * 2) for f in frames], iters=iters, warmup=20)
        ref.close()
        return {"value": 1e3 / ms, "unit": "frames/s", "ms_per_frame": ms, "kind": "reference kernels recompiled for sm_100a "
                "(oracle/_ref/librefgpu.so), synchronous Detect per frame, pageable H2D, decode excluded",
                "sample": f"{iters} frames, {len(frames)} distinct"}
    except Exception as e:  # reporting leg only
        return {"unavailable": repr(e)[:200]}


def opencv_aruco_leg(frames, seconds_budget=4.0):
    """Independent CPU datapoint (SURVEY 8d): OpenCV's ArucoDetector with the AprilTag 36h11 dictionary and AprilTag
    corner refinement on the luma plane of the same frames, OpenCV's own threading.  Not the reference and not the
    target -- a different detector, reported for orientation only."""
    try:
        import cv2
        ar = cv2.aruco
        params = ar.DetectorParameters()
        params.cornerRefinementMethod = ar.CORNER_REFINE_APRILTAG
        params.aprilTagQuadDecimate = float(DECIMATE)
        det = ar.ArucoDetector(ar.getPredefinedDictionary(ar.DICT_APRILTAG_36h11), params)
        bpp = {"gray": 1, "yuyv": 2, "bgr": 3}[FMT]
        grays = []
        for f in frames[:8]:
            a = f.reshape(H, W, bpp) if bpp > 1 else f.reshape(H, W)
            grays.append(np.ascontiguousarray(a[:, :, 0] if FMT == "yuyv" else (a if bpp == 1 else cv2.cvtColor(a, cv2.COLOR_BGR2GRAY))))
        det.detectMarkers(grays[0])
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds_budget:
            det.detectMarkers(grays[n % len(grays)])
            n += 1
        dt = time.perf_counter() - t0
        return {"value": n / dt, "unit": "frames/s", "kind": f"cv2 {cv2.__version__} aruco.ArucoDetector, DICT_APRILTAG_36h11, "
                "CORNER_REFINE_APRILTAG", "threads": cv2.getNumThreads(), "sample": f"{n} frames in {dt:.1f} s"}
    except Exception as e:  # reporting leg only
        return {"unavailable": repr(e)[:200]}


def safe_leg(fn, *a):
    """Informational legs must never cost the bench line: a failure is reported in place of their result."""
    try:
        return fn(*a)
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"}


def mjpg_leg(local: int, rank: int = 0, world: int = 1, steps: int = 18, quality: int = 75):
    """SURVEY section 8 row f2, at every N: the same config-2 scenes as 4:2:2 JPEG bitstreams in host memory ->
    b200tag_enqueue_mjpg (hand-written JPEG luminance decode kernels + detection) -> detections on the host; wall clock
    around `steps` 128-frame batches on three detectors per GPU, barrier on both sides, max over ranks.  It moves 1/18 of
    the raw-YUYV bytes over PCIe, so it shows what the box does when the host->device link is not the limit.
    None when OpenCV (the test encoder) is missing."""
    try:
        import cv2
    except ImportError:
        return None
    import torch
    import torch.distributed as dist
    from ros_vision_b200 import detector as D, synth
    jpgs, present = [], 0
    for i in range(16):
        _, _, w, h, dec, sigma, sc = synth.config_frame(2, i)
        bgr = synth.gray_to_bgr(sc.gray, np.random.default_rng(i))
        ok, buf = cv2.imencode(".jpg", bgr, [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                                              cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422])
        if not ok:
            return None
        jpgs.append(buf.tobytes())
        present += len(sc.tags)
    nb = 128
    batch = [jpgs[(i + 3 * rank) % len(jpgs)] for i in range(nb)]
    lanes = 3  # detectors (streams) in flight
    dets = [D.GpuDetector(w, h, "gray", quad_decimate=dec, quad_sigma=sigma, max_batch=nb, device=local) for _ in range(lanes)]
    for _ in range(3):
        for d in dets:
            d.EnqueueMjpg(batch)
        for d in dets:
            d.Finish()
    found = sum(len(dets[0].Detections(f)) for f in range(len(jpgs)))
    parallel = dets[0].MjpgParallelFrames()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pending = []
    for it in range(steps):
        d = dets[it % lanes]
        if len(pending) == lanes:
            pending.pop(0).Finish()
        d.EnqueueMjpg(batch)
        pending.append(d)
    for d in pending:
        d.Finish()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    out = {"value": nb * steps * world / dt, "unit": "frames/s", "what": "JPEG bytes in host memory -> detections on the host",
           "jpeg_bytes_per_frame": int(np.mean([len(j) for j in jpgs])), "quality": quality, "sampling": "4:2:2",
           "h2d_bytes_per_step": int(sum(len(j) for j in batch)), "frames_per_step_per_gpu": nb, "steps": steps, "lanes": lanes,
           "n_gpus": world, "decoder": dets[0].mjpg_backend, "frames_decoded_by_parallel_kernels": parallel,
           "tags_found": found, "tags_present": present}
    for d in dets:
        d.close()
    if rank == 0 and world == 1:
        # the reference's way for this step, timed beside it: OpenCV (libjpeg-turbo) decodes each frame to bgr8 on a host
        # core (cv::VideoCapture with CAP_PROP_CONVERT_RGB, camera_publisher.cpp:198,336); bounded to about two seconds
        t0, n = time.perf_counter(), 0
        while time.perf_counter() - t0 < 2.0:
            cv2.imdecode(np.frombuffer(jpgs[n % len(jpgs)], np.uint8), cv2.IMREAD_COLOR)
            n += 1
        out["cpu_opencv_decode_only"] = {"value": n / (time.perf_counter() - t0), "unit": "frames/s", "threads": 1,
                                         "what": "cv2.imdecode to bgr8 alone (no detection), one host thread"}
    return out


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path -- the classic detector -- on the box's host
    cores, every thread busy (frames in parallel), same workload / metric / unit as our arm."""
    rank, world, local = dist_setup(args.gpus)
    if rank != 0:
        return
    frames = make_frames()
    from oracle import pyoracle
    pyoracle.build()
    cfg = pyoracle.make_config(W, H, "gray", DECIMATE, SIGMA)
    grays = gray_planes(frames)
    threads = os.cpu_count() or 1
    classic = lambda g: pyoracle.classic_detect_raw(cfg, g)  # noqa: E731
    t0 = time.perf_counter()
    classic(grays[0])
    one = max(time.perf_counter() - t0, 1e-3)
    # one step = a bounded sample sized so that steps + warmup finish in about a minute and a half
    total_steps = args.steps + args.warmup
    per_step = max(threads, min(4096, int(90.0 / total_steps / one) * threads))
    work = [grays[i % len(grays)] for i in range(per_step)]
    for _ in range(args.warmup):
        cpu_timed(classic, work, threads)
    dts = [cpu_timed(classic, work, threads) for _ in range(args.steps)]
    dt = sum(dts)
    value = per_step * args.steps / dt
    sample = (f"{per_step} luma frames per step of the bench workload, classic CPU detector (oracle/classic_detector.c; upstream "
              f"libapriltag is not vendored), {threads} host threads, frames in parallel")
    line = {
        "impl": "reference", "metric": "frames/s", "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step": per_step},
        "step_stats": {"min": min(dts) * 1e3, "median": float(np.median(dts)) * 1e3, "max": max(dts) * 1e3, "n": len(dts)},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample,
                         "cpu_model": cpu_model()},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
class Timing:
    """barrier + synchronize on both sides, CUDA events on the detectors' own streams, max over lanes and ranks."""

    def __init__(self, torch, dist, world, local):
        self.torch, self.dist, self.world, self.local = torch, dist, world, local

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())


DUMP_CAP_BYTES = 64 << 20   # --dump-outputs writes at most this much


def dump_outputs(out_dir, dlanes, B):
    """Writes what the detectors return for their last batch as DIR/<name>.npy (float64), one row per frame or per
    detection, lanes in order: frames are numbered lane * B + frame.  Detections keep the engine's order (by id).
    Past DUMP_CAP_BYTES, every array keeps the same fixed, seeded fraction of its rows (frame_index and det_frame say
    which frames they are)."""
    os.makedirs(out_dir, exist_ok=True)
    infos, per_frame = [], []
    for d in dlanes:
        for f in range(B):
            i = d.FrameInfo(f)
            infos.append([getattr(i, n) for n, _ in i._fields_])
            per_frame.append(d.Detections(f))
    det = np.concatenate(per_frame)
    frame_rows = {
        "frame_index": np.arange(len(infos)),
        "frame_info": np.array(infos),   # b200tag_frame_info fields in their C order (status, num_points, ...)
    }
    det_rows = {
        "det_frame": np.concatenate([np.full(len(x), g) for g, x in enumerate(per_frame)]),
        "det_id": det["id"],
        "det_hamming": det["hamming"],
        "det_decision_margin": det["decision_margin"],
        "det_center": det["c"],
        "det_corners": det["p"],
        "det_homography": det["H"].reshape(-1, 3, 3),
    }
    groups = [frame_rows, det_rows]
    total = sum(8 * a.size for g in groups for a in g.values())
    budget = DUMP_CAP_BYTES - 4096 * sum(len(g) for g in groups)   # room for the .npy headers
    if total > budget:
        rng = np.random.default_rng(0)
        for g in groups:
            n = len(next(iter(g.values())))
            keep = np.sort(rng.choice(n, size=int(n * budget / total), replace=False))
            g.update({name: a[keep] for name, a in g.items()})
    for g in groups:
        for name, a in g.items():
            np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def device_resident_leg(T: Timing, D, rank, frames, B, DL, steps, warmup, clocks=None, dump_dir=None):
    """`DL` detectors, one CUDA stream each, take turns on batches that already sit in HBM: while the host collects
    lane k's results (the only host work between two batches) lane k+1's kernels keep the GPU busy.  One step = one
    batch per lane.  Returns the first detector (kept open, warm) and the device batch for the profiling leg.
    With `dump_dir`, every lane's results of the last step are written there after the timed region."""
    torch, local = T.torch, T.local
    host_batch = np.stack([frames[(i + rank * 3) % len(frames)] for i in range(B)])
    dev_batch = torch.from_numpy(host_batch).cuda()
    dlanes = [D.GpuDetector(W, H, FMT, quad_decimate=DECIMATE, quad_sigma=SIGMA, max_batch=B, device=local) for _ in range(DL)]
    dbatches = [dev_batch] + [dev_batch.clone() for _ in range(DL - 1)]
    dstreams = [torch.cuda.ExternalStream(d.stream, device=torch.device("cuda", local)) for d in dlanes]
    for d, b in zip(dlanes, dbatches):
        for _ in range(max(3, warmup)):
            d.DetectDevice(b.data_ptr(), B)
    det = dlanes[0]
    infos = [det.FrameInfo(f) for f in range(B)]
    assert all(i.status == 0 for i in infos), "device buffer overflow during warm-up"
    e0 = torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]   # lane 0, after each of its batches
    e_end = [torch.cuda.Event(enable_timing=True) for _ in dlanes]
    T.barrier()
    ctx = clocks if clocks is not None else _Null()
    with ctx:
        e0.record(dstreams[0])
        for s_ in range(steps):
            for li, (d, b) in enumerate(zip(dlanes, dbatches)):
                d.EnqueueDevice(b.data_ptr(), B)  # this lane's previous results are collected here
                if li == 0:
                    marks[s_].record(dstreams[0])
        for d, st, ev in zip(dlanes, dstreams, e_end):
            d.Finish()
            ev.record(st)
        T.barrier()
    ms = T.max_ranks(max(e0.elapsed_time(ev) for ev in e_end))
    # per-step spread: lane 0's batch-to-batch intervals (its stream is busy back to back in steady state)
    gaps = [marks[k - 1].elapsed_time(marks[k]) for k in range(1, steps)]
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, dlanes, B)
    for d in dlanes[1:]:
        d.close()
    return det, dev_batch, host_batch, ms, gaps, infos


class _Null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def end_to_end_leg(T: Timing, D, host_batch, frame_bytes, B, L, steps, expect_dets_of, wc=False, clocks=None):
    """`L` detectors (one CUDA stream each) take turns, so lane k's host->device copy overlaps lane k-1's kernels;
    every frame crosses PCIe inside the timed region (one cudaMemcpyAsync per lane batch from one pinned block, as a
    camera ring buffer would be) and its detections are collected on the host before the lane is reused."""
    torch, local = T.torch, T.local
    per_lane = B // L
    lanes = [D.GpuDetector(W, H, FMT, quad_decimate=DECIMATE, quad_sigma=SIGMA, max_batch=per_lane, device=local) for _ in range(L)]
    pinned = D.PinnedBuffer(frame_bytes * B, write_combined=wc)
    pinned.array[:] = host_batch.reshape(-1)
    lane_ptrs = [pinned.ptr + l * per_lane * frame_bytes for l in range(L)]
    for _ in range(3):
        for l, ld in enumerate(lanes):
            ld.EnqueueHostBlock(lane_ptrs[l], per_lane)
    for ld in lanes:
        ld.Finish()
    T.barrier()
    ctx = clocks if clocks is not None else _Null()
    with ctx:
        t0 = time.perf_counter()
        for _ in range(steps):
            for l, ld in enumerate(lanes):
                ld.EnqueueHostBlock(lane_ptrs[l], per_lane)   # waits for + collects this lane's previous batch first
        ndets = 0
        for ld in lanes:
            ld.Finish()
            ndets += sum(len(ld.Detections(f)) for f in range(per_lane))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    dt = T.max_ranks(dt)
    if expect_dets_of is not None:
        assert ndets == sum(len(expect_dets_of.Detections(f)) for f in range(per_lane * L)), "end-to-end path lost detections"
    for ld in lanes:
        ld.close()
    return per_lane * L * steps * T.world / dt, per_lane * L, ndets, pinned


def latency_leg(D, local, pinned, frame_bytes, nframes, iters):
    """One frame at a time: pinned host frame in, detections on the host out (GpuDetector::Detect as the node calls it)."""
    det1 = D.GpuDetector(W, H, FMT, quad_decimate=DECIMATE, quad_sigma=SIGMA, max_batch=1, device=local)
    lat = []
    for i in range(iters + 10):
        t0 = time.perf_counter()
        det1.DetectPointers([pinned.ptr + (i % nframes) * frame_bytes])
        lat.append((time.perf_counter() - t0) * 1e3)
    det1.close()
    lat = np.sort(np.array(lat[10:]))
    return float(lat[len(lat) // 2]), float(lat[int(len(lat) * 0.99)])


def extra_config_leg(T: Timing, D, rank, cfg, steps):
    """BASELINE configs 4 and 5 at N GPUs (reference scaling model: one detector per camera,
    launch_vision.py:231-310).  config 4: camera stream s -> GPU s, one detector + CUDA stream per camera stream;
    config 5: the 4K clutter scene, batch 16 per GPU.  Same engine, same legs, fewer steps."""
    saved = (W, H, FMT, DECIMATE, SIGMA, WORKLOAD, UNIQUE_FRAMES, BATCH, CONFIG)
    select_config(cfg)
    try:
        # config 4: every rank renders ITS camera stream (seeds 4000 + 1000 * stream + frame); config 5: frames 16*gpu ...
        frames = []
        from ros_vision_b200 import synth
        for i in range(UNIQUE_FRAMES):
            idx = (1000 * rank + i) if cfg == 4 else (16 * rank + i)
            frames.append(np.ascontiguousarray(synth.config_frame(cfg, idx)[0]).reshape(-1))
        B = BATCH
        det, dev_batch, host_batch, ms, gaps, infos = device_resident_leg(T, D, rank, frames, B, 2, steps, 3)
        value = B * 2 * steps * T.world / (ms * 1e-3)
        ndet = sum(len(det.Detections(f)) for f in range(B))
        e2e, per_step, _, pinned = end_to_end_leg(T, D, host_batch, frames[0].size, B, 2, steps, det)
        p50, p99 = latency_leg(D, T.local, pinned, frames[0].size, B, 60)
        p50, p99 = T.max_ranks(p50), T.max_ranks(p99)
        pinned.close()
        det.close()
        P = float(np.mean([i.num_points for i in infos]))
        return {"workload": WORKLOAD, "frames_per_batch": B, "streams_per_gpu": 2, "steps": steps, "value": value, "unit": "frames/s",
                "e2e": e2e, "p50_latency_ms": p50, "p99_latency_ms": p99, "latency_note": "max over ranks of each rank's p50 / p99",
                "h2d_bytes_per_frame": int(frames[0].size), "points_per_frame": P, "detections_per_batch": ndet, "n_gpus": T.world,
                "whole_path_hbm_frac": algorithmic_bytes_per_frame(P) * value / T.world / 1e9 / PEAK[0]}
    finally:
        globals().update(dict(zip(("W", "H", "FMT", "DECIMATE", "SIGMA", "WORKLOAD", "UNIQUE_FRAMES", "BATCH", "CONFIG"), saved)))


PEAK = [6650.0, "fallback (B200_PROFILING.md)"]


def load_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        PEAK[0], PEAK[1] = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"


def run_ours(args):
    import torch
    import torch.distributed as dist
    from ros_vision_b200 import detector as D

    rank, world, local = dist_setup(args.gpus)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    numa_cpus = pin_to_gpu_numa_node(local) if world > 1 else None
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    D.load_library()
    load_peak()
    peak, peak_src = PEAK
    T = Timing(torch, dist, world, local)
    frames = make_frames()
    frame_bytes = frames[0].size
    B = args.batch
    DL = max(1, args.device_lanes)
    clocks = ClockSampler(local)

    # --- device-resident throughput (the line's `value`) ------------------------------------------
    det, dev_batch, host_batch, ms, gaps, infos = device_resident_leg(T, D, rank, frames, B, DL, args.steps, args.warmup, clocks,
                                                                      args.dump_outputs)
    value = B * DL * args.steps * world / (ms * 1e-3)
    ndet_per_batch = sum(len(det.Detections(f)) for f in range(B))
    P = float(np.mean([i.num_points for i in infos]))
    Psel = float(np.mean([i.num_selected_points for i in infos]))
    nblobs = float(np.mean([i.num_blobs for i in infos]))
    # points per blob tier (candidate blobs: within the point-count limits), from the blob lists of the distinct frames
    tiers = {"small": 0.0, "medium": 0.0, "large": 0.0}
    nd = min(B, len(frames))
    for f in range(nd):
        cnts = det.CopyStage(D.STAGE_BLOBS, f)["count"].astype(np.int64)
        tiers["small"] += float(cnts[cnts <= SMALL_CAP].sum()) / nd
        tiers["medium"] += float(cnts[(cnts > SMALL_CAP) & (cnts <= MEDIUM_CAP)].sum()) / nd
        tiers["large"] += float(cnts[cnts > MEDIUM_CAP].sum()) / nd
    launches_per_step = det.kernels_per_batch()

    # --- end to end: pinned host frames -> detections on the host (the line's `e2e`) --------------
    L = max(1, args.lanes)
    e2e_value, e2e_frames_per_step, _, pinned = end_to_end_leg(T, D, host_batch, frame_bytes, B, L, args.steps, det, args.wc, clocks)
    d2h = 128 * e2e_frames_per_step + 176 * ndet_per_batch  # counters + detection records written to pinned host memory

    # --- single-frame latency ----------------------------------------------------------------------
    p50, p99 = latency_leg(D, local, pinned, frame_bytes, B, args.latency_iters)
    pinned.close()

    # --- per-kernel times (CUDA events around each launch, kernels serialised on the detector's stream) ----
    prof = det.ProfileDevice(dev_batch.data_ptr(), B, iters=5)
    kern = []
    for name, kms in prof:
        by = kernel_bytes(name, P, tiers) * B
        kern.append({"kernel": name, "ms": kms, "alg_bytes": by, "gbs": (by / (kms * 1e-3) / 1e9) if kms > 0 else None,
                     "frac": (by / (kms * 1e-3) / 1e9 / peak) if kms > 0 else None})
    step_kernel_ms = sum(k["ms"] for k in kern)
    fe = [k for k in kern if k["kernel"] in FRONT_END]
    fe_ms, fe_bytes = sum(k["ms"] for k in fe), sum(k["alg_bytes"] for k in fe)
    # The headline kernel is the SLOWEST FRONT-END kernel (the front end is what the HBM roofline is about; the
    # per-blob kernels are latency / issue bound and are reported with their issue-slot utilisation instead).
    dom = max(fe, key=lambda k: k["ms"])
    ncu = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        ncu = json.load(open(tpath))
    t = ncu.get(dom["kernel"]) if B == BATCH else None
    traffic = (t["dram_read_bytes"] + t["dram_write_bytes"]) if t else None
    traffic_src = f"profiles/summary_{t['tag']}.md ({t['report']})" if t else None
    for k in kern:
        e = ncu.get(k["kernel"])
        if e and "issue_active_pct" in e:
            k["ncu_issue_active_pct"] = e["issue_active_pct"]
            k["ncu_dram_bytes"] = e["dram_read_bytes"] + e["dram_write_bytes"]
    b_frame = algorithmic_bytes_per_frame(P)
    roof = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["gbs"], "peak": peak, "unit": "GB/s",
            "frac": dom["frac"], "traffic": traffic, "traffic_source": traffic_src,
            "alg_bytes_per_launch": dom["alg_bytes"], "peak_source": peak_src,
            "share_of_step": dom["ms"] / step_kernel_ms if step_kernel_ms else None,
            "selection": "slowest front-end kernel by CUDA-event time (per-blob kernels are not HBM bound)",
            "whole_path": {"alg_bytes_per_frame": b_frame,
                           "achieved": b_frame * B * DL / (ms / args.steps * 1e-3) / 1e9,
                           "frac": b_frame * B * DL / (ms / args.steps * 1e-3) / 1e9 / peak},
            "front_end": {"kernels": [k["kernel"] for k in fe], "ms": fe_ms, "alg_bytes": fe_bytes,
                          "achieved": fe_bytes / (fe_ms * 1e-3) / 1e9 if fe_ms else None,
                          "frac": fe_bytes / (fe_ms * 1e-3) / 1e9 / peak if fe_ms else None,
                          "compulsory": {"alg_bytes": b_frame * B, "what": "B_frame of SURVEY 8(d): every array once",
                                         "frac": b_frame * B / (fe_ms * 1e-3) / 1e9 / peak if fe_ms else None}},
            "note": "per-kernel times are CUDA events around each launch with the kernels serialised on one stream; in the "
                    "timed run the fit kernels overlap on side streams.  fit_*, quads and decode are latency / issue bound: "
                    "their alg_bytes is the 4-byte segment point they read, ncu_issue_active_pct (profiles/traffic.json) is "
                    "the figure that describes them.",
            "kernels": kern}
    det.close()
    del dev_batch

    # --- the other multi-GPU BASELINE configs and the MJPG input path, at this N -------------------
    extra = {}
    if not args.no_extra and CONFIG == 2 and FMT == "yuyv":
        for cfg in (4, 5):
            try:
                extra[f"config{cfg}"] = extra_config_leg(T, D, rank, cfg, max(3, args.steps // 8))
            except Exception as e:  # noqa: BLE001 -- reporting legs never cost the contract line (all ranks fail alike or not at all)
                extra[f"config{cfg}"] = {"error": f"{type(e).__name__}: {e}"}
        try:
            extra["e2e_mjpg"] = mjpg_leg(local, rank, world)
        except Exception as e:  # noqa: BLE001
            extra["e2e_mjpg"] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        solo = world == 1 and not args.no_cpu
        g = np.array(gaps) if gaps else np.array([ms / args.steps])
        line = {
            "metric": "frames/s", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": B * DL, "frames_per_batch": B, "streams_per_gpu": DL,
                       "distinct_frames": len(frames),
                       "l2": f"inputs ({frame_bytes * B / 1e6:.0f} MB/step/GPU) and intermediates exceed the 126 MB L2; no explicit flush",
                       "sharding": "frames by rank, no collective",
                       "cpu_affinity": (f"rank 0 on {len(numa_cpus)} cores next to its GPU (NVML ideal CPU set)" if numa_cpus else "unchanged")},
            "step_stats": {"what": "rank 0, stream 0: interval between consecutive batches of one lane (one step), ms",
                           "min": float(g.min()), "median": float(np.median(g)), "max": float(g.max()), "n": int(g.size)},
            "p50_latency_ms": p50, "p99_latency_ms": p99,
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": frame_bytes * e2e_frames_per_step,
                    "d2h_bytes_per_step": d2h, "lanes": L},
            "gpu_launches": launches_per_step * args.steps * DL,
            "roofline": roof,
            "cpu_baseline": safe_leg(cpu_baseline, frames) if solo else None,
            "reference_gpu": safe_leg(reference_gpu_leg, frames) if (solo and CONFIG in (2, 4)) else None,
            "cpu_opencv_aruco": safe_leg(opencv_aruco_leg, frames) if solo else None,
            "e2e_mjpg": extra.pop("e2e_mjpg", None),
            "extra": extra,
            "clocks": clocks.summary(),
            "stats": {"points_per_frame": P, "selected_points_per_frame": Psel, "blobs_per_frame": nblobs, "candidate_points_by_tier": tiers,
                      "detections_per_batch": ndet_per_batch},
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--latency-iters", type=int, default=200)
    ap.add_argument("--lanes", type=int, default=2, help="detector instances (CUDA streams) used by the end-to-end leg")
    ap.add_argument("--device-lanes", type=int, default=2,
                    help="detector instances (CUDA streams) taking turns in the device-resident leg")
    ap.add_argument("--wc", action="store_true", help="write-combined pinned frame buffer in the end-to-end leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU / reference-GPU reporting legs (profiling runs)")
    ap.add_argument("--no-extra", action="store_true", help="skip the config 4 / config 5 / MJPG legs (profiling runs)")
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5],
                    help="BASELINE.json config to measure; the contract line is config 2 (the default)")
    ap.add_argument("--format", default=None, choices=["gray", "yuyv", "bgr"],
                    help="pixel format of the frames (default: the config's own; the contract line is YUYV)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the device-resident leg's results of its last step (rank 0, every lane) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    select_config(args.config)
    if args.format:
        global FMT, WORKLOAD
        if args.format != FMT:
            WORKLOAD += f" [frames delivered as {args.format}]"
        FMT = args.format
    if args.batch == 128 and args.config != 2:
        args.batch = BATCH
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
