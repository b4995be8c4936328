#!/usr/bin/env python3
"""What the device pose step (GpuDetector.SetPoseEstimation) costs, on config 2 (bench.py's workload:
synth.config_frame(2, i), 1280x800 YUYV, 1-6 tags per frame), in one run on one GPU:

  * device-resident frames/s of 128-frame batches with the pose step off and on, alternating in the same run;
  * single-frame latency (pinned host frame in -> detections and poses out), p50, off and on, alternating;
  * the `pose` kernel's device time per 128-frame batch (b200tag_profile_device);
  * the host time of b200tag_locate_tags on the same detections, on one CPU core of the same machine.

--method ippe measures the IPPE method instead (SetPoseEstimation(..., method="ippe"), the `pose_ippe` kernel), and the
host leg times estimate_poses(..., method="ippe") against estimate_poses with the default method on the same
detections.

--field measures the field pose step (GpuDetector.SetFieldLayout, the `field_pose` kernel) on top of IPPE:
  * frames/s of 128-frame batches and single-frame p50 for three arms alternating in the same run: pose off, IPPE on,
    IPPE + field (a layout holding every tag36h11 id, so every detection takes part);
  * the `field_pose` kernel's device time per 128-frame batch on two workloads: config-2 frames with that all-ids
    layout (geometry that fits no frame, so Levenberg-Marquardt runs to its cap: the worst case), and synth.field_scene
    frames of one 6-tag layout seen from 16 robot poses (consistent geometry);
  * the host estimate_field_pose per field_scene frame on one CPU core.

Prints one JSON record, and writes it to --out when given.  Needs a CUDA device."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TAGSIZE = 0.1651
FX, FY, CX, CY = 905.5, 907.9, 640.0, 400.0
ROTATION = [[0, 0, 1], [-1, 0, 0], [0, -1, 0]]
OFFSET = [0.1, -0.2, 0.5]
BATCH, UNIQUE = 128, 16


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=6, help="alternations of the off / on measurements")
    ap.add_argument("--steps", type=int, default=40, help="128-frame batches per throughput measurement")
    ap.add_argument("--latency-iters", type=int, default=400, help="single frames per latency measurement")
    ap.add_argument("--method", choices=("oi", "ippe"), default="oi", help="pose method of the device step")
    ap.add_argument("--field", action="store_true", help="measure the field pose step (IPPE + SetFieldLayout)")
    ap.add_argument("--out", help="also write the JSON to this file (e.g. profiles/pose_r03.json)")
    args = ap.parse_args()
    if args.field:
        return field_main(args)

    import torch
    from ros_vision_b200 import detector as D, synth
    frames = [np.ascontiguousarray(synth.config_frame(2, i)[0]).reshape(-1) for i in range(UNIQUE)]
    host_batch = np.stack([frames[i % UNIQUE] for i in range(BATCH)])
    dev_batch = torch.from_numpy(host_batch).cuda()
    ptr = dev_batch.data_ptr()

    def detector(pose, max_batch):
        d = D.GpuDetector(1280, 800, "yuyv", quad_decimate=2, max_batch=max_batch)
        if pose:
            d.SetPoseEstimation(TAGSIZE, FX, FY, CX, CY, rotation=ROTATION, offset=OFFSET, method=args.method)
        return d

    # throughput: 128-frame device-resident batches, off and on alternating
    big = {False: detector(False, BATCH), True: detector(True, BATCH)}
    for d in big.values():
        for _ in range(5):
            d.DetectDevice(ptr, BATCH)
    fps = {False: [], True: []}
    for _ in range(args.rounds):
        for pose in (False, True):
            d = big[pose]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                d.DetectDevice(ptr, BATCH)
            fps[pose].append(BATCH * args.steps / (time.perf_counter() - t0))
    dets_per_batch = sum(len(big[True].Detections(f)) for f in range(BATCH))
    raw_per_batch = sum(int(big[True].FrameInfo(f).num_detections) for f in range(BATCH))

    # the pose kernel's device time per batch
    prof = big[True].ProfileDevice(ptr, BATCH, iters=20)
    kernel = "pose" if args.method == "oi" else "pose_ippe"
    pose_ms = [ms for name, ms in prof if name == kernel]
    total_ms = sum(ms for _, ms in prof)

    # single-frame latency from a pinned host frame, off and on alternating over the 16 frames
    one = {False: detector(False, 1), True: detector(True, 1)}
    pins = []
    for f in frames:
        pb = D.PinnedBuffer(f.size)
        pb.array[:] = f
        pins.append(pb)
    lat = {False: [], True: []}
    for d in one.values():
        for pb in pins:
            d.DetectPointers([pb.ptr])
    for i in range(args.latency_iters):
        pb = pins[i % UNIQUE]
        for pose in ((False, True) if i % 2 == 0 else (True, False)):
            t0 = time.perf_counter()
            one[pose].DetectPointers([pb.ptr])
            lat[pose].append((time.perf_counter() - t0) * 1e6)

    # the host step on the same detections, one core: the median of 20 calls per frame
    per_frame_dets = []
    for pb_i in range(UNIQUE):
        one[False].DetectPointers([pins[pb_i].ptr])
        per_frame_dets.append(one[False].Detections(0))
    n_dets = [len(d) for d in per_frame_dets]
    cpu = sorted(os.sched_getaffinity(0))[0]
    saved = os.sched_getaffinity(0)

    def host_leg(step):
        os.sched_setaffinity(0, {cpu})
        host_us = []
        try:
            for dets in per_frame_dets:
                step(dets)
                reps = []
                for _ in range(20):
                    t0 = time.perf_counter()
                    step(dets)
                    reps.append((time.perf_counter() - t0) * 1e6)
                host_us.append(float(np.median(reps)))
        finally:
            os.sched_setaffinity(0, saved)
        return {"per_frame": host_us, "detections": n_dets, "median": float(np.median(host_us)),
                "us_per_detection": float(sum(host_us) / max(1, sum(n_dets))), "cpu": cpu}

    p50 = {k: float(np.percentile(v, 50)) for k, v in lat.items()}
    ratio = float(np.median(fps[True]) / np.median(fps[False]))
    if args.method == "oi":
        host = {"host_locate_tags_us_per_frame": host_leg(lambda d: D.locate_tags(d, TAGSIZE, FX, FY, CX, CY, ROTATION, OFFSET))}
        host_frame_p50 = host["host_locate_tags_us_per_frame"]["median"]
        targets = {"batch_ratio_at_least_0.95": bool(ratio >= 0.95),
                   "p50_on_below_p50_off_plus_host_pose": bool(p50[True] < p50[False] + host_frame_p50)}
    else:
        host = {"host_estimate_poses_ippe_us_per_frame": host_leg(lambda d: D.estimate_poses(d, TAGSIZE, FX, FY, CX, CY, method="ippe")),
                "host_estimate_poses_oi_us_per_frame": host_leg(lambda d: D.estimate_poses(d, TAGSIZE, FX, FY, CX, CY))}
        ippe_us = host["host_estimate_poses_ippe_us_per_frame"]["us_per_detection"]
        oi_us = host["host_estimate_poses_oi_us_per_frame"]["us_per_detection"]
        targets = {"batch_ratio_at_least_0.95": bool(ratio >= 0.95),
                   "p50_on_at_most_p50_off_plus_20us": bool(p50[True] <= p50[False] + 20),
                   "pose_kernel_at_most_0.05ms_per_batch": bool(pose_ms and pose_ms[0] <= 0.05),
                   "host_ippe_at_least_10x_cheaper_than_host_oi": bool(10 * ippe_us <= oi_us)}
    res = {
        "method": args.method,
        "gpu": gpu_identity(),
        "torch_device": torch.cuda.get_device_name(0),
        "workload": "config2: 1280x800 YUYV, synth.config_frame(2, 0..15) tiled to 128-frame batches, tag36h11, decimate 2",
        "batch_frames_per_s": {"pose_off": fps[False], "pose_on": fps[True],
                               "median_off": float(np.median(fps[False])), "median_on": float(np.median(fps[True])),
                               "ratio_on_over_off": ratio},
        "detections_per_batch": dets_per_batch, "raw_detections_per_batch": raw_per_batch,
        "pose_kernel_ms_per_batch": pose_ms[0] if pose_ms else None,
        "all_kernels_ms_per_batch_serial": total_ms,
        "single_frame_latency_us": {"p50_off": p50[False], "p50_on": p50[True], "p90_off": float(np.percentile(lat[False], 90)),
                                    "p90_on": float(np.percentile(lat[True], 90)), "iters": args.latency_iters},
        **host,
        "targets": targets,
    }
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    for d in list(big.values()) + list(one.values()):
        d.close()
    for pb in pins:
        pb.close()


def all_ids_layout(D, seed=1):
    """Every tag36h11 id at a random field pose."""
    from ros_vision_b200.field_layout import quaternion_matrix
    rng = np.random.default_rng(seed)
    lay = np.zeros(587, dtype=D.FIELD_TAG_DT)
    lay["id"] = np.arange(587)
    for i in range(587):
        lay["R"][i] = quaternion_matrix(*rng.normal(size=4))
        lay["t"][i] = rng.uniform(-8, 8, size=3)
    return lay


def field_frames(D, synth, n):
    """One layout of 6 tags 1.5-4 m in front of a nominal robot pose, and `n` field_scene frames (YUYV) from robot poses
    within 0.3 m / 5 deg of it."""
    rng = np.random.default_rng(6)
    R0 = np.array(ROTATION, dtype=np.float64)
    lay = np.zeros(6, dtype=D.FIELD_TAG_DT)
    lay["id"] = rng.choice(587, 6, replace=False)
    for j in range(6):
        z = rng.uniform(1.5, 4.0)
        a = rng.uniform(-0.4, 0.4, size=3)
        Rx = np.array([[1, 0, 0], [0, np.cos(a[0]), -np.sin(a[0])], [0, np.sin(a[0]), np.cos(a[0])]])
        Ry = np.array([[np.cos(a[1]), 0, np.sin(a[1])], [0, 1, 0], [-np.sin(a[1]), 0, np.cos(a[1])]])
        lay["R"][j] = R0 @ Ry @ Rx
        lay["t"][j] = R0 @ np.array([rng.uniform(-0.3, 0.3) * z, rng.uniform(-0.2, 0.2) * z, z]) + [0, 0, 0.6]
    frames = []
    for i in range(n):
        yaw = np.radians(rng.uniform(-5, 5))
        Rz = np.array([[np.cos(yaw), -np.sin(yaw), 0], [np.sin(yaw), np.cos(yaw), 0], [0, 0, 1]])
        t = np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3), 0.6])
        sc = synth.field_scene(1280, 800, lay, TAGSIZE, Rz @ R0, t, FX, FY, CX, CY, seed=i, noise_sigma=4.0)
        frames.append(np.ascontiguousarray(synth.gray_to_yuyv(sc.gray)).reshape(-1))
    return lay, frames


def field_main(args):
    import torch
    from ros_vision_b200 import detector as D, synth
    arms = ("pose_off", "ippe", "ippe_field")
    lay_all = all_ids_layout(D)
    frames = [np.ascontiguousarray(synth.config_frame(2, i)[0]).reshape(-1) for i in range(UNIQUE)]
    dev_batch = torch.from_numpy(np.stack([frames[i % UNIQUE] for i in range(BATCH)])).cuda()
    ptr = dev_batch.data_ptr()
    fs_lay, fs_frames = field_frames(D, synth, UNIQUE)
    fs_batch = torch.from_numpy(np.stack([fs_frames[i % UNIQUE] for i in range(BATCH)])).cuda()

    def detector(arm, max_batch, lay=lay_all):
        d = D.GpuDetector(1280, 800, "yuyv", quad_decimate=2, max_batch=max_batch)
        if arm != "pose_off":
            d.SetPoseEstimation(TAGSIZE, FX, FY, CX, CY, rotation=ROTATION, offset=OFFSET, method="ippe")
        if arm == "ippe_field":
            d.SetFieldLayout(lay)
        return d

    big = {a: detector(a, BATCH) for a in arms}
    for d in big.values():
        for _ in range(5):
            d.DetectDevice(ptr, BATCH)
    fps = {a: [] for a in arms}
    for _ in range(args.rounds):
        for a in arms:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                big[a].DetectDevice(ptr, BATCH)
            fps[a].append(BATCH * args.steps / (time.perf_counter() - t0))
    kpb = {a: big[a].kernels_per_batch() for a in arms}
    raw_per_batch = sum(int(big["ippe_field"].FrameInfo(f).num_detections) for f in range(BATCH))
    used_cfg2 = [int(big["ippe_field"].FieldPose(f)["num_tags"]) for f in range(BATCH)]
    iters_cfg2 = [int(big["ippe_field"].FieldPose(f)["iterations"]) for f in range(BATCH)]

    def kernel_ms(det, p):
        prof = det.ProfileDevice(p, BATCH, iters=20)
        return [ms for name, ms in prof if name == "field_pose"][0]

    worst_ms = kernel_ms(big["ippe_field"], ptr)
    fs_det = detector("ippe_field", BATCH, fs_lay)
    fs_det.DetectDevice(fs_batch.data_ptr(), BATCH)
    fs_used = [int(fs_det.FieldPose(f)["num_tags"]) for f in range(BATCH)]
    fs_iters = [int(fs_det.FieldPose(f)["iterations"]) for f in range(BATCH)]
    fs_ms = kernel_ms(fs_det, fs_batch.data_ptr())

    # single-frame latency from a pinned host frame, the three arms in rotating order
    one = {a: detector(a, 1) for a in arms}
    pins = []
    for f in frames:
        pb = D.PinnedBuffer(f.size)
        pb.array[:] = f
        pins.append(pb)
    for d in one.values():
        for pb in pins:
            d.DetectPointers([pb.ptr])
    lat = {a: [] for a in arms}
    for i in range(args.latency_iters):
        pb = pins[i % UNIQUE]
        for k in range(3):
            a = arms[(i + k) % 3]
            t0 = time.perf_counter()
            one[a].DetectPointers([pb.ptr])
            lat[a].append((time.perf_counter() - t0) * 1e6)

    # the host solve on the field_scene frames' detections, one core: the median of 20 calls per frame
    fs_one = detector("ippe", 1)
    per_frame = []
    for f in fs_frames:
        fs_one.Detect(f)
        per_frame.append(fs_one.Detections(0))
    cpu = sorted(os.sched_getaffinity(0))[0]
    saved = os.sched_getaffinity(0)
    host_us = []
    os.sched_setaffinity(0, {cpu})
    try:
        for dets in per_frame:
            reps = []
            for _ in range(21):
                t0 = time.perf_counter()
                D.estimate_field_pose(dets, fs_lay, TAGSIZE, FX, FY, CX, CY, ROTATION, OFFSET)
                reps.append((time.perf_counter() - t0) * 1e6)
            host_us.append(float(np.median(reps[1:])))
    finally:
        os.sched_setaffinity(0, saved)

    med = {a: float(np.median(fps[a])) for a in arms}
    p50 = {a: float(np.percentile(lat[a], 50)) for a in arms}
    ratio = med["ippe_field"] / med["pose_off"]
    res = {
        "mode": "field",
        "gpu": gpu_identity(),
        "torch_device": torch.cuda.get_device_name(0),
        "workload": "config2: 1280x800 YUYV, synth.config_frame(2, 0..15) tiled to 128-frame batches, tag36h11, decimate 2; "
                    "field arm: layout with all 587 tag36h11 ids at random field poses",
        "batch_frames_per_s": {"rounds": fps, "median": med, "ratio_ippe_field_over_off": ratio,
                               "ratio_ippe_field_over_ippe": med["ippe_field"] / med["ippe"]},
        "kernels_per_batch": kpb,
        "single_frame_latency_us": {"p50": p50, "p90": {a: float(np.percentile(lat[a], 90)) for a in arms},
                                    "iters": args.latency_iters},
        "field_pose_kernel_ms_per_batch": {
            "config2_all_ids_layout": worst_ms, "config2_raw_detections_per_batch": raw_per_batch,
            "config2_tags_used_per_batch": sum(used_cfg2), "config2_max_iterations": max(iters_cfg2),
            "field_scene": fs_ms, "field_scene_tags_used_per_batch": sum(fs_used),
            "field_scene_iterations_median": float(np.median(fs_iters))},
        "host_estimate_field_pose_us_per_frame": {"per_frame": host_us, "median": float(np.median(host_us)),
                                                  "tags": [int(len(d)) for d in per_frame], "cpu": cpu},
        "targets": {"batch_ratio_at_least_0.95": bool(ratio >= 0.95),
                    "p50_field_at_most_p50_ippe_plus_40us": bool(p50["ippe_field"] <= p50["ippe"] + 40),
                    "field_kernel_worst_at_most_0.1ms_per_batch": bool(worst_ms <= 0.1)},
    }
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))
    for d in list(big.values()) + list(one.values()) + [fs_det, fs_one]:
        d.close()
    for pb in pins:
        pb.close()


if __name__ == "__main__":
    main()
