"""The floor pose on the device (b200tag_set_floor_pose, k_floor_pose): bit-identical to the host's
b200tag_estimate_floor_pose on hook inputs and real frames, per-frame gyro headings and their lifetime, the other
results unchanged, and accuracy on rendered field scenes."""
import ctypes as C
import math

import numpy as np
import pytest

import pose_records as PR
from test_floor_pose import WEIGHT, WIDE, wrap
from test_gpu_field_pose import (OFFSET, ROTATION, all_ids_layout, field_case, frames_of, intrinsics, raw_list)

pytestmark = pytest.mark.gpu

TAGSIZE = PR.TAGSIZE
SIGMA = 0.3
E_INVALID = -1


@pytest.fixture(scope="module")
def D():
    from ros_vision_b200 import build, detector
    build.build_native()
    detector.load_library()
    return detector


def check_floor(D, det, f, lay, params, heading=np.nan, weight=np.inf, distortion=None, sigma=0.0):
    """FloorPose(f) (and FloorCovariance(f)) bit-identical to the host solve on Detections(f); the field pose's tag
    count equal to the floor pose's."""
    got = det.FloorPose(f)
    want, cov = D.estimate_floor_pose(det.Detections(f), lay, *params, rotation=ROTATION, offset=OFFSET, heading=heading,
                                      heading_weight=weight, distortion=distortion, sigma=sigma)
    assert got is not None and got.tobytes() == want.tobytes(), (f, got, want)
    assert got["num_tags"] == det.FieldPose(f)["num_tags"]
    if sigma > 0:
        assert det.FloorCovariance(f).tobytes() == cov.tobytes()
    else:
        assert det.FloorCovariance(f) is None
    return got


def test_hook_is_bit_identical_to_the_host(D):
    rng = np.random.default_rng(31)
    params = (TAGSIZE, 905.5, 907.9, 640.0, 400.0)
    lays = [all_ids_layout(D, 1, 40)]
    for k in range(3):
        lay = np.zeros(30, dtype=D.FIELD_TAG_DT)
        lay["id"] = rng.choice(587, 30, replace=False)
        lay["family"] = rng.integers(0, 2, size=30)
        for j in range(30):
            lay["R"][j] = PR.rot(*rng.uniform(-0.5, 0.5, size=3))
            lay["t"][j] = [rng.uniform(-1.5, 1.5), rng.uniform(-1, 1), rng.uniform(1.0, 6.0)]
        lays.append(lay)
    counts = {"empty": 0, "one": 0, "many": 0}
    modes = {0: 0, 1: 0, 2: 0}
    for trial in range(3000):
        lay = lays[trial % len(lays)]
        raw = raw_list(D, rng, lay, params)
        rot = PR.rot(*rng.uniform(-1, 1, size=3)) if trial % 2 else None
        off = rng.uniform(-1, 1, size=3) if trial % 2 else None
        heading = np.nan if trial % 3 == 0 else rng.uniform(-4, 4)
        weight = np.inf if trial % 3 == 1 else rng.uniform(0.5, 50)
        kw = dict(rotation=rot, offset=off, heading=heading, heading_weight=weight,
                  distortion=WIDE if trial % 4 >= 2 else None, sigma=SIGMA if trial % 5 < 3 else 0.0)
        host, hc = D.estimate_floor_pose(raw, lay, *params, **kw)
        dev, dc = D.estimate_floor_pose_device(raw, lay, *params, **kw)
        assert dev.tobytes() == host.tobytes(), trial
        assert (hc is None and dc is None) or hc.tobytes() == dc.tobytes(), trial
        counts["empty" if host["num_tags"] == 0 else "one" if host["num_tags"] == 1 else "many"] += 1
        modes[int(host["mode"])] += 1
    assert min(counts.values()) >= 100 and min(modes.values()) >= 500, (counts, modes)


@pytest.mark.parametrize("cfg,n", [(2, 16), (4, 4), (5, 2)])
def test_config_frames(D, cfg, n):
    frames, fmt, w, h, dec, sigma = frames_of(cfg, n)
    params = (TAGSIZE, *intrinsics(w, h))
    lay = all_ids_layout(D, cfg)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=n)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    det.SetFieldLayout(lay)
    rng = np.random.default_rng(cfg)
    for weight, sig, dist in ((np.inf, 0.0, None), (WEIGHT, SIGMA, None), (np.inf, SIGMA, WIDE)):
        det.SetFloorPose(weight)
        det.SetPoseCovariance(sig)
        det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe", distortion=dist)
        for _ in range(2):  # the second call replays the captured graph
            heads = np.where(rng.uniform(size=n) < 0.3, np.nan, rng.uniform(-np.pi, np.pi, size=n))
            det.SetRobotHeadings(heads[: n - 1])  # the last frame has none
            det.DetectBatch(frames)
            for f in range(n):
                got = check_floor(D, det, f, lay, params, heads[f] if f < n - 1 else np.nan, weight, dist, sig)
                assert got["mode"] == (0 if f == n - 1 or np.isnan(heads[f]) else 1 if weight < np.inf else 2)
    det.close()


def test_mjpg_frame(D):
    cv2 = pytest.importorskip("cv2")
    w, h = 1280, 800
    params = (TAGSIZE, 905.5, 907.9, 640.0, 400.0)
    lay, sc, cR, ct = field_case(D, 5, w, h, params)
    ok, buf = cv2.imencode(".jpg", sc.gray, [cv2.IMWRITE_JPEG_QUALITY, 90])
    det = D.GpuDetector(w, h, "gray", quad_decimate=2)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    det.SetFieldLayout(lay)
    det.SetFloorPose(WEIGHT)
    yaw = math.atan2(cR[1, 2], cR[0, 2])
    det.SetRobotHeadings([yaw])
    det.DetectMjpg([buf.tobytes()])
    assert check_floor(D, det, 0, lay, params, yaw, WEIGHT)["num_tags"] >= 3
    det.close()


def test_heading_lifetime(D):
    frames, fmt, w, h, dec, sigma = frames_of(2, 4)
    params = (TAGSIZE, *intrinsics(w, h))
    lay = all_ids_layout(D, 2)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=4)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    det.SetFieldLayout(lay)
    det.SetFloorPose(np.inf)
    a, b = [0.1, 0.2, 0.3, 0.4], [-1.0, np.nan, 2.0]
    det.SetRobotHeadings(a)
    det.DetectBatch(frames)
    for f in range(4):
        assert check_floor(D, det, f, lay, params, a[f])["mode"] == 2
    # the next call without a new set runs in free mode
    det.DetectBatch(frames)
    for f in range(4):
        assert check_floor(D, det, f, lay, params)["mode"] == 0
    # headings set while a batch is in flight belong to the next call
    ptrs = [fr.ctypes.data for fr in frames]
    det.SetRobotHeadings(a)
    det.EnqueuePointers(ptrs)
    det.SetRobotHeadings(b)
    det.Finish()
    for f in range(4):
        check_floor(D, det, f, lay, params, a[f])
    det.DetectBatch(frames)
    for f in range(4):
        check_floor(D, det, f, lay, params, b[f] if f < 3 else np.nan)
    # rejected: more headings than max_batch, an infinite heading, NULL with a count; the pending set is kept
    det.SetRobotHeadings(a)
    lib = D.load_library()
    five = np.zeros(5)
    assert lib.b200tag_set_robot_headings(det._h, five.ctypes.data_as(C.c_void_p), 5) == E_INVALID
    for bad in (np.inf, -np.inf):
        arr = np.array([0.0, bad])
        assert lib.b200tag_set_robot_headings(det._h, arr.ctypes.data_as(C.c_void_p), 2) == E_INVALID
    assert lib.b200tag_set_robot_headings(det._h, None, 2) == E_INVALID
    assert lib.b200tag_set_robot_headings(det._h, None, -1) == E_INVALID
    det.DetectBatch(frames)
    for f in range(4):
        check_floor(D, det, f, lay, params, a[f])
    for bad in (-1.0, np.nan, -np.inf):
        assert lib.b200tag_set_floor_pose(det._h, bad) == E_INVALID
    det.DetectBatch(frames)
    assert det.FloorPose(0)["mode"] == 0  # still on, with the weight it had
    det.close()


def _results(det, n):
    out = []
    for f in range(n):
        fc = det.FieldCovariance(f)
        out.append((det.Detections(f).tobytes(), det.Poses(f).tobytes(), det.TagPositions(f).tobytes(),
                    det.FieldPose(f).tobytes(), det.PoseCovariances(f).tobytes(), None if fc is None else fc.tobytes()))
    return out


@pytest.mark.parametrize("sig", [0.0, SIGMA])
def test_switching_leaves_the_other_results(D, sig):
    frames, fmt, w, h, dec, sigma = frames_of(2, 8)
    params = (TAGSIZE, *intrinsics(w, h))
    lay = all_ids_layout(D, 11)
    plain = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    for d in (plain, det):
        d.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
        d.SetFieldLayout(lay)
        d.SetPoseCovariance(sig)
    heads = np.linspace(-3, 3, 8)
    for weight in (0.0, np.inf, 0.0, WEIGHT, 0.0):
        det.SetFloorPose(weight)
        for _ in range(2):
            det.SetRobotHeadings(heads)
            plain.DetectBatch(frames)
            det.DetectBatch(frames)
            assert _results(det, 8) == _results(plain, 8)
            if weight == 0:
                assert det.FloorPose(0) is None and det.kernels_per_batch() == plain.kernels_per_batch()
            else:
                assert det.kernels_per_batch() == plain.kernels_per_batch() + 1
                for f in range(8):
                    check_floor(D, det, f, lay, params, heads[f], weight, sigma=sig)
    # without the field step there is no floor step
    det.SetFloorPose(np.inf)
    det.SetFieldLayout(None)
    plain.SetFieldLayout(None)
    det.DetectBatch(frames)
    plain.DetectBatch(frames)
    assert det.FloorPose(0) is None and det.kernels_per_batch() == plain.kernels_per_batch()
    plain.close()
    det.close()


def test_field_scene_frames(D):
    """On rendered field scenes the fixed-heading floor pose is within 1 cm of the robot, the free heading within 0.1 deg."""
    w, h = 1280, 800
    params = (TAGSIZE, 905.5, 907.9, 640.0, 400.0)
    det = D.GpuDetector(w, h, "gray", quad_decimate=2)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    det.SetFloorPose(np.inf)
    worst = [0.0, 0.0]
    for i in range(8):
        lay, sc, cR, ct = field_case(D, 100 + i, w, h, params)
        yaw = math.atan2(cR[1, 2], cR[0, 2])  # the camera looks along the robot's +x
        xy = (ct - (np.array([[np.cos(yaw), -np.sin(yaw), 0], [np.sin(yaw), np.cos(yaw), 0], [0, 0, 1]]) @ OFFSET))[:2]
        det.SetFieldLayout(lay)
        det.SetRobotHeadings([yaw])
        det.Detect(sc.gray)
        fixed = check_floor(D, det, 0, lay, params, yaw)
        det.Detect(sc.gray)
        free = check_floor(D, det, 0, lay, params)
        d = float(np.hypot(fixed["x"] - xy[0], fixed["y"] - xy[1]))
        a = abs(np.degrees(wrap(free["heading"] - yaw)))
        worst = [max(worst[0], d), max(worst[1], a)]
        assert fixed["num_tags"] >= 3 and d <= 0.01 and a <= 0.1, (i, d, a)
    print(f"worst field_scene floor error: fixed {worst[0] * 100:.3f} cm, free heading {worst[1]:.4f} deg")
    det.close()
