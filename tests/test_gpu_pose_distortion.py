"""Lens distortion in the device pose steps (GpuDetector.SetPoseEstimation(..., distortion=...), the kDistorted variants
of k_pose, k_pose_ippe and k_field_pose) against the host functions they share their arithmetic with, and end to end on
frames rendered through a wide-angle lens."""
import ctypes as C
import functools

import numpy as np
import pytest

import pose_records as PR
from test_gpu_field_pose import all_ids_layout, raw_list
from test_gpu_pose import assert_poses_match
from test_gpu_pose_ippe import expected_positions

pytestmark = pytest.mark.gpu

TAGSIZE = 0.1651
ROTATION = np.array([[0.0, 0, 1], [-1, 0, 0], [0, -1, 0]])  # camera looking along the robot's +x
OFFSET = np.array([0.25, -0.1, 0.6])
WIDE = (-0.28, 0.08, 0.0006, 0.0, -0.01)
REFERENCE = (0.059238, -0.075154, -0.003801, 0.001113, 0.0)
TANGENTIAL = (0.0, 0.0, 0.002, -0.003, 0.0)
MODELS = (WIDE, REFERENCE, TANGENTIAL)


@pytest.fixture(scope="module")
def D():
    from ros_vision_b200 import build, detector
    build.build_native()
    detector.load_library()
    return detector


def intrinsics(w, h):
    return 0.9 * w, 0.9 * w + 1.5, w / 2 - 3.25, h / 2 + 2.5  # fx, fy, cx, cy


@functools.lru_cache(maxsize=None)
def frames_of(cfg, n):
    from ros_vision_b200 import synth
    out = [synth.config_frame(cfg, i) for i in range(n)]
    frame, fmt, w, h, dec, sigma, _ = out[0]
    return [np.ascontiguousarray(o[0]).reshape(-1) for o in out], fmt, w, h, dec, sigma


def past_the_fold(recs, every=7):
    """Every `every`-th record with corner 2 moved 3 focal lengths right of the centre: past the fold of WIDE and
    REFERENCE, so those records fail there."""
    out = recs.copy()
    out["p"][::every, 2] = (PR.CX + 3.0 * PR.FX, PR.CY + 0.5 * PR.FY)
    return out


@pytest.mark.parametrize("k", range(len(MODELS)))
def test_pose_hooks_equal_the_host(D, k):
    dist = MODELS[k]
    recs = past_the_fold(PR.records(20000, 60 + k))
    params = (PR.TAGSIZE, PR.FX, PR.FY, PR.CX, PR.CY)
    host = D.estimate_poses(recs, *params, method="ippe", distortion=dist)
    dev = D.estimate_poses_device(recs, *params, method="ippe", distortion=dist)
    assert dev.tobytes() == host.tobytes()
    assert np.isinf(host["err"]).sum() >= len(recs) // 7  # the failing corners and the collapsed quads
    host = D.estimate_poses(recs, *params, distortion=dist)
    dev = D.estimate_poses_device(recs, *params, distortion=dist)
    assert_poses_match(dev, host)
    failed = np.isinf(host["err"]) & np.isinf(host["err_other"])
    assert failed.sum() >= len(recs) // 7 and (host["R"][failed] == np.eye(3)).all()


def test_field_hook_equals_the_host(D):
    rng = np.random.default_rng(61)
    params = (TAGSIZE, PR.FX, PR.FY, PR.CX, PR.CY)
    lays = [all_ids_layout(D, 3, 40)]
    for _ in range(3):
        lay = np.zeros(30, dtype=D.FIELD_TAG_DT)
        lay["id"] = rng.choice(587, 30, replace=False)
        for j in range(30):
            lay["R"][j] = PR.rot(*rng.uniform(-0.5, 0.5, size=3))
            lay["t"][j] = [rng.uniform(-1.5, 1.5), rng.uniform(-1, 1), rng.uniform(1.0, 6.0)]
        lays.append(lay)
    left_out = 0
    for trial in range(3000):
        lay, dist = lays[trial % len(lays)], MODELS[trial % len(MODELS)]
        raw = raw_list(D, rng, lay, params)
        if len(raw) and trial % 5 == 0:
            raw = past_the_fold(raw, 3)
        rot = PR.rot(*rng.uniform(-1, 1, size=3)) if trial % 2 else None
        off = rng.uniform(-1, 1, size=3) if trial % 2 else None
        host = D.estimate_field_pose(raw, lay, *params, rotation=rot, offset=off, distortion=dist)
        dev = D.estimate_field_pose_device(raw, lay, *params, rotation=rot, offset=off, distortion=dist)
        assert dev.tobytes() == host.tobytes(), trial
        left_out += host["num_tags"] < D.estimate_field_pose(raw, lay, *params)["num_tags"]
    assert left_out >= 50


def check_frame(D, det, f, params, method, dist, lay=None):
    dets, poses, tags = det.Detections(f), det.Poses(f), det.TagPositions(f)
    host = D.estimate_poses(dets, *params, method=method, distortion=dist)
    if method == "ippe":
        assert poses.tobytes() == host.tobytes()
    else:
        assert_poses_match(poses, host)
    order, ids, cam, robot, dist_, err = expected_positions(dets, poses, ROTATION, OFFSET)
    assert list(tags["index"]) == list(order) and list(tags["id"]) == list(ids)
    assert tags["camera"].tobytes() == cam.tobytes() and tags["distance"].tobytes() == dist_.tobytes()
    assert np.abs(tags["robot"] - robot).max(initial=0) <= 1e-12
    if lay is not None:
        got = det.FieldPose(f)
        field = D.estimate_field_pose(dets, lay, *params, rotation=ROTATION, offset=OFFSET, distortion=dist)
        assert got is not None and got.tobytes() == field.tobytes()
    return len(dets)


@pytest.mark.parametrize("method", ["oi", "ippe"])
@pytest.mark.parametrize("cfg,n", [(2, 16), (4, 4), (5, 1)])
def test_detector_equals_host(D, cfg, n, method):
    frames, fmt, w, h, dec, sigma = frames_of(cfg, n)
    params = (TAGSIZE, *intrinsics(w, h))
    lay = all_ids_layout(D, cfg)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=n)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method=method, distortion=WIDE)
    det.SetFieldLayout(lay)
    for _ in range(2):  # the second call replays the captured graph
        det.DetectBatch(frames)
        assert sum(check_frame(D, det, f, params, method, WIDE, lay) for f in range(n)) >= n
    det.close()


def test_mjpg_frames(D):
    cv2 = pytest.importorskip("cv2")
    from ros_vision_b200 import synth
    frame, _, w, h, dec, sigma, _ = synth.config_frame(1)
    ok, buf = cv2.imencode(".jpg", np.ascontiguousarray(frame).reshape(h, w), [cv2.IMWRITE_JPEG_QUALITY, 90])
    params = (TAGSIZE, *intrinsics(w, h))
    det = D.GpuDetector(w, h, "gray", quad_decimate=dec, quad_sigma=sigma)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe", distortion=REFERENCE)
    det.DetectMjpg([buf.tobytes()])
    assert check_frame(D, det, 0, params, "ippe", REFERENCE) == 4
    det.close()


def test_toggling_distortion(D):
    """On, off, on again between calls, two calls each (the second replays the graph): every call returns the poses of
    its own setting, and the kernel count does not change."""
    frames, fmt, w, h, dec, sigma = frames_of(2, 8)
    params = (TAGSIZE, *intrinsics(w, h))
    lay = all_ids_layout(D, 9)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    det.SetFieldLayout(lay)
    lib = D.load_library()
    counts = set()
    for method in ("ippe", "oi"):
        det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method=method)
        for dist in (WIDE, None, WIDE, [0.0] * 5):
            d = None if dist is None else np.ascontiguousarray(dist, dtype=np.float64)
            assert lib.b200tag_set_pose_distortion(det._h, None if d is None else d.ctypes.data_as(C.c_void_p)) == 0
            for _ in range(2):
                det.DetectBatch(frames)
                counts.add(det.kernels_per_batch())
                assert sum(check_frame(D, det, f, params, method, dist, lay) for f in range(8)) > 0
    assert len(counts) == 1
    bad = np.array([0.1, np.nan, 0, 0, 0])
    assert lib.b200tag_set_pose_distortion(det._h, bad.ctypes.data_as(C.c_void_p)) == -1
    det.DetectBatch(frames)  # the state is unchanged: still no distortion
    check_frame(D, det, 0, params, "oi", None, lay)
    det.close()


def lens_case(D, seed, w, h, params, dist, ntags=5, zmax=4.0):
    """test_gpu_field_pose.field_case's scene rendered through the lens `dist`: (layout, Scene, camera_R, camera_t)."""
    from ros_vision_b200 import synth
    rng = np.random.default_rng(seed)
    yaw = rng.uniform(-np.pi, np.pi)
    Ry = np.array([[np.cos(yaw), -np.sin(yaw), 0], [np.sin(yaw), np.cos(yaw), 0], [0, 0, 1]])
    camera_R, camera_t = Ry @ ROTATION, np.array([rng.uniform(0, 16), rng.uniform(0, 8), 0.6])
    lay = np.zeros(ntags, dtype=D.FIELD_TAG_DT)
    lay["id"] = rng.choice(587, ntags, replace=False)
    for j in range(ntags):
        z = rng.uniform(1.0, zmax)
        lay["R"][j] = camera_R @ PR.rot(rng.uniform(-0.5, 0.5), rng.uniform(-0.5, 0.5), rng.uniform(-0.3, 0.3))
        lay["t"][j] = camera_R @ np.array([rng.uniform(-0.5, 0.5) * z, rng.uniform(-0.35, 0.35) * z, z]) + camera_t
    sc = synth.field_scene(w, h, lay, TAGSIZE, camera_R, camera_t, *params[1:], seed=seed, noise_sigma=2.0, distortion=dist)
    return lay, sc, camera_R, camera_t


def test_field_pose_through_a_wide_angle_lens(D):
    """8 field_scene frames seen through WIDE (p2 = 0, so the decoder's reference UnDistort inverts the model), detected
    with the same coefficients and refine_edges on.  With the correction the field pose is within 2 cm and 0.5 deg of the
    truth; without it the worst error is at least 5x larger."""
    w, h = 1280, 800
    params = (TAGSIZE, PR.FX, PR.FY, PR.CX, PR.CY)
    cases = [lens_case(D, 200 + i, w, h, params, WIDE) for i in range(8)]
    worst = {}
    for dist in (WIDE, None):
        det = D.GpuDetector(w, h, "gray", quad_decimate=2, refine_edges=True, camera_matrix=(PR.FX, PR.CX, PR.FY, PR.CY),
                            distortion_coefficients=WIDE)
        det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe", distortion=dist)
        worst[dist] = (0.0, 0.0)
        for k, (lay, sc, cR, ct) in enumerate(cases):
            det.SetFieldLayout(lay)
            for _ in range(2):  # the second call replays the captured graph
                det.Detect(sc.gray)
                got = det.FieldPose(0)
                want = D.estimate_field_pose(det.Detections(0), lay, *params, rotation=ROTATION, offset=OFFSET, distortion=dist)
                assert got.tobytes() == want.tobytes()
            assert got["num_tags"] >= 3, (k, got["num_tags"], len(sc.tags))
            ang = np.degrees(np.arccos(np.clip((np.trace(got["camera_R"].T @ cR) - 1) / 2, -1, 1)))
            err = float(np.linalg.norm(got["camera_t"] - ct))
            worst[dist] = (max(worst[dist][0], err), max(worst[dist][1], ang))
            if dist is not None:
                assert err <= 0.02 and ang <= 0.5, (k, err, ang)
        det.close()
    on, off = worst[WIDE], worst[None]
    print(f"worst field pose error through the lens: corrected {on[0] * 100:.3f} cm / {on[1]:.4f} deg, "
          f"uncorrected {off[0] * 100:.3f} cm / {off[1]:.4f} deg")
    assert off[0] >= 5 * on[0]
