"""Pose covariances on the device (GpuDetector.SetPoseCovariance: k_pose_cov and k_field_pose's variants with the
covariance) against the host functions they share their arithmetic with, on caller records and in detection runs."""
import ctypes as C

import numpy as np
import pytest

import pose_records as PR
from test_gpu_field_pose import all_ids_layout, raw_list
from test_gpu_pose_distortion import MODELS, TAGSIZE, WIDE, frames_of, intrinsics, past_the_fold

pytestmark = pytest.mark.gpu

ROTATION = np.array([[0.0, 0, 1], [-1, 0, 0], [0, -1, 0]])
OFFSET = np.array([0.25, -0.1, 0.6])
SIGMA = 0.3


@pytest.fixture(scope="module")
def D():
    from ros_vision_b200 import build, detector
    build.build_native()
    detector.load_library()
    return detector


@pytest.mark.parametrize("dist", [None, *MODELS])
@pytest.mark.parametrize("method", ["oi", "ippe"])
def test_pose_hook_equals_the_host(D, method, dist):
    recs = PR.records(20000, 70)
    if dist is not None:
        recs = past_the_fold(recs)
    params = (PR.TAGSIZE, PR.FX, PR.FY, PR.CX, PR.CY)
    poses = D.estimate_poses(recs, *params, method=method, distortion=dist)
    host = D.estimate_pose_covariances(recs, poses, *params, SIGMA, distortion=dist)
    dev = D.estimate_pose_covariances_device(recs, poses, *params, SIGMA, distortion=dist)
    assert dev.tobytes() == host.tobytes()
    failed = np.isinf(host["C"]).all(axis=(1, 2))
    assert failed.sum() >= len(recs) // 4 and np.isfinite(host["C"][~failed]).all()


def test_field_hook_equals_the_host(D):
    rng = np.random.default_rng(71)
    params = (TAGSIZE, PR.FX, PR.FY, PR.CX, PR.CY)
    lays = [all_ids_layout(D, 3, 40)]
    for _ in range(3):
        lay = np.zeros(30, dtype=D.FIELD_TAG_DT)
        lay["id"] = rng.choice(587, 30, replace=False)
        for j in range(30):
            lay["R"][j] = PR.rot(*rng.uniform(-0.5, 0.5, size=3))
            lay["t"][j] = [rng.uniform(-1.5, 1.5), rng.uniform(-1, 1), rng.uniform(1.0, 6.0)]
        lays.append(lay)
    finite = 0
    for trial in range(3000):
        lay, dist = lays[trial % len(lays)], (None, *MODELS)[trial % 4]
        raw = raw_list(D, rng, lay, params)
        rot = PR.rot(*rng.uniform(-1, 1, size=3)) if trial % 2 else None
        off = rng.uniform(-1, 1, size=3) if trial % 2 else None
        hp, hc = D.estimate_field_pose_covariance(raw, lay, *params, SIGMA, rotation=rot, offset=off, distortion=dist)
        dp, dc = D.estimate_field_pose_covariance_device(raw, lay, *params, SIGMA, rotation=rot, offset=off, distortion=dist)
        assert dp.tobytes() == hp.tobytes() and dc.tobytes() == hc.tobytes(), trial
        finite += bool(np.isfinite(hc["robot"]).all())
    assert 300 <= finite <= 2900  # both finite covariances and failures (no tags, corners behind the camera)


def check_frame(D, det, ref, f, params, method, dist, sigma, lay):
    """det's results of frame f: the covariances equal the host functions; everything else equals `ref`'s (the same
    settings without covariance)."""
    dets, poses = det.Detections(f), det.Poses(f)
    assert dets.tobytes() == ref.Detections(f).tobytes() and poses.tobytes() == ref.Poses(f).tobytes()
    assert det.TagPositions(f).tobytes() == ref.TagPositions(f).tobytes()
    assert det.FieldPose(f).tobytes() == ref.FieldPose(f).tobytes()
    cov = det.PoseCovariances(f)
    if sigma == 0:
        assert len(cov) == 0 and det.FieldCovariance(f) is None
        return 0
    assert cov.tobytes() == D.estimate_pose_covariances(dets, poses, *params, sigma, distortion=dist).tobytes()
    fp, fc = D.estimate_field_pose_covariance(dets, lay, *params, sigma, rotation=ROTATION, offset=OFFSET, distortion=dist)
    assert fp.tobytes() == det.FieldPose(f).tobytes() and fc.tobytes() == det.FieldCovariance(f).tobytes()
    return len(dets)


@pytest.mark.parametrize("method", ["oi", "ippe"])
@pytest.mark.parametrize("cfg,n", [(2, 16), (4, 4), (5, 1)])
def test_detector_equals_host(D, cfg, n, method):
    """Batches and single frames, graph replays, covariance on, off and at a new sigma between calls, with and without
    the lens: the covariances equal the host's, and every other result and the kernel count equal a detector's without
    covariance, plus one kernel while it is on."""
    frames, fmt, w, h, dec, sigma = frames_of(cfg, n)
    params = (TAGSIZE, *intrinsics(w, h))
    lay = all_ids_layout(D, cfg)
    for dist in (None, WIDE):
        dets = []
        for _ in range(2):
            d = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=n)
            d.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method=method, distortion=dist)
            d.SetFieldLayout(lay)
            dets.append(d)
        det, ref = dets
        for s in (SIGMA, 0.0, 1.7):
            det.SetPoseCovariance(s)
            for _ in range(2):  # the second call replays the captured graph
                det.DetectBatch(frames)
                ref.DetectBatch(frames)
                assert det.kernels_per_batch() == ref.kernels_per_batch() + (s > 0)
                got = sum(check_frame(D, det, ref, f, params, method, dist, s, lay) for f in range(n))
                assert s == 0 or got >= n
        det.close()
        ref.close()


def test_mjpg_and_single_frames(D):
    cv2 = pytest.importorskip("cv2")
    from ros_vision_b200 import synth
    frame, _, w, h, dec, sigma, _ = synth.config_frame(1)
    ok, buf = cv2.imencode(".jpg", np.ascontiguousarray(frame).reshape(h, w), [cv2.IMWRITE_JPEG_QUALITY, 90])
    params = (TAGSIZE, *intrinsics(w, h))
    lay = all_ids_layout(D, 1)
    dets = []
    for s in (SIGMA, 0.0):
        d = D.GpuDetector(w, h, "gray", quad_decimate=dec, quad_sigma=sigma)
        d.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe", distortion=WIDE)
        d.SetFieldLayout(lay)
        d.SetPoseCovariance(s)
        d.DetectMjpg([buf.tobytes()])
        dets.append(d)
    assert check_frame(D, dets[0], dets[1], 0, params, "ippe", WIDE, SIGMA, lay) == 4
    for d in dets:
        d.close()


def test_setter_checks_and_off_is_unchanged(D):
    """A bad sigma is rejected with the state unchanged; a detector that turns the covariance on and off again returns
    and launches what one that never turned it on does."""
    frames, fmt, w, h, dec, sigma = frames_of(2, 8)
    params = (TAGSIZE, *intrinsics(w, h))
    lay = all_ids_layout(D, 9)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    ref = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    for d in (det, ref):
        d.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
        d.SetFieldLayout(lay)
    lib = D.load_library()
    det.SetPoseCovariance(SIGMA)
    for bad in (-1.0, np.nan, np.inf):
        assert lib.b200tag_set_pose_covariance(det._h, C.c_double(bad)) == -1
    det.DetectBatch(frames)
    ref.DetectBatch(frames)
    assert sum(check_frame(D, det, ref, f, params, "ippe", None, SIGMA, lay) for f in range(8)) > 0
    det.SetPoseCovariance(0)
    for _ in range(2):
        det.DetectBatch(frames)
        ref.DetectBatch(frames)
        assert det.kernels_per_batch() == ref.kernels_per_batch()
        for f in range(8):
            check_frame(D, det, ref, f, params, "ippe", None, 0.0, lay)
    det.close()
    ref.close()
