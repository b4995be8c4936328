"""The IPPE pose method on the device (GpuDetector.SetPoseEstimation(..., method="ippe"), k_pose_ippe) against the host
function it shares its arithmetic with (estimate_poses(..., method="ippe"), csrc/pose_core.h).  IPPE uses only
+ - * /, sqrt, fabs and fmax, built without contraction on both sides, so every field is bit-identical."""
import functools

import numpy as np
import pytest

import pose_records as PR

pytestmark = pytest.mark.gpu

TAGSIZE = 0.1651
ROTATION = PR.rot(0.3, -1.1, 0.7)
OFFSET = np.array([0.25, -0.1, 0.6])
E_INVALID = -1


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


def expected_positions(dets, poses, rotation, offset):
    """The node's records from the poses, restated: robot = rotation t + offset, distance |t|, closest first."""
    t = poses["t"]
    dist = np.sqrt(t[:, 0] * t[:, 0] + t[:, 1] * t[:, 1] + t[:, 2] * t[:, 2])
    order = np.argsort(dist, kind="stable")
    robot = t @ np.asarray(rotation, dtype=np.float64).T + np.asarray(offset, dtype=np.float64)
    return order, dets["id"][order], t[order], robot[order], dist[order], poses["err"][order]


def check_frame(D, det, f, params, rotation=ROTATION, offset=OFFSET):
    """Poses(f) bit-identical to host IPPE on Detections(f); TagPositions(f) the records made from them."""
    dets, poses, tags = det.Detections(f), det.Poses(f), det.TagPositions(f)
    assert len(poses) == len(dets) == len(tags)
    assert poses.tobytes() == D.estimate_poses(dets, *params, method="ippe").tobytes()
    order, ids, cam, robot, dist, err = expected_positions(dets, poses, rotation, offset)
    assert list(tags["index"]) == list(order) and list(tags["id"]) == list(ids)
    assert tags["camera"].tobytes() == cam.tobytes() and tags["distance"].tobytes() == dist.tobytes()
    assert tags["err"].tobytes() == err.tobytes()
    assert np.abs(tags["robot"] - robot).max(initial=0) <= 1e-12
    return len(dets)


def test_hook_is_bit_identical_to_the_host(D):
    recs = PR.records(20000, 7)
    params = (PR.TAGSIZE, PR.FX, PR.FY, PR.CX, PR.CY)
    dev = D.estimate_poses_device(recs, *params, method="ippe")
    host = D.estimate_poses(recs, *params, method="ippe")
    assert dev.tobytes() == host.tobytes()
    assert int(np.isinf(host["err"]).sum()) == len(recs) // 4  # the collapsed quads
    assert not np.isnan(dev["R"]).any() and not np.isnan(dev["t"]).any()
    assert len(D.estimate_poses_device(recs[:0], *params, method="ippe")) == 0


@pytest.mark.parametrize("cfg,n", [(2, 32), (1, 1), (4, 4), (5, 1)])
def test_device_equals_host_on_frames(D, cfg, n):
    frames, fmt, w, h, dec, sigma = frames_of(cfg, n)
    params = (TAGSIZE, *intrinsics(w, h))
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=n)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    for _ in range(2):  # the second call replays the captured graph
        det.DetectBatch(frames)
        total = sum(check_frame(D, det, f, params) for f in range(n))
        assert total >= n
    det.close()


def _raw_results(det, n):
    """Detections, quads (blob_index, a slot filled through atomics, left out) and frame info as bytes."""
    out = []
    for f in range(n):
        quads = det.FitQuads(f)
        quads["blob_index"] = 0
        out.append((det.Detections(f).tobytes(), quads.tobytes(), bytes(det.FrameInfo(f))))
    return out


def test_switching_methods(D):
    """OI -> IPPE -> OI on one detector, two calls each (the second replays the graph): every call returns its own
    method's poses, and the detection results and kernel count are those of a pose-off detector plus one kernel."""
    frames, fmt, w, h, dec, sigma = frames_of(2, 8)
    params = (TAGSIZE, *intrinsics(w, h))
    plain = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    oi_only = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    oi_only.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET)
    lib = D.load_library()
    for method in ("oi", "ippe", "oi"):
        assert lib.b200tag_set_pose_method(det._h, D.POSE_METHODS[method]) == 0
        for _ in range(2):
            plain.DetectBatch(frames)
            det.DetectBatch(frames)
            assert _raw_results(det, 8) == _raw_results(plain, 8)
            assert det.kernels_per_batch() == plain.kernels_per_batch() + 1
            if method == "ippe":
                assert sum(check_frame(D, det, f, params) for f in range(8)) > 0
            else:
                oi_only.DetectBatch(frames)
                for f in range(8):
                    dets, poses = det.Detections(f), det.Poses(f)
                    assert poses.tobytes() == oi_only.Poses(f).tobytes()
                    assert det.TagPositions(f).tobytes() == oi_only.TagPositions(f).tobytes()
                    host = D.estimate_poses(dets, *params)
                    assert np.abs(poses["R"] - host["R"]).max(initial=0) <= 1e-9
                    assert np.abs(poses["t"] - host["t"]).max(initial=0) <= 1e-9
    for d in (plain, oi_only, det):
        d.close()


def test_batch_with_empty_frames(D):
    frames, fmt, w, h, dec, sigma = frames_of(2, 3)
    blank = np.full_like(frames[0], 128)
    batch = [blank, frames[0], blank, blank, frames[1], frames[2], blank]
    params = (TAGSIZE, *intrinsics(w, h))
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=len(batch))
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    det.DetectBatch(batch)
    counts = [check_frame(D, det, f, params) for f in range(len(batch))]
    assert [counts[i] for i in (0, 2, 3, 6)] == [0, 0, 0, 0] and min(counts[i] for i in (1, 4, 5)) > 0
    det.close()


def test_capped_detections(D):
    frames, fmt, w, h, dec, sigma = frames_of(5, 1)
    params = (TAGSIZE, *intrinsics(w, h))
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_detections=5)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    assert det.DetectBatch(frames, allow_overflow=True) == -4
    assert det.FrameInfo(0).status & D.ST_DETS_OVERFLOW
    assert 0 < check_frame(D, det, 0, params) <= 5
    det.close()


def test_mjpg_frames_get_poses(D):
    cv2 = pytest.importorskip("cv2")
    from ros_vision_b200 import synth
    frame, _, w, h, dec, sigma, _ = synth.config_frame(1)
    ok, buf = cv2.imencode(".jpg", np.ascontiguousarray(frame).reshape(h, w), [cv2.IMWRITE_JPEG_QUALITY, 90])
    params = (TAGSIZE, *intrinsics(w, h))
    det = D.GpuDetector(w, h, "gray", quad_decimate=dec, quad_sigma=sigma)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    det.DetectMjpg([buf.tobytes()])
    assert check_frame(D, det, 0, params) == 4
    det.close()


def test_invalid_method_keeps_the_state(D):
    frames, fmt, w, h, dec, sigma = frames_of(1, 1)
    params = (TAGSIZE, *intrinsics(w, h))
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    det.Detect(frames[0])
    before = (det.Poses(0).tobytes(), det.TagPositions(0).tobytes())
    lib = D.load_library()
    for bad in (2, -1, 100):
        assert lib.b200tag_set_pose_method(det._h, bad) == E_INVALID
    assert lib.b200tag_set_pose_method(None, D.POSE_METHODS["ippe"]) == E_INVALID
    with pytest.raises(ValueError):
        det.SetPoseEstimation(*params, method="epnp")
    det.Detect(frames[0])
    assert check_frame(D, det, 0, params) == 4
    assert (det.Poses(0).tobytes(), det.TagPositions(0).tobytes()) == before
    # turning the step off and on again keeps the method
    det.SetPoseEstimation(0, *intrinsics(w, h), method="ippe")
    det.Detect(frames[0])
    assert len(det.Poses(0)) == 0
    assert lib.b200tag_set_pose_estimation(det._h, *params, None, None) == 0
    det.Detect(frames[0])
    assert check_frame(D, det, 0, params, rotation=np.eye(3), offset=np.zeros(3)) == 4
    det.close()
