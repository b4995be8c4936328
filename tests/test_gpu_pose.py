"""The pose step on the device (GpuDetector.SetPoseEstimation, k_pose) against the host functions it shares its
arithmetic with (estimate_poses / locate_tags, csrc/pose_core.h).

The homography start and the orthogonal iteration use only + - * /, sqrt, fabs and fmax, built without contraction on
both sides, so the first local minimum is bit-identical.  The second-minimum search calls tan / atan / atan2 / sin /
cos, where the device's libm and glibc may differ by an ulp: a pose that is the second minimum agrees to 1e-9."""
import functools
import os
import subprocess

import numpy as np
import pytest

import pose_records as PR

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
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


def _rel(a, b):
    return np.abs(a - b) <= 1e-9 * np.maximum(np.abs(a), np.abs(b))


def assert_poses_match(dev, host):
    """Per record: the first minimum returned -> R, t, err bit-identical, err_other within 1e-9 (or both HUGE_VAL);
    the second minimum returned -> its err_other (the first minimum's error) bit-identical, R and t within 1e-9, err
    within a relative 1e-9.  Either way both sides returned the same minimum."""
    assert len(dev) == len(host)
    for i, (d, h) in enumerate(zip(dev, host)):
        first = (d["R"].tobytes() == h["R"].tobytes() and d["t"].tobytes() == h["t"].tobytes()
                 and d["err"].tobytes() == h["err"].tobytes())
        if first:
            assert (np.isinf(d["err_other"]) and np.isinf(h["err_other"])) or _rel(d["err_other"], h["err_other"]), (i, d, h)
        else:
            assert d["err_other"].tobytes() == h["err_other"].tobytes(), (i, d, h)
            assert np.abs(d["R"] - h["R"]).max() <= 1e-9 and np.abs(d["t"] - h["t"]).max() <= 1e-9, (i, d, h)
            assert _rel(d["err"], h["err"]), (i, d, h)


def assert_positions_match(dev, host):
    assert list(dev["index"]) == list(host["index"]) and list(dev["id"]) == list(host["id"])
    for k in ("camera", "robot", "distance"):
        assert np.abs(dev[k] - host[k]).max(initial=0) <= 1e-9, k
    assert np.all(_rel(dev["err"], host["err"]) | (np.isinf(dev["err"]) & np.isinf(host["err"])))


def check_frame(D, det, f, params, rotation=ROTATION, offset=OFFSET):
    dets = det.Detections(f)
    poses = det.Poses(f)
    assert len(poses) == len(dets)
    assert_poses_match(poses, D.estimate_poses(dets, *params))
    assert_positions_match(det.TagPositions(f), D.locate_tags(dets, *params, rotation, offset))
    return len(dets)


@functools.lru_cache(maxsize=None)
def frames_of(cfg, n):
    from ros_vision_b200 import synth
    out = [synth.config_frame(cfg, i) for i in range(n)]
    frame, fmt, w, h, dec, sigma, _ = out[0]
    return [np.ascontiguousarray(o[0]).reshape(-1) for o in out], fmt, w, h, dec, sigma


@pytest.mark.parametrize("cfg,n", [(2, 32), (1, 1), (4, 4), (5, 1)])
def test_device_equals_host_on_frames(D, cfg, n):
    frames, fmt, w, h, dec, sigma = frames_of(cfg, n)
    params = (TAGSIZE, *intrinsics(w, h))
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=n)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET)
    det.DetectBatch(frames)
    total = sum(check_frame(D, det, f, params) for f in range(n))
    assert total >= n
    det.close()


def test_random_records_through_the_hook(D):
    recs = PR.records(20000, 7)
    params = (PR.TAGSIZE, PR.FX, PR.FY, PR.CX, PR.CY)
    dev = D.estimate_poses_device(recs, *params)
    host = D.estimate_poses(recs, *params)
    assert_poses_match(dev, host)
    assert int(np.isfinite(dev["err_other"]).sum()) == int(np.isfinite(host["err_other"]).sum()) > 5000
    assert int(np.isinf(host["err"]).sum()) > 0
    assert len(D.estimate_poses_device(recs[:0], *params)) == 0


def _raw_results(det, n):
    """Detections, quads and frame info as bytes.  A quad's blob_index is its slot in a work list that the fit kernels
    fill through atomics, so it differs between any two runs: it is left out."""
    out = []
    for f in range(n):
        quads = det.FitQuads(f)
        quads["blob_index"] = 0
        out.append((det.Detections(f).tobytes(), quads.tobytes(), bytes(det.FrameInfo(f))))
    return out


def test_pose_off_changes_nothing(D):
    frames, fmt, w, h, dec, sigma = frames_of(2, 8)
    params = (TAGSIZE, *intrinsics(w, h))
    plain = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    posed = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    posed.SetPoseEstimation(*params)
    for _ in range(2):  # the second call replays the captured graphs
        plain.DetectBatch(frames)
        posed.DetectBatch(frames)
        assert _raw_results(plain, 8) == _raw_results(posed, 8)
        assert posed.kernels_per_batch() == plain.kernels_per_batch() + 1
        assert len(plain.Poses(0)) == 0 and len(plain.TagPositions(0)) == 0
        assert sum(len(posed.Poses(f)) for f in range(8)) == sum(len(plain.Detections(f)) for f in range(8))
    posed.SetPoseEstimation(0, *intrinsics(w, h))
    posed.DetectBatch(frames)
    assert _raw_results(plain, 8) == _raw_results(posed, 8)
    assert posed.kernels_per_batch() == plain.kernels_per_batch()
    assert all(len(posed.Poses(f)) == 0 and len(posed.TagPositions(f)) == 0 for f in range(8))
    plain.close()
    posed.close()


def test_parameter_changes_reach_the_device(D):
    frames, fmt, w, h, dec, sigma = frames_of(4, 2)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=2)
    params = (TAGSIZE, *intrinsics(w, h))
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET)
    det.DetectBatch(frames)
    for f in range(2):
        check_frame(D, det, f, params)
    params2 = (0.2032, 1100.0, 1090.0, w / 2 + 11.0, h / 2 - 7.0)
    det.SetPoseEstimation(*params2)
    det.DetectBatch(frames)
    for f in range(2):
        check_frame(D, det, f, params2, rotation=None, offset=None)
    det.close()


def test_batch_with_empty_frames(D):
    frames, fmt, w, h, dec, sigma = frames_of(2, 3)
    blank = np.full_like(frames[0], 128)
    batch = [blank, frames[0], blank, blank, frames[1], frames[2], blank]
    params = (TAGSIZE, *intrinsics(w, h))
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=len(batch))
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET)
    det.DetectBatch(batch)
    counts = [check_frame(D, det, f, params) for f in range(len(batch))]
    assert [counts[i] for i in (0, 2, 3, 6)] == [0, 0, 0, 0] and min(counts[i] for i in (1, 4, 5)) > 0
    det.close()


def test_capped_detections(D):
    frames, fmt, w, h, dec, sigma = frames_of(5, 1)
    params = (TAGSIZE, *intrinsics(w, h))
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_detections=5)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET)
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
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET)
    det.DetectMjpg([buf.tobytes()])
    assert check_frame(D, det, 0, params) == 4
    det.close()


def test_bad_arguments_keep_the_state(D):
    frames, fmt, w, h, dec, sigma = frames_of(1, 1)
    params = (TAGSIZE, *intrinsics(w, h))
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET)
    lib, fx, fy, cx, cy = D.load_library(), *intrinsics(w, h)
    assert lib.b200tag_set_pose_estimation(det._h, -0.1, fx, fy, cx, cy, None, None) == E_INVALID
    assert lib.b200tag_set_pose_estimation(det._h, 0.5, 0.0, fy, cx, cy, None, None) == E_INVALID
    assert lib.b200tag_set_pose_estimation(det._h, 0.5, fx, 0.0, cx, cy, None, None) == E_INVALID
    with pytest.raises(D.B200TagError):
        det.SetPoseEstimation(float("nan"), fx, fy, cx, cy)
    det.Detect(frames[0])
    assert check_frame(D, det, 0, params) == 4
    det.close()


def test_cpp_class_through_handle(D, tmp_path):
    from ros_vision_b200 import build, synth
    build.build_cpp_class()
    frame, fmt, w, h, dec, sigma, _ = synth.config_frame(1)
    fx, fy, cx, cy = intrinsics(w, h)
    inc, lib = os.path.join(ROOT, "include"), build.LIBDIR
    exe = tmp_path / "pose_step_test"
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", inc, "-I", os.path.join(inc, "apriltag_compat"),
                           os.path.join(ROOT, "tests", "cpp", "pose_step_test.cc"), "-o", str(exe), "-L", lib,
                           "-lapriltags_cuda_core", "-lb200tag", f"-Wl,-rpath,{lib}"])
    raw = tmp_path / "gray.raw"
    raw.write_bytes(np.ascontiguousarray(frame).tobytes())
    r = subprocess.run([str(exe), str(raw), str(w), str(h)] + [repr(float(x)) for x in (fx, fy, cx, cy, TAGSIZE)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [ln.split() for ln in r.stdout.splitlines()]
    rotation = np.array([[0, 0, 1], [-1, 0, 0], [0, -1, 0]], dtype=np.float64)
    offset = np.array([0.1, -0.2, 0.5])
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, camera_matrix=(fx, cx, fy, cy))
    det.SetPoseEstimation(TAGSIZE, fx, fy, cx, cy, rotation=rotation, offset=offset)
    det.Detect(frame)
    dets, poses, tags = det.Detections(0), det.Poses(0), det.TagPositions(0)
    want = [["pose", str(int(d["id"]))] + [float(x) for x in (*p["t"], p["err"])] for d, p in zip(dets, poses)]
    want += [["tag", str(int(t["index"])), str(int(t["id"]))] + [float(x) for x in (*t["robot"], t["distance"])] for t in tags]
    got = [ln[:2] + [float(x) for x in ln[2:]] if ln[0] == "pose" else ln[:3] + [float(x) for x in ln[3:]] for ln in lines]
    assert len(dets) == 4 and got == want
    det.close()
