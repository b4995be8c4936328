"""The field pose step on the device (GpuDetector.SetFieldLayout, k_field_pose) against the host function it shares its
arithmetic with (estimate_field_pose, csrc/pose_core.h): only + - * /, sqrt, fabs and fmax, built without contraction on
both sides and every sum in one order, so every field is bit-identical."""
import ctypes as C
import functools

import numpy as np
import pytest

import pose_records as PR

pytestmark = pytest.mark.gpu

TAGSIZE = 0.1651
ROTATION = np.array([[0.0, 0, 1], [-1, 0, 0], [0, -1, 0]])  # camera looking along the robot's +x
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


def all_ids_layout(D, seed, n=587):
    """Every tag36h11 id at a random field pose: geometry that does not fit any frame, so the solve runs to its cap."""
    from ros_vision_b200.field_layout import quaternion_matrix
    rng = np.random.default_rng(seed)
    lay = np.zeros(n, dtype=D.FIELD_TAG_DT)
    lay["id"] = np.arange(n)
    for i in range(n):
        lay["R"][i] = quaternion_matrix(*rng.normal(size=4))
        lay["t"][i] = rng.uniform(-8, 8, size=3)
    return lay


@functools.lru_cache(maxsize=None)
def frames_of(cfg, n):
    from ros_vision_b200 import synth
    out = [synth.config_frame(cfg, i) for i in range(n)]
    frame, fmt, w, h, dec, sigma, _ = out[0]
    return [np.ascontiguousarray(o[0]).reshape(-1) for o in out], fmt, w, h, dec, sigma


def field_case(D, seed, w, h, params, ntags=5, zmax=4.0):
    """A camera on a robot somewhere on the field and `ntags` layout tags 1..zmax m in front of it, tilted up to ~30 deg;
    the field_scene frame of it.  Returns (layout, Scene, camera_R, camera_t)."""
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
        lay["t"][j] = camera_R @ np.array([rng.uniform(-0.4, 0.4) * z, rng.uniform(-0.3, 0.3) * z, z]) + camera_t
    sc = synth.field_scene(w, h, lay, TAGSIZE, camera_R, camera_t, *params[1:], seed=seed, noise_sigma=2.0)
    return lay, sc, camera_R, camera_t


def check_frame(D, det, f, lay, params, rotation=ROTATION, offset=OFFSET):
    """FieldPose(f) bit-identical to the host solve on Detections(f)."""
    got = det.FieldPose(f)
    want = D.estimate_field_pose(det.Detections(f), lay, *params, rotation=rotation, offset=offset)
    assert got is not None and got.tobytes() == want.tobytes()
    return got


def raw_list(D, rng, lay, params):
    """A random raw list against `lay`: projections of a random subset of its tags through a random camera, with
    overlapping and distant duplicates, ids and families outside the layout and collapsed quads, in random order."""
    fx, fy, cx, cy = params[1:]
    s = TAGSIZE / 2
    P = np.array([[-s, s, 0], [s, s, 0], [s, -s, 0], [-s, -s, 0]])
    Rcf = PR.rot(*rng.uniform(-np.pi, np.pi, size=3))
    tcf = rng.uniform(-3, 3, size=3)
    recs = []
    for L in lay[rng.permutation(len(lay))[:rng.integers(0, min(len(lay), 12) + 1)]]:
        cam = (P @ np.asarray(L["R"]).T + L["t"]) @ Rcf.T + tcf
        d = np.zeros(1, dtype=D.DETECTION_DT)[0]
        d["id"], d["family"] = L["id"], L["family"]
        d["hamming"], d["decision_margin"] = rng.integers(0, 3), rng.uniform(20, 150)
        z = np.where(np.abs(cam[:, 2]) < 1e-3, 1e-3, cam[:, 2])
        d["p"] = np.stack([fx * cam[:, 0] / z + cx, fy * cam[:, 1] / z + cy], axis=1) + rng.normal(0, 0.5, size=(4, 2))
        kind = rng.integers(0, 6)
        if kind == 0:
            d["p"] = d["p"][0]  # collapsed
        recs.append(d)
        if kind in (1, 2):  # an overlapping duplicate, and sometimes one with equal hamming and margin
            e = d.copy()
            e["p"] = d["p"] + rng.uniform(-0.5, 0.5, size=(4, 2))
            if kind == 2:
                e["hamming"], e["decision_margin"] = rng.integers(0, 3), rng.uniform(20, 150)
            recs.append(e)
        if kind == 3:  # a distant duplicate
            e = d.copy()
            e["p"] = d["p"] + 400.0
            e["hamming"] = rng.integers(0, 3)
            recs.append(e)
        if kind == 4:  # the same id in another family, and an id outside the layout
            for fam, idv in ((d["family"] + 1, d["id"]), (d["family"], 5000)):
                e = d.copy()
                e["family"], e["id"] = fam, idv
                recs.append(e)
    out = np.array(recs, dtype=D.DETECTION_DT) if recs else np.zeros(0, dtype=D.DETECTION_DT)
    out["c"] = out["p"].mean(axis=1) if len(out) else out["c"]
    return out[rng.permutation(len(out))]


def test_hook_is_bit_identical_to_the_host(D):
    rng = np.random.default_rng(21)
    params = (TAGSIZE, 905.5, 907.9, 640.0, 400.0)
    lays = [all_ids_layout(D, 1, 40)]
    for k in range(3):  # layouts of consistent geometry in two families
        lay = np.zeros(30, dtype=D.FIELD_TAG_DT)
        lay["id"] = rng.choice(587, 30, replace=False)
        lay["family"] = rng.integers(0, 2, size=30)
        for j in range(30):
            lay["R"][j] = PR.rot(*rng.uniform(-0.5, 0.5, size=3))
            lay["t"][j] = [rng.uniform(-1.5, 1.5), rng.uniform(-1, 1), rng.uniform(1.0, 6.0)]
        lays.append(lay)
    counts = {"empty": 0, "one": 0, "many": 0}
    for trial in range(3000):
        lay = lays[trial % len(lays)]
        raw = raw_list(D, rng, lay, params)
        rot = PR.rot(*rng.uniform(-1, 1, size=3)) if trial % 2 else None
        off = rng.uniform(-1, 1, size=3) if trial % 2 else None
        host = D.estimate_field_pose(raw, lay, *params, rotation=rot, offset=off)
        dev = D.estimate_field_pose_device(raw, lay, *params, rotation=rot, offset=off)
        assert dev.tobytes() == host.tobytes(), trial
        counts["empty" if host["num_tags"] == 0 else "one" if host["num_tags"] == 1 else "many"] += 1
    assert min(counts.values()) >= 100, counts


@pytest.mark.parametrize("method", ["oi", "ippe"])
def test_field_scene_frames(D, method):
    w, h = 1280, 800
    params = (TAGSIZE, 905.5, 907.9, 640.0, 400.0)
    cases = [field_case(D, 100 + i, w, h, params) for i in range(8)]
    det = D.GpuDetector(w, h, "gray", quad_decimate=2)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method=method)
    worst = (0.0, 0.0)
    for k, (clay, sc, cR, ct) in enumerate(cases):
        det.SetFieldLayout(clay)
        for _ in range(2):  # the second call replays the captured graph
            det.Detect(sc.gray)
            got = check_frame(D, det, 0, clay, params)
        assert got["num_tags"] >= 3, k
        ang = np.degrees(np.arccos(np.clip((np.trace(got["camera_R"].T @ cR) - 1) / 2, -1, 1)))
        dist = float(np.linalg.norm(got["camera_t"] - ct))
        worst = (max(worst[0], dist), max(worst[1], ang))
        assert dist <= 0.02 and ang <= 0.5, (k, dist, ang)
        robot_R = got["camera_R"] @ ROTATION.T
        assert np.abs(got["robot_t"] - (got["camera_t"] - robot_R @ OFFSET)).max() <= 1e-12
    print(f"worst field_scene error ({method}): {worst[0] * 100:.3f} cm, {worst[1]:.4f} deg")
    det.close()


@pytest.mark.parametrize("cfg,n", [(2, 16), (4, 4), (5, 2)])
def test_config_frames_with_an_all_ids_layout(D, cfg, n):
    frames, fmt, w, h, dec, sigma = frames_of(cfg, n)
    params = (TAGSIZE, *intrinsics(w, h))
    lay = all_ids_layout(D, cfg)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=n)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    det.SetFieldLayout(lay)
    for _ in range(2):  # the second call replays the captured graph
        det.DetectBatch(frames)
        used = [int(check_frame(D, det, f, lay, params)["num_tags"]) for f in range(n)]
        assert sum(used) >= n
    det.close()


def test_batch_with_empty_frames_and_capped_lists(D):
    frames, fmt, w, h, dec, sigma = frames_of(2, 3)
    blank = np.full_like(frames[0], 128)
    batch = [blank, frames[0], blank, blank, frames[1], frames[2], blank]
    params = (TAGSIZE, *intrinsics(w, h))
    lay = all_ids_layout(D, 7)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=len(batch))
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET)
    det.SetFieldLayout(lay)
    det.DetectBatch(batch)
    used = [int(check_frame(D, det, f, lay, params)["num_tags"]) for f in range(len(batch))]
    assert [used[i] for i in (0, 2, 3, 6)] == [0, 0, 0, 0] and min(used[i] for i in (1, 4, 5)) > 0
    det.close()
    frames, fmt, w, h, dec, sigma = frames_of(5, 1)
    params = (TAGSIZE, *intrinsics(w, h))
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_detections=5)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    det.SetFieldLayout(lay)
    assert det.DetectBatch(frames, allow_overflow=True) == -4
    assert 0 < check_frame(D, det, 0, lay, params)["num_tags"] <= 5
    det.close()


def test_mjpg_frames_get_a_field_pose(D):
    cv2 = pytest.importorskip("cv2")
    w, h = 1280, 800
    params = (TAGSIZE, 905.5, 907.9, 640.0, 400.0)
    lay, sc, cR, ct = field_case(D, 5, w, h, params)
    ok, buf = cv2.imencode(".jpg", sc.gray, [cv2.IMWRITE_JPEG_QUALITY, 90])
    det = D.GpuDetector(w, h, "gray", quad_decimate=2)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    det.SetFieldLayout(lay)
    det.DetectMjpg([buf.tobytes()])
    assert check_frame(D, det, 0, lay, params)["num_tags"] >= 3
    det.close()


def _results(det, n):
    return [(det.Detections(f).tobytes(), det.Poses(f).tobytes(), det.TagPositions(f).tobytes()) for f in range(n)]


def test_switching_and_other_results(D):
    """On, off, on, a replaced layout and the pose step off, each from the next call; the other results and the kernel
    count are those of a detector without a layout, plus one kernel while the step runs."""
    frames, fmt, w, h, dec, sigma = frames_of(2, 8)
    params = (TAGSIZE, *intrinsics(w, h))
    lay_a, lay_b = all_ids_layout(D, 11), all_ids_layout(D, 12)[::3].copy()
    plain = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma, max_batch=8)
    for d in (plain, det):
        d.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    assert det.FieldPose(0) is None
    for lay in (lay_a, None, lay_a, lay_b, np.zeros(0, dtype=D.FIELD_TAG_DT), lay_b):
        det.SetFieldLayout(lay)
        for _ in range(2):
            plain.DetectBatch(frames)
            det.DetectBatch(frames)
            assert _results(det, 8) == _results(plain, 8)
            if lay is None or len(lay) == 0:
                assert det.FieldPose(0) is None and det.kernels_per_batch() == plain.kernels_per_batch()
            else:
                assert det.kernels_per_batch() == plain.kernels_per_batch() + 1
                assert sum(int(check_frame(D, det, f, lay, params)["num_tags"]) for f in range(8)) > 0
    # the pose step off: no field pose, and no kernel, though the layout stays set
    det.SetPoseEstimation(0, *params[1:])
    plain.SetPoseEstimation(0, *params[1:])
    det.DetectBatch(frames)
    plain.DetectBatch(frames)
    assert det.FieldPose(0) is None and det.kernels_per_batch() == plain.kernels_per_batch()
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET)
    det.DetectBatch(frames)
    assert sum(int(check_frame(D, det, f, lay_b, params)["num_tags"]) for f in range(8)) > 0
    plain.close()
    det.close()


def test_invalid_layout_keeps_the_state(D):
    frames, fmt, w, h, dec, sigma = frames_of(1, 1)
    params = (TAGSIZE, *intrinsics(w, h))
    lay = all_ids_layout(D, 3, 8)
    det = D.GpuDetector(w, h, fmt, quad_decimate=dec, quad_sigma=sigma)
    det.SetPoseEstimation(*params, rotation=ROTATION, offset=OFFSET, method="ippe")
    det.SetFieldLayout(lay)
    det.Detect(frames[0])
    before = det.FieldPose(0).tobytes()
    lib = D.load_library()
    bads = []
    for field, idx, v in [("family", 2, 1), ("family", 2, -1), ("id", 2, 587), ("id", 2, -1), ("id", 2, 1),
                          ("R", (2, 0, 0), 1.1), ("R", (2, 0, 0), np.nan), ("t", (2, 1), np.inf)]:
        bad = lay.copy()
        bad[field][idx] = v
        bads.append(bad)
    mirror = lay.copy()
    mirror["R"][2] = -mirror["R"][2]
    bads.append(mirror)
    big = np.zeros(1025, dtype=D.FIELD_TAG_DT)
    big["R"] = np.eye(3)
    bads.append(big)
    for bad in bads:
        assert lib.b200tag_set_field_layout(det._h, bad.ctypes.data_as(C.c_void_p), len(bad)) == E_INVALID
    assert lib.b200tag_set_field_layout(det._h, None, 3) == E_INVALID
    assert lib.b200tag_set_field_layout(None, lay.ctypes.data_as(C.c_void_p), len(lay)) == E_INVALID
    with pytest.raises(D.B200TagError):
        det.SetFieldLayout(bads[0])
    det.Detect(frames[0])
    assert det.FieldPose(0).tobytes() == before
    check_frame(D, det, 0, lay, params)
    det.close()
