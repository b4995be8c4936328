"""Lens distortion in the pose step on the host (undistort_points, estimate_poses / estimate_field_pose with
distortion=...): the exact inverse of OpenCV's 5-coefficient model against cv2.projectPoints, neutral settings that
leave every result bit-identical, poses of distorted projections against ground truth and against OpenCV on
undistorted points, and the failure conventions.  Pure host code: runs without a GPU."""
import ctypes as C

import numpy as np
import pytest

import pose_records as PR
from test_field_pose import ROTATION, OFFSET, field_points, ours_cf, scene, tag_points

TAGSIZE = PR.TAGSIZE
CAM = (PR.FX, PR.FY, PR.CX, PR.CY)
K = np.array([[PR.FX, 0, PR.CX], [0, PR.FY, PR.CY], [0, 0, 1]])
WIDE = (-0.28, 0.08, 0.0006, 0.0, -0.01)                 # a wide-angle lens at 1280 x 800
REFERENCE = (0.059238, -0.075154, -0.003801, 0.001113, 0.0)  # the reference's test camera (p2 != 0)
TANGENTIAL = (0.0, 0.0, 0.002, -0.003, 0.0)
MODELS = {"wide": WIDE, "reference": REFERENCE, "tangential": TANGENTIAL}
STRONG_BARREL = (-0.5, 0.0, 0.0, 0.0, 0.0)  # folds at r^2 = 2/3: no distorted point beyond r' = 0.544 has a preimage
E_INVALID = -1


@pytest.fixture(scope="module")
def D():
    from ros_vision_b200 import build, detector
    build.build_native()
    detector.load_library()
    return detector


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def distort(cv2, px, dist):
    """Ideal pinhole pixels (N, 2) as the lens `dist` shows them (cv2.projectPoints)."""
    px = np.asarray(px, dtype=np.float64).reshape(-1, 2)
    rays = np.concatenate([(px - [PR.CX, PR.CY]) / [PR.FX, PR.FY], np.ones((len(px), 1))], axis=1)
    return cv2.projectPoints(rays, np.zeros(3), np.zeros(3), K, np.asarray(dist, dtype=np.float64))[0].reshape(-1, 2)


def undistort_iter(cv2, px, dist):
    """OpenCV's iterative undistortion run to convergence."""
    crit = (cv2.TERM_CRITERIA_COUNT | cv2.TERM_CRITERIA_EPS, 200, 1e-14)
    return cv2.undistortPointsIter(np.asarray(px, dtype=np.float64).reshape(-1, 1, 2), K, np.asarray(dist, dtype=np.float64),
                                   None, K, crit).reshape(-1, 2)


def frame_points(cv2, dist):
    """Ideal points whose distorted images cover the 1280 x 800 frame, corners included."""
    u, v = np.meshgrid(np.linspace(-200, 1480, 85), np.linspace(-150, 950, 56))
    ideal = np.stack([u.ravel(), v.ravel()], axis=1)
    seen = distort(cv2, ideal, dist)
    keep = (seen[:, 0] >= 0) & (seen[:, 0] <= 1280) & (seen[:, 1] >= 0) & (seen[:, 1] <= 800)
    return ideal[keep], seen[keep]


@pytest.mark.parametrize("model", sorted(MODELS))
def test_undistort_points_inverts_project_points(D, cv2, model):
    ideal, seen = frame_points(cv2, MODELS[model])
    assert len(ideal) > 2000
    got = D.undistort_points(seen, *CAM, MODELS[model])
    assert np.abs(got - ideal).max() <= 1e-9, np.abs(got - ideal).max()
    if model == "reference":
        # the reference's UnDistort inverts this model only when p2 = 0: here it is off by up to ~1 px
        ref = np.array([D.GpuDetector.UnDistort(u, v, (PR.FX, PR.CX, PR.FY, PR.CY), MODELS[model])[:2] for u, v in seen])
        assert np.abs(ref - ideal).max() > 0.1


def test_opencv_default_undistort_is_not_a_reference(D, cv2):
    """cv2.undistortPoints stops after 5 fixed-point iterations, which is far from the inverse near the corners of a
    wide-angle frame; undistortPointsIter run to convergence agrees with projectPoints' ground truth."""
    ideal, seen = frame_points(cv2, WIDE)
    five = cv2.undistortPoints(seen.reshape(-1, 1, 2), K, np.asarray(WIDE), P=K).reshape(-1, 2)
    assert np.abs(five - ideal).max() > 1.0
    assert np.abs(undistort_iter(cv2, seen, WIDE) - ideal).max() <= 1e-9
    assert np.abs(D.undistort_points(seen, *CAM, WIDE) - undistort_iter(cv2, seen, WIDE)).max() <= 1e-9


def test_points_past_the_fold_fail(D):
    r = np.array([0.3, 0.5, 0.54, 0.55, 0.6, 0.9])  # distorted radius; the model reaches 0.5443 at most
    seen = np.stack([PR.CX + PR.FX * r, np.full_like(r, PR.CY)], axis=1)
    got = D.undistort_points(seen, *CAM, STRONG_BARREL)
    assert np.isfinite(got[:3]).all() and np.isnan(got[3:]).all()
    x = (got[:3, 0] - PR.CX) / PR.FX
    assert np.abs(x * (1 - 0.5 * x * x) - r[:3]).max() <= 1e-9 and (x * x < 2 / 3).all()


def test_no_distortion_is_no_step(D):
    recs = PR.records(400, 31)
    pts = recs["p"].reshape(-1, 2)
    for dist in (None, [0.0] * 5):
        assert D.undistort_points(pts, *CAM, dist).tobytes() == pts.tobytes()
        for method in ("oi", "ippe"):
            want = D.estimate_poses(recs, TAGSIZE, *CAM, method=method)
            got = D.estimate_poses(recs, TAGSIZE, *CAM, method=method, distortion=dist)
            assert got.tobytes() == want.tobytes()
            lib = D.load_library()
            out = np.zeros(len(recs), dtype=D.POSE_DT)
            d = None if dist is None else np.zeros(5)
            assert lib.b200tag_estimate_poses_distorted(recs.ctypes.data_as(C.c_void_p), len(recs), D.POSE_METHODS[method],
                                                        TAGSIZE, *CAM, None if d is None else d.ctypes.data_as(C.c_void_p),
                                                        out.ctypes.data_as(C.c_void_p)) == 0
            assert out.tobytes() == want.tobytes()
    rng = np.random.default_rng(4)
    for trial in range(20):
        layout, dets, _, _ = scene(rng, int(rng.integers(1, 7)), 2, noise=0.3)
        want = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM, rotation=ROTATION, offset=OFFSET)
        for dist in (None, np.zeros(5)):
            got = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM, rotation=ROTATION, offset=OFFSET, distortion=dist)
            assert got.tobytes() == want.tobytes(), trial


def distorted_records(cv2, n, seed, dist, noise=0.0):
    """Tags of pose_records' kinds 0-2 (general, far near-frontal, near edge-on), seen through `dist`: (records, true
    R, true t, ideal corners)."""
    from ros_vision_b200 import detector as D
    rng = np.random.default_rng(seed)
    P = tag_points()
    out = np.zeros(n, dtype=D.DETECTION_DT)
    Rs, ts, ideal = np.zeros((n, 3, 3)), np.zeros((n, 3)), np.zeros((n, 4, 2))
    i = 0
    while i < n:
        kind = i % 3
        if kind == 1:
            R = PR.rot(np.pi + rng.uniform(-0.05, 0.05), rng.uniform(-0.05, 0.05), rng.uniform(-np.pi, np.pi))
            t = np.array([rng.uniform(-0.5, 0.5), rng.uniform(-0.3, 0.3), rng.uniform(4.0, 8.0)])
        elif kind == 2:
            tilt = rng.choice([-1, 1]) * rng.uniform(1.3, 1.5)
            R = PR.rot(np.pi + tilt, rng.uniform(-0.2, 0.2), rng.uniform(-np.pi, np.pi))
            t = np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2), rng.uniform(0.5, 2.0)])
        else:
            R = PR.rot(np.pi + rng.uniform(-0.6, 0.6), rng.uniform(-0.6, 0.6), rng.uniform(-np.pi, np.pi))
            z = rng.uniform(0.5, 4.0)
            t = np.array([rng.uniform(-0.6, 0.6) * z, rng.uniform(-0.4, 0.4) * z, z])
        cam = P @ R.T + t
        px = np.stack([PR.FX * cam[:, 0] / cam[:, 2] + PR.CX, PR.FY * cam[:, 1] / cam[:, 2] + PR.CY], axis=1)
        seen = distort(cv2, px, dist) + (rng.normal(0, noise, size=(4, 2)) if noise else 0)
        if not ((seen >= 0).all() and (seen[:, 0] <= 1280).all() and (seen[:, 1] <= 800).all()):
            continue
        out["p"][i] = seen
        out["H"][i] = PR.homography([(-1, 1), (1, 1), (1, -1), (-1, -1)], seen)
        out["c"][i] = seen.mean(axis=0)
        out["id"][i] = i % 587
        Rs[i], ts[i], ideal[i] = R, t, px
        i += 1
    return out, Rs, ts, ideal


@pytest.mark.parametrize("model", sorted(MODELS))
@pytest.mark.parametrize("method", ["oi", "ippe"])
def test_noise_free_poses_are_recovered(D, cv2, model, method):
    recs, Rs, ts, _ = distorted_records(cv2, 300, 40, MODELS[model])
    got = D.estimate_poses(recs, TAGSIZE, *CAM, method=method, distortion=MODELS[model])
    assert np.abs(got["R"] - Rs).max() <= 1e-9, np.abs(got["R"] - Rs).max()
    assert np.abs(got["t"] - ts).max() <= 1e-9, np.abs(got["t"] - ts).max()
    plain = D.estimate_poses(recs, TAGSIZE, *CAM, method=method)
    if model == "wide":  # without the correction the same records are far off
        assert np.abs(plain["t"] - ts).max() > 1e-2


def test_oi_reads_the_rebuilt_homography(D, cv2):
    """The OI start reads H: with distortion it is rebuilt from the undistorted corners (c = H (0, 0) too), so a
    record whose H is garbage gives the same pose as one with the right H."""
    recs, _, _, _ = distorted_records(cv2, 60, 41, WIDE)
    bad = recs.copy()
    bad["H"] = np.eye(3).reshape(9)
    bad["c"] = 0
    a = D.estimate_poses(recs, TAGSIZE, *CAM, distortion=WIDE)
    b = D.estimate_poses(bad, TAGSIZE, *CAM, distortion=WIDE)
    assert a.tobytes() == b.tobytes()


@pytest.mark.parametrize("model", sorted(MODELS))
def test_noisy_ippe_equals_opencv_on_undistorted_points(D, cv2, model):
    from test_pose_ippe import opencv_candidates
    recs, _, _, _ = distorted_records(cv2, 300, 42, MODELS[model], noise=0.3)
    got = D.estimate_poses(recs, TAGSIZE, *CAM, method="ippe", distortion=MODELS[model])
    worst = 0.0
    for i in range(len(recs)):
        cands = opencv_candidates(cv2, undistort_iter(cv2, recs["p"][i], MODELS[model]))
        dev = min(max(np.abs(got["R"][i] - R).max(), np.linalg.norm(got["t"][i] - t) / np.linalg.norm(t)) for R, t in cands)
        worst = max(worst, dev)
        assert dev <= 1e-7, (i, dev)
    print(f"worst deviation from OpenCV ({model}): {worst:.2e}")


def distorted_scene(cv2, rng, ntags, planes, dist, noise=0.0):
    """test_field_pose.scene with the corners seen through `dist`; tags that leave the frame are redrawn."""
    for _ in range(100):
        layout, dets, Rcf, tcf = scene(rng, ntags, planes)
        seen = distort(cv2, dets["p"].reshape(-1, 2), dist).reshape(-1, 4, 2)
        if (seen >= 0).all() and (seen[..., 0] <= 1280).all() and (seen[..., 1] <= 800).all():
            dets["p"] = seen + (rng.normal(0, noise, size=seen.shape) if noise else 0)
            dets["c"] = dets["p"].mean(axis=1)
            return layout, dets, Rcf, tcf
    raise AssertionError("no scene fits the frame")


@pytest.mark.parametrize("model", sorted(MODELS))
def test_noise_free_field_scenes_return_the_truth(D, cv2, model):
    rng = np.random.default_rng(50)
    for trial in range(30):
        layout, dets, Rcf, tcf = distorted_scene(cv2, rng, int(rng.integers(2, 9)), 1 + trial % 3, MODELS[model])
        out = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM, distortion=MODELS[model])
        assert out["num_tags"] == len(layout)
        R, t = ours_cf(out)
        assert np.abs(R - Rcf).max() <= 1e-9 and np.abs(t - tcf).max() <= 1e-9, trial
        assert out["rms"] < 1e-9


@pytest.mark.parametrize("model", sorted(MODELS))
def test_noisy_field_scenes_reach_opencvs_minimum(D, cv2, model):
    rng = np.random.default_rng(51)
    crit = (cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_COUNT, 200, 1e-15)
    for trial in range(30):
        layout, dets, _, _ = distorted_scene(cv2, rng, int(rng.integers(2, 9)), 1 + trial % 3, MODELS[model], noise=0.3)
        obj = field_points(layout)
        img = undistort_iter(cv2, dets["p"].reshape(-1, 2), MODELS[model])
        ok, rvec, tvec = cv2.solvePnP(obj, img, K, None, flags=cv2.SOLVEPNP_SQPNP)
        assert ok
        rvec, tvec = cv2.solvePnPRefineLM(obj, img, K, None, rvec, tvec, crit)
        Rcv, tcv = cv2.Rodrigues(rvec)[0], tvec.reshape(3)
        out = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM, distortion=MODELS[model])
        R, t = ours_cf(out)

        def cost(R, t):  # squared pixel error in the ideal image, where the solve measures rms
            cam = obj @ R.T + t
            return float(((np.stack([PR.FX * cam[:, 0] / cam[:, 2] + PR.CX, PR.FY * cam[:, 1] / cam[:, 2] + PR.CY], 1) - img) ** 2).sum())

        assert cost(R, t) <= cost(Rcv, tcv) * (1 + 1e-9), trial
        assert np.abs(R - Rcv).max() <= 1e-6 and np.abs(t - tcv).max() <= 1e-6 * np.linalg.norm(tcv), trial
        assert abs(out["rms"] - np.sqrt(cost(R, t) / len(obj))) <= 1e-6 * out["rms"]


def test_failing_corners(D, cv2):
    """A record with a corner past the fold gets R = I, t = 0, HUGE_VAL errors with both methods, and is left out of the
    field solve; a collapsed quad has no homography, which OI needs."""
    recs, _, _, _ = distorted_records(cv2, 8, 43, STRONG_BARREL)
    bad = recs.copy()
    bad["p"][::2, 1] = (PR.CX + 0.6 * PR.FX, PR.CY)  # beyond r' = 0.544
    for method in ("oi", "ippe"):
        got = D.estimate_poses(bad, TAGSIZE, *CAM, method=method, distortion=STRONG_BARREL)
        good = D.estimate_poses(recs[1::2], TAGSIZE, *CAM, method=method, distortion=STRONG_BARREL)
        assert got[1::2].tobytes() == good.tobytes()
        failed = got[::2]
        assert (failed["R"] == np.eye(3)).all() and (failed["t"] == 0).all()
        assert np.isinf(failed["err"]).all() and np.isinf(failed["err_other"]).all()
    collapsed = recs[:1].copy()
    collapsed["p"][0] = collapsed["p"][0, 0]
    got = D.estimate_poses(collapsed, TAGSIZE, *CAM, distortion=STRONG_BARREL)[0]
    assert (got["R"] == np.eye(3)).all() and np.isinf(got["err"])

    rng = np.random.default_rng(52)
    layout, dets, _, _ = distorted_scene(cv2, rng, 4, 2, WIDE, noise=0.3)
    base = D.estimate_field_pose(dets[1:], layout, TAGSIZE, *CAM, distortion=WIDE)
    dets["p"][0, 2] = (PR.CX + 3.0 * PR.FX, PR.CY)  # past the wide model's fold
    assert np.isnan(D.undistort_points(dets["p"][0], *CAM, WIDE)).any()
    got = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM, distortion=WIDE)
    assert got["num_tags"] == 3 and got.tobytes() == base.tobytes()


def test_invalid_arguments(D):
    lib = D.load_library()
    recs = PR.records(4, 44)
    out = np.zeros(4, dtype=D.POSE_DT)
    for bad in (np.nan, np.inf, -np.inf):
        d = np.array(WIDE, dtype=np.float64)
        d[3] = bad
        with pytest.raises(D.B200TagError):
            D.estimate_poses(recs, TAGSIZE, *CAM, distortion=d)
        with pytest.raises(D.B200TagError):
            D.undistort_points(recs["p"], *CAM, d)
        with pytest.raises(D.B200TagError):
            D.estimate_field_pose(recs, np.zeros(0, dtype=D.FIELD_TAG_DT), TAGSIZE, *CAM, distortion=d)
    d = np.array(WIDE)
    assert lib.b200tag_estimate_poses_distorted(recs.ctypes.data_as(C.c_void_p), 4, 2, TAGSIZE, *CAM,
                                                d.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)) == E_INVALID
    assert lib.b200tag_estimate_poses_distorted(recs.ctypes.data_as(C.c_void_p), 4, 1, 0.0, *CAM,
                                                d.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)) == E_INVALID
    with pytest.raises(ValueError):
        D.estimate_poses(recs, TAGSIZE, *CAM, distortion=WIDE[:4])
