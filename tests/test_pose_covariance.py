"""Pose covariances on the host (b200tag_estimate_pose_covariances, b200tag_estimate_field_pose_covariance): against an
independent numpy restatement (central finite differences of the projection, the undistortion's Jacobian by finite
differences of cv2.undistortPointsIter), the frame conventions, Monte Carlo runs of the field solve and of the OI and
IPPE tag poses, exactness and failures.  Pure host code: runs without a GPU."""
import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import pose_records as PR
from test_field_pose import OFFSET, ROTATION, project, scene, tag_points
from test_pose_distortion import K, distort, undistort_iter

TAGSIZE = PR.TAGSIZE
CAM = (PR.FX, PR.FY, PR.CX, PR.CY)
WIDE = (-0.28, 0.08, 0.0006, 0.0, -0.01)  # a wide-angle lens at 1280 x 800
SIGMA = 0.3
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


# ---- the numpy restatement ----

def perturbed(R, t, xi):
    """(exp([r]x) R, t + dt) for xi = (r, dt)."""
    return Rotation.from_rotvec(xi[:3]).as_matrix() @ R, t + xi[3:]


def pose_error(R, t, R0, t0):
    """xi with perturbed(R0, t0, xi) = (R, t)."""
    return np.concatenate([Rotation.from_matrix(R @ R0.T).as_rotvec(), t - t0])


def jacobian(f, n=6, h=1e-6):
    """Central differences of f(xi) (a flat array) at xi = 0."""
    cols = []
    for k in range(n):
        e = np.zeros(n)
        e[k] = h
        cols.append((f(e) - f(-e)) / (2 * h))
    return np.stack(cols, axis=1)


def undistortion_jacobians(cv2, raw, dist, h=1e-3):
    """A_i (2x2) of every raw corner: central differences of cv2.undistortPointsIter run to 1e-14."""
    raw = np.asarray(raw, dtype=np.float64).reshape(-1, 2)
    A = np.zeros((len(raw), 2, 2))
    for k in range(2):
        e = np.zeros(2)
        e[k] = h
        A[:, :, k] = (undistort_iter(cv2, raw + e, dist) - undistort_iter(cv2, raw - e, dist)) / (2 * h)
    return A


def sandwich(J, A, sigma):
    """sigma^2 M^-1 B M^-1 over the 2x6 blocks of J (2n x 6); A: (n, 2, 2) or None (A_i = I)."""
    Mi = np.linalg.inv(J.T @ J)
    if A is None:
        return sigma ** 2 * Mi
    B = sum(Ji.T @ Ai @ Ai.T @ Ji for Ji, Ai in zip(J.reshape(-1, 2, 6), A))
    return sigma ** 2 * Mi @ B @ Mi


def tag_reference(cv2, det, pose, dist, sigma):
    """The tag pose's covariance, camera frame."""
    P = tag_points()
    R0, t0 = pose["R"], pose["t"]
    J = jacobian(lambda xi: project(P @ perturbed(R0, t0, xi)[0].T + perturbed(R0, t0, xi)[1]).ravel())
    A = None if dist is None else undistortion_jacobians(cv2, det["p"], dist)
    return sandwich(J, A, sigma)


def robot_of(Rc, tc):
    Rr = Rc @ ROTATION.T
    return Rr, tc - Rr @ OFFSET


def field_reference(cv2, layout, dets, out, dist, sigma):
    """(camera, robot) covariances of field record `out`, both in the field frame; J perturbs the camera in the field
    directly, and the robot's G comes from finite differences of the camera -> robot mapping."""
    obj = np.concatenate([tag_points() @ np.asarray(L["R"]).T + L["t"] for L in layout])
    Rc, tc = out["camera_R"], out["camera_t"]

    def proj(xi):
        R, t = perturbed(Rc, tc, xi)
        return project((obj - t) @ R).ravel()  # X_cam = R^T (X_field - t)
    raw = np.concatenate([d["p"] for d in dets])
    A = None if dist is None else undistortion_jacobians(cv2, raw, dist)
    Cc = sandwich(jacobian(proj), A, sigma)
    Rr0, tr0 = robot_of(Rc, tc)
    G = jacobian(lambda xi: pose_error(*robot_of(*perturbed(Rc, tc, xi)), Rr0, tr0))
    return Cc, G @ Cc @ G.T, G


def assert_close(C, ref, tol=1e-6):
    """Entries within tol of the reference, relative to sqrt(C_ii C_jj)."""
    d = np.sqrt(np.abs(np.diag(ref)))
    rel = np.abs(C - ref) / np.outer(d, d)
    assert rel.max() <= tol, rel.max()


def tag_records(rng, n, zmax=3.0, min_tilt=15.0):
    """`n` detections of tags 0.5..zmax m away, tilted at least min_tilt deg from head-on, their noise-free corners."""
    from ros_vision_b200 import detector as Dm
    dets = np.zeros(n, dtype=Dm.DETECTION_DT)
    truth = []
    P = tag_points()
    while len(truth) < n:
        R = PR.rot(np.pi + rng.uniform(-0.9, 0.9), rng.uniform(-0.9, 0.9), rng.uniform(-np.pi, np.pi))
        t = np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2), 1.0]) * rng.uniform(0.5, zmax)
        tilt = np.degrees(np.arccos(abs(R[2, 2])))
        px = project(P @ R.T + t)
        if tilt < min_tilt or (px < 0).any() or (px[:, 0] > 1280).any() or (px[:, 1] > 800).any():
            continue
        i = len(truth)
        dets["p"][i] = px
        dets["c"][i] = px.mean(axis=0)
        dets["H"][i] = PR.homography([(-1, 1), (1, 1), (1, -1), (-1, -1)], px)
        truth.append((R, t))
    return dets, truth


# ---- 1, 2: the formula, the Jacobian and the frames ----

@pytest.mark.parametrize("method", ["oi", "ippe"])
@pytest.mark.parametrize("lens", [None, WIDE])
def test_tag_covariance_equals_the_restatement(D, cv2, method, lens):
    rng = np.random.default_rng(1)
    dets, _ = tag_records(rng, 40)
    if lens is not None:
        dets["p"] = distort(cv2, dets["p"].reshape(-1, 2), lens).reshape(-1, 4, 2)
    dets["p"] += rng.normal(0, 0.3, size=dets["p"].shape)
    poses = D.estimate_poses(dets, TAGSIZE, *CAM, method=method, distortion=lens)
    cov = D.estimate_pose_covariances(dets, poses, TAGSIZE, *CAM, SIGMA, distortion=lens)
    for i in range(len(dets)):
        assert_close(cov["C"][i], tag_reference(cv2, dets[i], poses[i], lens, SIGMA))


@pytest.mark.parametrize("lens", [None, WIDE])
@pytest.mark.parametrize("ntags,planes", [(1, 1), (3, 1), (5, 2), (8, 3)])
def test_field_covariance_equals_the_restatement(D, cv2, lens, ntags, planes):
    rng = np.random.default_rng(2 + ntags)
    for trial in range(8):
        layout, dets, _, _ = scene(rng, ntags, planes, noise=0.3)
        if lens is not None:
            dets["p"] = distort(cv2, dets["p"].reshape(-1, 2), lens).reshape(-1, 4, 2)
        out, cov = D.estimate_field_pose_covariance(dets, layout, TAGSIZE, *CAM, SIGMA, rotation=ROTATION, offset=OFFSET,
                                                    distortion=lens)
        assert out["num_tags"] == ntags
        assert out.tobytes() == D.estimate_field_pose(dets, layout, TAGSIZE, *CAM, rotation=ROTATION, offset=OFFSET,
                                                      distortion=lens).tobytes()
        Cc, Cr, G = field_reference(cv2, layout, dets, out, lens, SIGMA)
        assert_close(cov["camera"], Cc)
        assert_close(cov["robot"], Cr)
        assert_close(cov["robot"], G @ cov["camera"] @ G.T, 1e-9)


def test_pose2d_stddevs(D):
    C = np.diag([1.0, 4.0, 9.0, 16.0, 25.0, 36.0])
    assert D.pose2d_stddevs(C) == (4.0, 5.0, 3.0)


# ---- 3, 4: Monte Carlo ----

def monte_carlo(errors, covs):
    """(mean Mahalanobis^2, per-component empirical / predicted standard deviation)."""
    errors, covs = np.asarray(errors), np.asarray(covs)
    m2 = np.einsum("ni,nij,nj->n", errors, np.linalg.inv(covs), errors)
    ratio = errors.std(axis=0) / np.sqrt(np.diagonal(covs, axis1=1, axis2=2).mean(axis=0))
    return float(m2.mean()), ratio


def field_monte_carlo(D, cv2, layout, ideal, truth, lens, trials, rng, without_lens=False):
    """Field solves of `trials` noisy copies of the ideal corners (seen through `lens` when given)."""
    Rc, tc = truth
    errors, covs = [], []
    dets = ideal.copy()
    seen = ideal["p"] if lens is None else distort(cv2, ideal["p"].reshape(-1, 2), lens).reshape(ideal["p"].shape)
    for _ in range(trials):
        dets["p"] = seen + rng.normal(0, SIGMA, size=seen.shape)
        out, cov = D.estimate_field_pose_covariance(dets, layout, TAGSIZE, *CAM, SIGMA, distortion=lens)
        C = cov["camera"]
        if without_lens:  # the same pose with A_i = I: the solve on the undistorted corners, without the lens
            und = dets.copy()
            und["p"] = D.undistort_points(dets["p"], *CAM, lens)
            out2, cov2 = D.estimate_field_pose_covariance(und, layout, TAGSIZE, *CAM, SIGMA)
            assert out2.tobytes() == out.tobytes()
            C = cov2["camera"]
        errors.append(pose_error(out["camera_R"], out["camera_t"], Rc, tc))
        covs.append(C)
    return monte_carlo(errors, covs)


def field_cases(rng):
    """(name, layout, noise-free detections, camera in the field): 2-8 tags on one to three planes, and single tags far
    from ambiguity (tilted more than 30 deg, at most 2 m away)."""
    out = []
    for ntags, planes in [(2, 1), (4, 2), (8, 3)]:
        layout, dets, Rcf, tcf = scene(rng, ntags, planes)
        out.append((f"{ntags} tags, {planes} planes", layout, dets, (Rcf.T, -Rcf.T @ tcf)))
    while len(out) < 5:
        layout, dets, Rcf, tcf = scene(rng, 1, 1, zmin=0.5, zmax=2.0)
        Rt = np.asarray(layout["R"][0]).T @ Rcf.T  # tag-from-camera
        if np.degrees(np.arccos(abs(Rt[2, 2]))) > 30:
            out.append(("1 tag", layout, dets, (Rcf.T, -Rcf.T @ tcf)))
    return out


@pytest.mark.parametrize("case", range(5))
def test_field_monte_carlo(D, cv2, case):
    rng = np.random.default_rng(30)
    name, layout, dets, truth = field_cases(rng)[case]
    m2, ratio = field_monte_carlo(D, cv2, layout, dets, truth, None, 2000, np.random.default_rng(31 + case))
    print(f"field, {name}: mean Mahalanobis^2 {m2:.3f}, std ratios {np.round(ratio, 3)}")
    assert 5.6 <= m2 <= 6.4 and (0.9 <= ratio).all() and (ratio <= 1.1).all(), (m2, ratio)


def edge_case(D, cv2, rng, ntags, planes):
    """A scene within 3.5 m whose tags sit towards the frame's corners of the wide-angle lens, where A_i is far from I:
    (layout, ideal corners, camera in the field)."""
    while True:
        layout, ideal, Rcf, tcf = scene(rng, ntags, planes, zmax=3.5)
        seen = distort(cv2, ideal["p"].reshape(-1, 2), WIDE).reshape(-1, 4, 2)
        r = np.hypot(seen[..., 0] - PR.CX, seen[..., 1] - PR.CY)
        inside = (seen >= 0).all() and (seen[..., 0] <= 1280).all() and (seen[..., 1] <= 800).all()
        if inside and (r.min(axis=1) > 420).all():
            return layout, ideal, (Rcf.T, -Rcf.T @ tcf)


@pytest.mark.parametrize("ntags,planes", [(3, 1), (4, 2)])
def test_field_monte_carlo_through_the_lens(D, cv2, ntags, planes):
    """Through the wide-angle lens: the covariance with A_i passes; the same pose's covariance without A_i fails."""
    rng = np.random.default_rng(40 + ntags)
    layout, ideal, truth = edge_case(D, cv2, rng, ntags, planes)
    m2, ratio = field_monte_carlo(D, cv2, layout, ideal, truth, WIDE, 2000, np.random.default_rng(41))
    print(f"field through the lens, {ntags} tags: mean Mahalanobis^2 {m2:.3f}, std ratios {np.round(ratio, 3)}")
    assert 5.6 <= m2 <= 6.4 and (0.9 <= ratio).all() and (ratio <= 1.1).all(), (m2, ratio)
    m2, ratio = field_monte_carlo(D, cv2, layout, ideal, truth, WIDE, 2000, np.random.default_rng(41), without_lens=True)
    print(f"  without A_i: mean Mahalanobis^2 {m2:.3f}, std ratios {np.round(ratio, 3)}")
    assert not (5.6 <= m2 <= 6.4 and (0.9 <= ratio).all() and (ratio <= 1.1).all()), (m2, ratio)


@pytest.mark.parametrize("method", ["oi", "ippe"])
def test_tag_monte_carlo(D, method):
    """OI and IPPE are not the pixel least-squares estimate; the ratios are recorded in DESIGN.md section 9.  A tag
    far off can come back on the other branch of its planar ambiguity, an error the local covariance does not describe:
    such trials (Mahalanobis^2 > 40, which the right branch reaches with probability 3e-7) are counted, held to 2 %,
    and left out of the ratios."""
    rng = np.random.default_rng(50)
    dets, truth = tag_records(rng, 12)
    lo, hi, flipped = 1.0, 1.0, 0
    for i in range(len(dets)):
        trials = np.repeat(dets[i:i + 1], 2000)
        trials["p"] += rng.normal(0, SIGMA, size=trials["p"].shape)
        poses = D.estimate_poses(trials, TAGSIZE, *CAM, method=method)
        cov = D.estimate_pose_covariances(trials, poses, TAGSIZE, *CAM, SIGMA)["C"]
        R0, t0 = truth[i]
        errors = np.array([pose_error(p["R"], p["t"], R0, t0) for p in poses])
        flips = np.einsum("ni,nij,nj->n", errors, np.linalg.inv(cov), errors) > 40
        m2, ratio = monte_carlo(errors[~flips], cov[~flips])
        print(f"{method}, tag {i} at {np.linalg.norm(t0):.2f} m: {flips.sum()} flips, mean Mahalanobis^2 {m2:.3f}, "
              f"std ratios {np.round(ratio, 3)}")
        lo, hi, flipped = min(lo, ratio.min()), max(hi, ratio.max()), flipped + flips.sum()
        assert flips.sum() <= 40 and (0.8 <= ratio).all() and (ratio <= 1.25).all(), (i, flips.sum(), m2, ratio)
    print(f"{method}: std ratios {lo:.3f}..{hi:.3f}, {flipped} of {2000 * len(dets)} trials on the other branch")


# ---- 5: exactness and failures ----

def test_exactly_symmetric_positive_definite_and_scaled_last(D, cv2):
    rng = np.random.default_rng(60)
    dets, _ = tag_records(rng, 50)
    for lens in (None, WIDE):
        poses = D.estimate_poses(dets, TAGSIZE, *CAM, method="ippe", distortion=lens)
        c1 = D.estimate_pose_covariances(dets, poses, TAGSIZE, *CAM, 0.3, distortion=lens)["C"]
        c2 = D.estimate_pose_covariances(dets, poses, TAGSIZE, *CAM, 0.6, distortion=lens)["C"]
        assert (c1 == np.swapaxes(c1, 1, 2)).all()
        assert (np.linalg.eigvalsh(c1) > 0).all()
        assert (c2 == 4 * c1).all()
        layout, fd, _, _ = scene(rng, 4, 2, noise=0.3)
        _, f1 = D.estimate_field_pose_covariance(fd, layout, TAGSIZE, *CAM, 0.3, rotation=ROTATION, offset=OFFSET, distortion=lens)
        _, f2 = D.estimate_field_pose_covariance(fd, layout, TAGSIZE, *CAM, 0.6, rotation=ROTATION, offset=OFFSET, distortion=lens)
        for k in ("camera", "robot"):
            assert (f1[k] == f1[k].T).all() and (np.linalg.eigvalsh(f1[k]) > 0).all() and (f2[k] == 4 * f1[k]).all()


def test_failures_give_huge_val(D):
    recs = PR.records(400, 61)  # every 4th record a collapsed quad
    poses = D.estimate_poses(recs, TAGSIZE, *CAM)
    cov = D.estimate_pose_covariances(recs, poses, TAGSIZE, *CAM, SIGMA)
    failed = np.isinf(poses["err"])
    assert failed.sum() >= 50
    assert np.isinf(cov["C"][failed]).all()
    # collapsed quads with a pose from IPPE, which fails them too
    ippe = D.estimate_poses(recs, TAGSIZE, *CAM, method="ippe")
    cov = D.estimate_pose_covariances(recs, ippe, TAGSIZE, *CAM, SIGMA)
    assert np.isinf(cov["C"][3::4]).all()
    ok = ~np.isinf(ippe["err"])
    assert np.isfinite(cov["C"][ok]).all()
    # a corner behind the camera
    behind = poses[~failed][:5].copy()
    behind["t"][:, 2] = -1.0
    assert np.isinf(D.estimate_pose_covariances(recs[~failed][:5], behind, TAGSIZE, *CAM, SIGMA)["C"]).all()
    # a field pose without tags
    from ros_vision_b200 import detector as Dm
    out, fc = D.estimate_field_pose_covariance(recs[:0], np.zeros(0, dtype=Dm.FIELD_TAG_DT), TAGSIZE, *CAM, SIGMA)
    assert out["num_tags"] == 0 and np.isinf(fc["camera"]).all() and np.isinf(fc["robot"]).all()


@pytest.mark.parametrize("sigma", [0.0, -1.0, np.nan, np.inf])
def test_bad_sigma_is_rejected(D, sigma):
    import ctypes as C
    lib = D.load_library()
    recs = PR.records(4, 62)
    poses = D.estimate_poses(recs, TAGSIZE, *CAM)
    out = np.zeros(4, dtype=D.COVARIANCE_DT)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    assert lib.b200tag_estimate_pose_covariances(ptr(recs), ptr(poses), 4, TAGSIZE, *CAM, None, sigma, ptr(out)) == E_INVALID
    layout, dets, _, _ = scene(np.random.default_rng(63), 2, 1)
    fp = np.zeros(1, dtype=D.FIELD_POSE_DT)
    fc = np.zeros(1, dtype=D.FIELD_COVARIANCE_DT)
    assert lib.b200tag_estimate_field_pose_covariance(ptr(dets), 2, ptr(layout), 2, TAGSIZE, *CAM, None, None, None, sigma,
                                                      ptr(fp), ptr(fc)) == E_INVALID
