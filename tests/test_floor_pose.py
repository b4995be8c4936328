"""The floor pose (b200tag_estimate_floor_pose, detector.estimate_floor_pose) on the host: ground truth in the three
modes, scipy's least squares over the same residuals, the planar ambiguity of a single far tag, the covariance against
a numpy restatement and in Monte Carlo runs, and argument checks.  Pure host code: runs without a GPU."""
import math

import numpy as np
import pytest

import pose_records as PR
from test_field_pose import OFFSET, ROTATION, project, tag_points
from test_pose_covariance import assert_close, undistortion_jacobians
from test_pose_distortion import K, distort, undistort_iter

TAGSIZE = PR.TAGSIZE
CAM = (PR.FX, PR.FY, PR.CX, PR.CY)
WIDE = (-0.28, 0.08, 0.0006, 0.0, -0.01)  # a wide-angle lens at 1280 x 800
SIGMA = 0.3
WEIGHT = 0.3 / 0.02  # corner noise 0.3 px over a gyro good to 0.02 rad
E_INVALID = -1
MODES = {"free": (False, np.inf), "prior": (True, WEIGHT), "fixed": (True, np.inf)}


@pytest.fixture(scope="module")
def D():
    from ros_vision_b200 import build, detector
    build.build_native()
    detector.load_library()
    return detector


@pytest.fixture(scope="module")
def cv2():
    return pytest.importorskip("cv2")


def Rz(theta):
    return np.array([[np.cos(theta), -np.sin(theta), 0], [np.sin(theta), np.cos(theta), 0], [0, 0, 1]])


def camera_of(x, y, theta):
    """The camera in the field of a robot at (x, y, theta) on the floor: (camera_R, camera_t)."""
    return Rz(theta) @ ROTATION, np.array([x, y, 0.0]) + Rz(theta) @ OFFSET


def floor_scene(rng, ntags, planes, noise=0.0, zmin=1.0, zmax=6.0, dist=None):
    """A robot at a random (x, y, theta) on the floor and `ntags` layout tags in front of its camera on `planes` planes.
    Returns (layout, detections, (x, y, theta)); with `dist` the corners are seen through that lens."""
    from ros_vision_b200 import detector as Dm
    while True:
        truth = (rng.uniform(0, 16), rng.uniform(0, 8), rng.uniform(-np.pi, np.pi))
        cR, ct = camera_of(*truth)
        layout = np.zeros(ntags, dtype=Dm.FIELD_TAG_DT)
        dets = np.zeros(ntags, dtype=Dm.DETECTION_DT)
        ids = rng.choice(587, size=ntags, replace=False)
        plane_R = [PR.rot(*rng.uniform(-0.6, 0.6, size=3)) for _ in range(planes)]
        plane_t = [np.array([rng.uniform(-0.4, 0.4), rng.uniform(-0.3, 0.3), 1.0]) * rng.uniform(zmin + 0.5, zmax - 0.5)
                   for _ in range(planes)]
        P = tag_points()
        for j in range(ntags):
            k = j % planes
            for _ in range(1000):
                t = plane_t[k] + plane_R[k] @ np.array([rng.uniform(-1.5, 1.5), rng.uniform(-1.0, 1.0), 0.0])
                cam = P @ plane_R[k].T + t
                px = project(cam) if (cam[:, 2] > zmin).all() and (cam[:, 2] < zmax).all() else None
                if px is not None and (px >= 0).all() and (px[:, 0] < 1280).all() and (px[:, 1] < 800).all():
                    break
            layout["id"][j] = ids[j]
            layout["R"][j] = cR @ plane_R[k]
            layout["t"][j] = cR @ t + ct
            dets["id"][j] = ids[j]
            dets["decision_margin"][j] = 100.0
            dets["p"][j] = px
        if dist is not None:
            import cv2 as cv
            seen = distort(cv, dets["p"].reshape(-1, 2), dist).reshape(-1, 4, 2)
            if not ((seen >= 0).all() and (seen[..., 0] <= 1280).all() and (seen[..., 1] <= 800).all()):
                continue
            dets["p"] = seen
        dets["p"] += rng.normal(0, noise, size=dets["p"].shape) if noise else 0
        dets["c"] = dets["p"].mean(axis=1)
        return layout, dets, truth


def field_points(layout):
    return np.concatenate([tag_points() @ np.asarray(L["R"]).T + L["t"] for L in layout])


def pixels(obj, x, y, theta):
    """Ideal-image projections of field points at robot pose (x, y, theta)."""
    cR, ct = camera_of(x, y, theta)
    return project((obj - ct) @ cR)


def rho(theta, heading, weight):
    c, s, cg, sg = np.cos(theta), np.sin(theta), np.cos(heading), np.sin(heading)
    return weight * 2 * (s * cg - c * sg) / (1 + c * cg + s * sg)


def wrap(a):
    return (a + np.pi) % (2 * np.pi) - np.pi


def solve(D, dets, layout, mode, heading, **kw):
    given, weight = MODES[mode]
    return D.estimate_floor_pose(dets, layout, TAGSIZE, *CAM, rotation=ROTATION, offset=OFFSET,
                                 heading=heading if given else np.nan, heading_weight=weight, **kw)


# ---- 1: ground truth ----

@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("ntags,planes", [(1, 1), (2, 1), (5, 2), (8, 3)])
def test_noise_free_scenes_return_the_truth(D, mode, ntags, planes):
    rng = np.random.default_rng(ntags * 10 + planes)
    for trial in range(25):
        layout, dets, (x, y, th) = floor_scene(rng, ntags, planes, zmax=4.0 if ntags == 1 else 6.0)
        out, cov = solve(D, dets, layout, mode, th)
        assert out["num_tags"] == ntags and out["mode"] == list(MODES).index(mode)
        assert abs(out["x"] - x) <= 1e-9 and abs(out["y"] - y) <= 1e-9, (trial, out)
        assert abs(wrap(out["heading"] - th)) <= 1e-9, trial
        assert out["heading"] == math.atan2(out["sin_heading"], out["cos_heading"])
        assert out["rms"] < 1e-9 and cov is None
        assert (out["rms_other"] == np.inf) == (mode != "free" or ntags > 1)


# ---- 2: an independent restatement ----

def scipy_solve(obj, img, mode, heading, x0):
    from scipy.optimize import least_squares
    given, weight = MODES[mode]

    def res(q):
        th = heading if mode == "fixed" else q[2]
        r = (pixels(obj, q[0], q[1], th) - img).ravel()
        return np.append(r, rho(th, heading, weight)) if mode == "prior" else r
    q0 = np.asarray(x0[:2] if mode == "fixed" else x0, dtype=np.float64)
    sol = least_squares(res, q0, method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=10000)
    return sol.x, float(2 * sol.cost)


def our_cost(out, obj, img, mode, heading):
    r = float(((pixels(obj, out["x"], out["y"], out["heading"]) - img) ** 2).sum())
    return r + (rho(out["heading"], heading, WEIGHT) ** 2 if mode == "prior" else 0.0)


@pytest.mark.parametrize("lens", [None, WIDE])
@pytest.mark.parametrize("mode", list(MODES))
def test_noisy_scenes_equal_scipy_least_squares(D, cv2, mode, lens):
    rng = np.random.default_rng(50 + list(MODES).index(mode))
    for trial in range(30):
        ntags, planes = [(1, 1), (3, 1), (5, 2), (8, 3)][trial % 4]
        layout, dets, truth = floor_scene(rng, ntags, planes, noise=SIGMA, zmax=4.0 if ntags == 1 else 6.0, dist=lens)
        heading = truth[2] + (rng.normal(0, 0.02) if mode == "prior" else 0.0)
        obj = field_points(layout)
        img = dets["p"].reshape(-1, 2) if lens is None else undistort_iter(cv2, dets["p"].reshape(-1, 2), lens)
        out, _ = solve(D, dets, layout, mode, heading, distortion=lens)
        q, c_sp = scipy_solve(obj, img, mode, heading, truth)
        c_ours = our_cost(out, obj, img, mode, heading)
        assert c_ours <= c_sp * (1 + 1e-9) + 1e-18, (trial, c_ours, c_sp)
        if ntags == 1 and mode == "free" and abs(out["rms"] - out["rms_other"]) < 0.05:
            continue  # two nearly equal branches: scipy from the truth may stay on the other one
        assert abs(out["x"] - q[0]) <= 1e-6 and abs(out["y"] - q[1]) <= 1e-6, (trial, out, q)
        if mode != "fixed":
            assert abs(wrap(out["heading"] - q[2])) <= 1e-6, trial
        n = 4 * ntags
        pix = float(((pixels(obj, out["x"], out["y"], out["heading"]) - img) ** 2).sum())
        assert abs(out["rms"] - np.sqrt(pix / n)) <= 1e-6 * out["rms"] + 1e-12


@pytest.mark.parametrize("lens", [None, WIDE])
def test_free_mode_cost_is_not_below_the_field_pose(D, lens):
    rng = np.random.default_rng(60)
    for trial in range(40):
        ntags, planes = [(1, 1), (2, 1), (4, 2), (6, 3)][trial % 4]
        layout, dets, truth = floor_scene(rng, ntags, planes, noise=SIGMA, dist=lens)
        out, _ = solve(D, dets, layout, "free", np.nan, distortion=lens)
        field = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM, rotation=ROTATION, offset=OFFSET, distortion=lens)
        assert out["num_tags"] == field["num_tags"]
        assert out["rms"] >= field["rms"] * (1 - 1e-9), trial


# ---- 3: the planar ambiguity of a single far tag ----

def far_tag(rng):
    """One tag 2.7-2.9 m in front of the camera, turned more than 15 deg from head-on."""
    while True:
        R = PR.rot(rng.uniform(-0.6, 0.6), rng.uniform(-0.6, 0.6), rng.uniform(-0.3, 0.3))
        if np.degrees(np.arccos(abs(R[2, 2]))) > 15:
            break
    d = rng.uniform(2.7, 2.9)
    t = np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2), 1.0])
    return R, t / np.linalg.norm(t) * d


def test_single_far_tag_ambiguity(D):
    from ros_vision_b200 import detector as Dm
    rng = np.random.default_rng(70)
    counts = {"6-DOF": 0, "free": 0, "fixed": 0}
    trials = 2000
    cases = 20
    for case in range(cases):
        R, t = far_tag(rng)
        truth = (rng.uniform(0, 16), rng.uniform(0, 8), rng.uniform(-np.pi, np.pi))
        cR, ct = camera_of(*truth)
        layout = np.zeros(1, dtype=Dm.FIELD_TAG_DT)
        layout["R"][0], layout["t"][0] = cR @ R, cR @ t + ct
        ideal = np.zeros(1, dtype=Dm.DETECTION_DT)
        ideal["p"][0] = project(tag_points() @ R.T + t)
        # predicted robot x / y standard deviations at the truth, per estimator
        _, fc = D.estimate_field_pose_covariance(ideal, layout, TAGSIZE, *CAM, SIGMA, rotation=ROTATION, offset=OFFSET)
        sd = {"6-DOF": np.sqrt(np.diag(fc["robot"])[3:5])}
        for mode in ("free", "fixed"):
            sd[mode] = np.sqrt(np.diag(solve(D, ideal, layout, mode, truth[2], sigma=SIGMA)[1])[:2])
        dets = ideal.copy()
        for _ in range(trials // cases):
            dets["p"] = ideal["p"] + rng.normal(0, SIGMA, size=ideal["p"].shape)
            f = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM, rotation=ROTATION, offset=OFFSET)
            err = {"6-DOF": f["robot_t"][:2] - truth[:2]}
            for mode in ("free", "fixed"):
                out, _ = solve(D, dets, layout, mode, truth[2])
                err[mode] = np.array([out["x"], out["y"]]) - truth[:2]
            for k in counts:
                counts[k] += int((np.abs(err[k]) > 10 * sd[k]).any())
    print(f"single tag 2.7-2.9 m, {trials} trials, wrong-branch counts: {counts}")
    assert counts["fixed"] == 0, counts
    assert counts["free"] <= counts["6-DOF"], counts


# ---- 4: the covariance ----

def floor_reference(cv2, layout, dets, out, mode, heading, dist, sigma):
    """sigma^2 H^-1 M H^-1 by central differences over (x, y, theta), g by differences of rho."""
    obj = field_points(layout)
    q0 = np.array([out["x"], out["y"], out["heading"]])
    h = 1e-6
    J = np.stack([(pixels(obj, *(q0 + e)) - pixels(obj, *(q0 - e))).ravel() / (2 * h) for e in np.eye(3) * h], axis=1)
    g = np.zeros(3)
    if mode == "prior":
        g[2] = (rho(q0[2] + h, heading, WEIGHT) - rho(q0[2] - h, heading, WEIGHT)) / (2 * h)
    n = 2 if mode == "fixed" else 3
    J, g = J[:, :n], g[:n]
    H = J.T @ J + np.outer(g, g)
    if dist is None:
        M = H
    else:
        A = undistortion_jacobians(cv2, dets["p"].reshape(-1, 2), dist)
        M = sum(Ji.T @ Ai @ Ai.T @ Ji for Ji, Ai in zip(J.reshape(-1, 2, n), A)) + np.outer(g, g)
    Hi = np.linalg.inv(H)
    C = np.zeros((3, 3))
    C[:n, :n] = sigma ** 2 * Hi @ M @ Hi
    return C


@pytest.mark.parametrize("lens", [None, WIDE])
@pytest.mark.parametrize("mode", list(MODES))
def test_covariance_equals_the_restatement(D, cv2, mode, lens):
    rng = np.random.default_rng(80)
    for trial in range(12):
        ntags, planes = [(1, 1), (3, 1), (5, 2), (8, 3)][trial % 4]
        layout, dets, truth = floor_scene(rng, ntags, planes, noise=SIGMA, zmax=4.0 if ntags == 1 else 6.0, dist=lens)
        heading = truth[2] + rng.normal(0, 0.02)
        out, cov = solve(D, dets, layout, mode, heading, distortion=lens, sigma=SIGMA)
        plain, none = solve(D, dets, layout, mode, heading, distortion=lens)
        assert out.tobytes() == plain.tobytes() and none is None
        ref = floor_reference(cv2, layout, dets, out, mode, heading, lens, SIGMA)
        if mode == "fixed":
            assert (cov[2] == 0).all() and (cov[:, 2] == 0).all()
            assert_close(cov[:2, :2], ref[:2, :2])
        else:
            assert_close(cov, ref)
        assert (cov == cov.T).all()


def floor_cases(rng):
    out = []
    for ntags, planes in [(2, 1), (4, 2), (8, 3)]:
        out.append((f"{ntags} tags, {planes} planes",) + floor_scene(rng, ntags, planes))
    while len(out) < 4:  # a near single tag, well away from its ambiguity
        layout, dets, truth = floor_scene(rng, 1, 1, zmin=0.5, zmax=2.0)
        cR, _ = camera_of(*truth)
        Rt = np.asarray(layout["R"][0]).T @ cR
        if np.degrees(np.arccos(abs(Rt[2, 2]))) > 30:
            out.append(("1 tag", layout, dets, truth))
    return out


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("case", range(4))
def test_monte_carlo(D, mode, case):
    rng = np.random.default_rng(90)
    name, layout, ideal, truth = floor_cases(rng)[case]
    rng = np.random.default_rng(91 + case)
    n = 2 if mode == "fixed" else 3
    errors, covs = [], []
    dets = ideal.copy()
    for _ in range(2000):
        dets["p"] = ideal["p"] + rng.normal(0, SIGMA, size=ideal["p"].shape)
        heading = truth[2] + (rng.normal(0, SIGMA / WEIGHT) if mode == "prior" else 0.0)
        out, cov = solve(D, dets, layout, mode, heading, sigma=SIGMA)
        errors.append(np.array([out["x"] - truth[0], out["y"] - truth[1], wrap(out["heading"] - truth[2])])[:n])
        covs.append(cov[:n, :n])
    errors, covs = np.asarray(errors), np.asarray(covs)
    m2 = float(np.einsum("ni,nij,nj->n", errors, np.linalg.inv(covs), errors).mean())
    ratio = errors.std(axis=0) / np.sqrt(np.diagonal(covs, axis1=1, axis2=2).mean(axis=0))
    print(f"floor {mode}, {name}: mean Mahalanobis^2 {m2:.3f}, std ratios {np.round(ratio, 3)}")
    lo, hi = (1.85, 2.15) if mode == "fixed" else (2.8, 3.2)
    assert lo <= m2 <= hi and (0.9 <= ratio).all() and (ratio <= 1.1).all(), (m2, ratio)


def test_covariance_is_scaled_last(D):
    rng = np.random.default_rng(95)
    for mode in MODES:
        for lens in (None, WIDE):
            layout, dets, truth = floor_scene(rng, 3, 2, noise=SIGMA, dist=lens)
            _, c1 = solve(D, dets, layout, mode, truth[2], distortion=lens, sigma=SIGMA)
            _, c2 = solve(D, dets, layout, mode, truth[2], distortion=lens, sigma=2 * SIGMA)
            assert (c2 == 4 * c1).all()


def test_pose2d_stddevs_of_a_floor_covariance(D):
    assert D.pose2d_stddevs(np.diag([4.0, 9.0, 16.0])) == (2.0, 3.0, 4.0)


# ---- failures and arguments ----

def test_no_usable_tag(D):
    layout, dets, truth = floor_scene(np.random.default_rng(3), 2, 1)
    for mode in MODES:
        out, cov = solve(D, dets[:0], layout, mode, truth[2], sigma=SIGMA)
        assert out["num_tags"] == 0 and out["x"] == 0 and out["y"] == 0 and out["heading"] == 0
        assert out["rms"] == np.inf and out["rms_other"] == np.inf and (cov == np.inf).all()


def test_heading_opposite_the_gyro_is_not_a_seed_winner(D):
    """A prior 180 deg off the truth makes E HUGE_VAL near the truth; the solve still returns a finite pose."""
    layout, dets, truth = floor_scene(np.random.default_rng(4), 3, 1, noise=SIGMA)
    out, _ = D.estimate_floor_pose(dets, layout, TAGSIZE, *CAM, rotation=ROTATION, offset=OFFSET,
                                   heading=truth[2] + np.pi, heading_weight=WEIGHT)
    assert out["num_tags"] == 3 and np.isfinite([out["x"], out["y"], out["heading"]]).all()


@pytest.mark.parametrize("kw", [dict(heading=np.inf), dict(heading=-np.inf), dict(heading_weight=0.0),
                                dict(heading_weight=-1.0), dict(heading_weight=np.nan), dict(sigma=-0.1),
                                dict(sigma=np.inf), dict(sigma=np.nan), dict(distortion=(np.nan, 0, 0, 0, 0))])
def test_bad_arguments_are_rejected(D, kw):
    layout, dets, truth = floor_scene(np.random.default_rng(5), 2, 1)
    args = dict(rotation=ROTATION, offset=OFFSET, heading=truth[2], heading_weight=WEIGHT)
    args.update(kw)
    with pytest.raises(D.B200TagError):
        D.estimate_floor_pose(dets, layout, TAGSIZE, *CAM, **args)
    bad = layout.copy()
    bad["R"][0] *= 2
    with pytest.raises(D.B200TagError):
        D.estimate_floor_pose(dets, bad, TAGSIZE, *CAM, rotation=ROTATION, offset=OFFSET)


def test_sigma_without_an_output_is_rejected(D):
    import ctypes as C
    lib = D.load_library()
    out = np.zeros(1, dtype=D.FLOOR_POSE_DT)
    rc = lib.b200tag_estimate_floor_pose(None, 0, None, 0, TAGSIZE, *CAM, None, None, None, np.nan, np.inf, SIGMA,
                                         out.ctypes.data_as(C.c_void_p), None)
    assert rc == E_INVALID
    assert lib.b200tag_estimate_floor_pose(None, 0, None, 0, TAGSIZE, *CAM, None, None, None, np.nan, np.inf, 0.0,
                                           out.ctypes.data_as(C.c_void_p), None) == 0
