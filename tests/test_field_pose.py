"""The field pose (b200tag_estimate_field_pose, detector.estimate_field_pose) on the host: against ground truth, against
OpenCV's least-squares PnP on the same correspondences, the robot-frame formula, which detections take part, the WPILib
layout loader and argument checks.  Pure host code: runs without a GPU."""
import ctypes as C

import numpy as np
import pytest

import pose_records as PR

TAGSIZE = PR.TAGSIZE
CAM = (PR.FX, PR.FY, PR.CX, PR.CY)
K = np.array([[PR.FX, 0, PR.CX], [0, PR.FY, PR.CY], [0, 0, 1]])
ROTATION = np.array([[0.0, 0, 1], [-1, 0, 0], [0, -1, 0]])  # camera looking along the robot's +x
OFFSET = np.array([0.25, -0.1, 0.6])
E_INVALID = -1


@pytest.fixture(scope="module")
def D():
    from ros_vision_b200 import build, detector
    build.build_native()
    detector.load_library()
    return detector


def tag_points(tagsize=TAGSIZE):
    s = tagsize / 2
    return np.array([[-s, s, 0], [s, s, 0], [s, -s, 0], [-s, -s, 0]], dtype=np.float64)


def project(cam_pts):
    return np.stack([PR.FX * cam_pts[:, 0] / cam_pts[:, 2] + PR.CX, PR.FY * cam_pts[:, 1] / cam_pts[:, 2] + PR.CY], axis=1)


def random_rotation(rng):
    q = rng.normal(size=4)
    from ros_vision_b200.field_layout import quaternion_matrix
    return quaternion_matrix(*q)


def scene(rng, ntags, planes, noise=0.0, zmin=1.0, zmax=6.0):
    """A random camera in the field and `ntags` layout tags in front of it on `planes` planes (1 = all coplanar).
    Returns (layout, detections, camera-from-field R, t)."""
    from ros_vision_b200 import detector as D
    Rcf, tcf = random_rotation(rng), rng.uniform(-5, 5, size=3)  # X_cam = Rcf X_field + tcf
    layout = np.zeros(ntags, dtype=D.FIELD_TAG_DT)
    dets = np.zeros(ntags, dtype=D.DETECTION_DT)
    ids = rng.choice(587, size=ntags, replace=False)
    plane_R = [PR.rot(*rng.uniform(-0.6, 0.6, size=3)) for _ in range(planes)]
    plane_t = [np.array([rng.uniform(-0.4, 0.4), rng.uniform(-0.3, 0.3), 1.0]) * rng.uniform(zmin + 0.5, zmax - 0.5)
               for _ in range(planes)]
    P = tag_points()
    for j in range(ntags):
        k = j % planes
        for _ in range(1000):  # a spot on plane k whose corners all lie in front of the camera, zmin..zmax away
            t = plane_t[k] + plane_R[k] @ np.array([rng.uniform(-1.5, 1.5), rng.uniform(-1.0, 1.0), 0.0])
            cam = P @ plane_R[k].T + t
            px = project(cam) if (cam[:, 2] > zmin).all() and (cam[:, 2] < zmax).all() else None
            if px is not None and (px >= 0).all() and (px[:, 0] < 1280).all() and (px[:, 1] < 800).all():
                break
        layout["id"][j] = ids[j]
        layout["R"][j] = Rcf.T @ plane_R[k]
        layout["t"][j] = Rcf.T @ (t - tcf)
        dets["id"][j] = ids[j]
        dets["decision_margin"][j] = 100.0
        dets["p"][j] = px + (rng.normal(0, noise, size=(4, 2)) if noise else 0)
        dets["c"][j] = dets["p"][j].mean(axis=0)
    return layout, dets, Rcf, tcf


def field_points(layout):
    P = tag_points()
    return np.concatenate([P @ np.asarray(L["R"]).T + L["t"] for L in layout])


def cost(obj, img, R, t):
    return float(((project(obj @ R.T + t) - img) ** 2).sum())


def ours_cf(out):
    """Our result as camera-from-field (R, t)."""
    R = out["camera_R"].T
    return R, -R @ out["camera_t"]


@pytest.mark.parametrize("planes", [1, 2, 3])
def test_noise_free_scenes_return_the_truth(D, planes):
    rng = np.random.default_rng(10 + planes)
    for trial in range(40):
        layout, dets, Rcf, tcf = scene(rng, int(rng.integers(max(2, planes), 9)), planes)
        out = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM)
        assert out["num_tags"] == len(layout)
        R, t = ours_cf(out)
        assert np.abs(R - Rcf).max() <= 1e-9 and np.abs(t - tcf).max() <= 1e-9, trial
        assert out["rms"] < 1e-9 and out["rms_other"] == np.inf
        assert 1 <= out["iterations"] <= 20


def test_noisy_scenes_reach_opencvs_minimum(D):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(77)
    crit = (cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_COUNT, 200, 1e-15)
    for trial in range(60):
        planes = 1 + trial % 3
        layout, dets, Rcf, tcf = scene(rng, int(rng.integers(2, 9)), planes, noise=0.3)
        obj, img = field_points(layout), dets["p"].reshape(-1, 2).copy()
        ok, rvec, tvec = cv2.solvePnP(obj, img, K, None, flags=cv2.SOLVEPNP_SQPNP)
        assert ok
        rvec, tvec = cv2.solvePnPRefineLM(obj, img, K, None, rvec, tvec, crit)
        Rcv, tcv = cv2.Rodrigues(rvec)[0], tvec.reshape(3)
        out = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM)
        R, t = ours_cf(out)
        c_ours, c_cv = cost(obj, img, R, t), cost(obj, img, Rcv, tcv)
        assert c_ours <= c_cv * (1 + 1e-9), trial
        assert np.abs(R - Rcv).max() <= 1e-6, trial
        assert np.abs(t - tcv).max() <= 1e-6 * np.linalg.norm(tcv), trial
        assert abs(out["rms"] - np.sqrt(c_ours / obj.shape[0])) <= 1e-9 * out["rms"]


def test_single_tag_returns_both_refined_ippe_branches(D):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(5)
    crit = (cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_COUNT, 200, 1e-15)
    same_other = 0
    for trial in range(60):
        layout, dets, Rcf, tcf = scene(rng, 1, 1, noise=0.3, zmin=1.0, zmax=4.0)
        P, img = tag_points(), dets["p"][0].copy()
        n, rvecs, tvecs, _ = cv2.solvePnPGeneric(P, img, K, None, flags=cv2.SOLVEPNP_IPPE_SQUARE)
        assert n == 2
        Rl, tl = np.asarray(layout["R"][0]), np.asarray(layout["t"][0])
        sols = []
        for rv, tv in zip(rvecs, tvecs):
            rv, tv = cv2.solvePnPRefineLM(P, img, K, None, rv.copy(), tv.copy(), crit)
            Rct, tct = cv2.Rodrigues(rv)[0], tv.reshape(3)
            Rf = Rct @ Rl.T
            sols.append((Rf, tct - Rf @ tl, np.sqrt(cost(P, img, Rct, tct) / 4)))
        out = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM)
        R, t = ours_cf(out)
        match = [i for i, (Rs, ts, _) in enumerate(sols) if np.abs(R - Rs).max() <= 1e-6 and np.abs(t - ts).max() <= 1e-6 * np.linalg.norm(ts)]
        assert match, trial
        i = match[0]
        assert abs(out["rms"] - sols[i][2]) <= 1e-6 * sols[i][2] + 1e-12
        assert out["rms"] <= sols[1 - i][2] * (1 + 1e-9) and out["rms"] <= out["rms_other"]
        # where the other branch has no minimum of its own it slides slowly towards the first one, and the two
        # refinements (ours capped at 20 iterations) stop at different points of that slope
        same_other += abs(out["rms_other"] - sols[1 - i][2]) <= 1e-6 * sols[1 - i][2] + 1e-12
    assert same_other >= 54


def test_robot_pose_is_the_extrinsic_formula(D):
    rng = np.random.default_rng(3)
    for _ in range(20):
        layout, dets, _, _ = scene(rng, 3, 2, noise=0.3)
        rot, off = random_rotation(rng), rng.uniform(-1, 1, size=3)
        out = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM, rotation=rot, offset=off)
        robot_R = out["camera_R"] @ rot.T
        assert np.abs(out["robot_R"] - robot_R).max() <= 1e-12
        assert np.abs(out["robot_t"] - (out["camera_t"] - robot_R @ off)).max() <= 1e-12
        plain = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM)
        assert plain["camera_R"].tobytes() == out["camera_R"].tobytes()
        assert plain["robot_R"].tobytes() == plain["camera_R"].tobytes()
        assert plain["robot_t"].tobytes() == plain["camera_t"].tobytes()


def with_duplicates(rng, dets):
    """`dets` plus, per record, an overlapping duplicate (corners moved by up to 0.5 px) and a distant one (300 px away),
    with hamming and decision margin drawn so that either may win; some duplicates tie on both and differ in corners."""
    extra = []
    for d in dets:
        for shift in (rng.uniform(-0.5, 0.5, size=(4, 2)), np.array([300.0, 0.0])):
            e = d.copy()
            e["p"] = d["p"] + shift
            e["c"] = e["p"].mean(axis=0)
            if rng.random() < 0.3:
                e["hamming"], e["decision_margin"] = d["hamming"], d["decision_margin"]
            else:
                e["hamming"] = rng.integers(0, 3)
                e["decision_margin"] = rng.uniform(50, 150)
            extra.append(e)
    out = np.concatenate([dets, np.array(extra, dtype=dets.dtype)])
    return out[rng.permutation(len(out))]


def reconciled(D, raw):
    v = raw.copy()
    n = D.load_library().b200tag_debug_reconcile(v.ctypes.data_as(C.c_void_p), len(v))
    return v[:n]


def test_raw_list_gives_the_reconciled_lists_pose(D):
    rng = np.random.default_rng(8)
    for trial in range(40):
        layout, dets, _, _ = scene(rng, int(rng.integers(1, 6)), 2 if trial % 2 else 1, noise=0.3)
        raw = with_duplicates(rng, dets)
        a = D.estimate_field_pose(raw, layout, TAGSIZE, *CAM, rotation=ROTATION, offset=OFFSET)
        b = D.estimate_field_pose(reconciled(D, raw), layout, TAGSIZE, *CAM, rotation=ROTATION, offset=OFFSET)
        assert a.tobytes() == b.tobytes(), trial
        assert a["num_tags"] == len(layout)


def test_other_detections_are_ignored(D):
    rng = np.random.default_rng(9)
    layout, dets, _, _ = scene(rng, 4, 2, noise=0.3)
    base = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM)
    assert base["num_tags"] == 4
    others = dets.copy()
    others["id"] = [i for i in range(587) if i not in set(layout["id"])][:4]  # ids outside the layout
    fam = dets.copy()
    fam["family"] = 1  # another family
    hidden = layout.copy()[:2]
    hidden["id"] = others["id"][:2] + 1000  # layout tags not otherwise in view, seen only as collapsed quads
    collapsed = dets[:2].copy()
    collapsed["id"] = hidden["id"]
    collapsed["p"] = collapsed["p"][:, :1, :]
    lay2 = np.concatenate([layout, hidden])
    got = D.estimate_field_pose(np.concatenate([others, fam, dets, collapsed]), lay2, TAGSIZE, *CAM)
    assert got.tobytes() == base.tobytes()
    none = D.estimate_field_pose(np.concatenate([others, fam, collapsed]), lay2, TAGSIZE, *CAM)
    assert none["num_tags"] == 0 and none["iterations"] == 0
    assert none["camera_R"].tobytes() == np.eye(3).tobytes() and not none["camera_t"].any()
    assert none["robot_R"].tobytes() == np.eye(3).tobytes() and not none["robot_t"].any()
    assert none["rms"] == np.inf and none["rms_other"] == np.inf
    assert D.estimate_field_pose(dets[:0], layout, TAGSIZE, *CAM).tobytes() == none.tobytes()
    assert D.estimate_field_pose(dets, layout[:0], TAGSIZE, *CAM).tobytes() == none.tobytes()


def wpilib_case(D, tag_xyz, tag_yaw, distance):
    """A tag on the field wall at tag_xyz, turned by tag_yaw about +Z (WPILib quaternion), and a robot `distance` m in
    front of it facing it, camera on the robot's front (ROTATION, offset 0).  Returns the tag's IPPE pose and the
    field pose, and the robot's true (x, y, yaw)."""
    from ros_vision_b200 import field_layout
    doc = {"tags": [{"ID": 7, "pose": {"translation": {"x": tag_xyz[0], "y": tag_xyz[1], "z": tag_xyz[2]},
                                        "rotation": {"quaternion": {"W": np.cos(tag_yaw / 2), "X": 0.0, "Y": 0.0,
                                                                    "Z": np.sin(tag_yaw / 2)}}}}],
           "field": {"length": 16.54, "width": 8.21}}
    layout = field_layout.from_wpilib(doc)
    assert layout["id"][0] == 7 and layout["family"][0] == 0
    normal = np.array([np.cos(tag_yaw), np.sin(tag_yaw), 0.0])  # WPILib +X: out of the tag face
    robot_xy = np.array(tag_xyz[:2]) + distance * normal[:2]
    yaw = tag_yaw + np.pi
    robot_R = np.array([[np.cos(yaw), -np.sin(yaw), 0], [np.sin(yaw), np.cos(yaw), 0], [0, 0, 1]])
    camera_R, camera_t = robot_R @ ROTATION, np.array([robot_xy[0], robot_xy[1], tag_xyz[2]])
    X = tag_points() @ np.asarray(layout["R"][0]).T + layout["t"][0]
    dets = np.zeros(1, dtype=D.DETECTION_DT)
    dets["id"] = 7
    dets["p"][0] = project((X - camera_t) @ camera_R)
    tag_pose = D.estimate_poses(dets, TAGSIZE, *CAM, method="ippe")[0]
    out = D.estimate_field_pose(dets, layout, TAGSIZE, *CAM, rotation=ROTATION, offset=np.zeros(3))
    return tag_pose, out, (robot_xy[0], robot_xy[1], yaw)


def test_wpilib_layout_head_on(D):
    tag_pose, out, (x, y, yaw) = wpilib_case(D, (0.0, 0.0, 0.5), 0.0, 3.0)
    # IPPE's out-of-plane terms are square roots of 1 - r^2, so a tag seen exactly head-on comes back within ~1e-7
    assert np.abs(tag_pose["R"] - np.eye(3)).max() <= 1e-6
    assert np.abs(tag_pose["t"] - [0, 0, 3]).max() <= 1e-9
    assert abs(out["robot_t"][0] - 3) <= 1e-9 and abs(out["robot_t"][1]) <= 1e-9
    got_yaw = np.arctan2(out["robot_R"][1, 0], out["robot_R"][0, 0])
    assert abs(np.angle(np.exp(1j * (got_yaw - np.pi)))) <= 1e-9


def test_wpilib_layout_yawed_tag(D):
    tag_pose, out, (x, y, yaw) = wpilib_case(D, (4.0, 2.5, 1.2), np.radians(-120.0), 2.0)
    # IPPE's out-of-plane terms are square roots of 1 - r^2, so a tag seen exactly head-on comes back within ~1e-7
    assert np.abs(tag_pose["R"] - np.eye(3)).max() <= 1e-6
    assert np.abs(tag_pose["t"] - [0, 0, 2]).max() <= 1e-9
    assert abs(out["robot_t"][0] - x) <= 1e-9 and abs(out["robot_t"][1] - y) <= 1e-9
    assert abs(out["robot_t"][2] - 1.2) <= 1e-6  # the head-on tilt above, 2 m away
    got_yaw = np.arctan2(out["robot_R"][1, 0], out["robot_R"][0, 0])
    assert abs(np.angle(np.exp(1j * (got_yaw - yaw)))) <= 1e-9


def test_invalid_arguments_are_rejected(D):
    lib = D.load_library()
    rng = np.random.default_rng(1)
    layout, dets, _, _ = scene(rng, 3, 1)
    out = np.zeros(1, dtype=D.FIELD_POSE_DT)

    def call(dets=dets, n=None, layout=layout, nl=None, tagsize=TAGSIZE, fx=PR.FX, fy=PR.FY, out=out):
        lay = None if layout is None else np.ascontiguousarray(layout)
        return lib.b200tag_estimate_field_pose(None if dets is None else dets.ctypes.data_as(C.c_void_p),
                                               len(dets) if n is None else n,
                                               None if lay is None else lay.ctypes.data_as(C.c_void_p),
                                               (0 if lay is None else len(lay)) if nl is None else nl,
                                               tagsize, fx, fy, PR.CX, PR.CY, None, None,
                                               None if out is None else out.ctypes.data_as(C.c_void_p))

    assert call() == 0
    assert call(layout=None, nl=3) == E_INVALID
    assert call(nl=-1) == E_INVALID
    assert call(dets=None, n=2) == E_INVALID
    assert call(n=-1) == E_INVALID
    assert call(out=None) == E_INVALID
    assert call(tagsize=0.0) == E_INVALID and call(tagsize=-1.0) == E_INVALID
    assert call(fx=0.0) == E_INVALID and call(fy=0.0) == E_INVALID
    big = np.zeros(1025, dtype=D.FIELD_TAG_DT)
    big["id"] = np.arange(1025)
    big["R"] = np.eye(3)
    assert call(layout=big) == E_INVALID and call(layout=big[:1024]) == 0
    dup = layout.copy()
    dup["id"][2] = dup["id"][0]
    assert call(layout=dup) == E_INVALID
    dup["family"][2] = 1  # the same id in another family is another tag
    assert call(layout=dup) == 0
    for k, v in [("R", 1 + 2e-6), ("R", 0.5)]:
        bad = layout.copy()
        bad["R"][1] = bad["R"][1] * v
        assert call(layout=bad) == E_INVALID
    near = layout.copy()
    near["R"][1] = near["R"][1] * (1 + 1e-7)
    assert call(layout=near) == 0
    mirror = layout.copy()
    mirror["R"][0] = -mirror["R"][0]  # orthonormal, but a reflection
    assert call(layout=mirror) == E_INVALID
    for field, idx in [("R", (1, 0, 0)), ("t", (2, 1))]:
        for v in (np.nan, np.inf):
            bad = layout.copy()
            bad[field][idx] = v
            assert call(layout=bad) == E_INVALID
    with pytest.raises(D.B200TagError):
        D.estimate_field_pose(dets, dup[[0, 0]], TAGSIZE, *CAM)
    assert (out["num_tags"] == 3)  # the last successful call's result, untouched by the rejected ones
