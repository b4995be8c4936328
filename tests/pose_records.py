"""Seeded synthetic detection records for the pose step, built like tests/test_pose.py::_detection (a tag projected
with a known pose, its homography from a DLT through the four corners).  Four kinds take turns so that every branch
of b200tag_estimate_pose is exercised: noisy corners, far near-frontal tags (the two local minima are close), near
edge-on tags, and collapsed quads whose I - mean(F) cannot be inverted (error HUGE_VAL)."""
import numpy as np

FX, FY, CX, CY = 905.5, 907.9, 640.0, 400.0
TAGSIZE = 0.1651


def rot(rx, ry, rz):
    cx, sx, cy, sy, cz, sz = np.cos(rx), np.sin(rx), np.cos(ry), np.sin(ry), np.cos(rz), np.sin(rz)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return Rz @ Ry @ Rx


def homography(src, dst):
    """DLT through 4 correspondences, H[2][2] = 1 (what quad_update_homographies produces)."""
    A, b = [], []
    for (x, y), (u, v) in zip(src, dst):
        A.append([x, y, 1, 0, 0, 0, -x * u, -y * u]); b.append(u)
        A.append([0, 0, 0, x, y, 1, -x * v, -y * v]); b.append(v)
    h = np.linalg.solve(np.array(A, dtype=np.float64), np.array(b, dtype=np.float64))
    return np.append(h, 1.0)


def records(n, seed):
    """`n` DETECTION_DT records; record i is of kind i % 4 (noisy, far near-frontal, near edge-on, collapsed)."""
    from ros_vision_b200 import detector as D
    rng = np.random.default_rng(seed)
    s = TAGSIZE / 2
    P = np.array([[-s, s, 0], [s, s, 0], [s, -s, 0], [-s, -s, 0]], dtype=np.float64)
    out = np.zeros(n, dtype=D.DETECTION_DT)
    for i in range(n):
        kind = i % 4
        if kind == 1:
            R = rot(np.pi + rng.uniform(-0.05, 0.05), rng.uniform(-0.05, 0.05), rng.uniform(-np.pi, np.pi))
            t = np.array([rng.uniform(-0.5, 0.5), rng.uniform(-0.3, 0.3), rng.uniform(4.0, 8.0)])
            noise = rng.normal(0, 0.3, size=(4, 2))
        elif kind == 2:
            tilt = rng.choice([-1, 1]) * rng.uniform(1.3, 1.5)
            R = rot(np.pi + tilt, rng.uniform(-0.2, 0.2), rng.uniform(-np.pi, np.pi))
            t = np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2), rng.uniform(0.5, 2.0)])
            noise = rng.normal(0, 0.1, size=(4, 2))
        else:
            R = rot(np.pi + rng.uniform(-0.6, 0.6), rng.uniform(-0.6, 0.6), rng.uniform(-np.pi, np.pi))
            t = np.array([rng.uniform(-0.8, 0.8), rng.uniform(-0.5, 0.5), rng.uniform(0.5, 4.0)])
            noise = rng.normal(0, 0.3, size=(4, 2))
        cam = (R @ P.T).T + t
        px = np.stack([FX * cam[:, 0] / cam[:, 2] + CX, FY * cam[:, 1] / cam[:, 2] + CY], axis=1) + noise
        out["H"][i] = homography([(-1, 1), (1, 1), (1, -1), (-1, -1)], px)
        if kind == 3:  # every corner on one ray: I - mean(F) is singular, exactly so on the optical axis
            px[:] = (CX, CY) if i % 8 == 7 else px[0]
        out["p"][i] = px
        out["c"][i] = px.mean(axis=0)
        out["id"][i] = i % 587
        out["frame"][i] = i
    return out
