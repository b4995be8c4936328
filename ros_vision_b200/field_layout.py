"""Field layouts for the field pose step (GpuDetector.SetFieldLayout, detector.estimate_field_pose).

A layout is an array of detector.FIELD_TAG_DT records: the family index, the tag id, and the pose of the tag's frame in
the field, X_field = R X_tag + t.  The tag frame is b200tag_pose's: x to the right and y down as the tag is read, z into
the tag.
"""
from __future__ import annotations

import json

import numpy as np

from .detector import FIELD_TAG_DT

# Columns: this project's tag x, y, z axes in WPILib's tag frame, where +X points out of the tag face and +Z up, so that
# +Y is the right-hand side of a viewer facing the tag.
WPILIB_FROM_TAG = np.array([[0.0, 0.0, -1.0], [1.0, 0.0, 0.0], [0.0, -1.0, 0.0]])


def quaternion_matrix(w: float, x: float, y: float, z: float) -> np.ndarray:
    """The rotation of the unit quaternion (w, x, y, z); the quaternion is normalised first."""
    n = np.sqrt(w * w + x * x + y * y + z * z)
    w, x, y, z = w / n, x / n, y / n, z / n
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def from_wpilib(json_path_or_dict, family: int = 0) -> np.ndarray:
    """FIELD_TAG_DT records of a WPILib AprilTagFieldLayout JSON (a path or the parsed dict):
    {"tags": [{"ID", "pose": {"translation": {x, y, z}, "rotation": {"quaternion": {W, X, Y, Z}}}}], "field": {...}}.
    Every tag gets the detector family index `family`."""
    if isinstance(json_path_or_dict, dict):
        doc = json_path_or_dict
    else:
        with open(json_path_or_dict) as f:
            doc = json.load(f)
    tags = doc["tags"]
    out = np.zeros(len(tags), dtype=FIELD_TAG_DT)
    for i, tag in enumerate(tags):
        tr, q = tag["pose"]["translation"], tag["pose"]["rotation"]["quaternion"]
        out["family"][i] = family
        out["id"][i] = int(tag["ID"])
        out["R"][i] = quaternion_matrix(q["W"], q["X"], q["Y"], q["Z"]) @ WPILIB_FROM_TAG
        out["t"][i] = (tr["x"], tr["y"], tr["z"])
    return out
