"""The host pose functions against tests/golden/pose_host.npz, bit for bit: b200tag_estimate_poses and
b200tag_locate_tags on seeded records (tests/pose_records.py) return exactly what they returned before the pose
arithmetic moved into csrc/pose_core.h, which the device kernel shares.  Pure host code: runs without a GPU."""
import os

import numpy as np
import pytest

import pose_records as PR

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pose_host.npz")


@pytest.fixture(scope="module")
def golden():
    from ros_vision_b200 import build, detector as D
    build.build_native()
    D.load_library()
    z = np.load(GOLDEN)
    return D, z["dets"].view(D.DETECTION_DT), z["poses"].view(D.POSE_DT), z["located"].view(D.TAG_POSITION_DT), z["rotation"], z["offset"]


def test_records_are_reproducible(golden):
    """The generator still makes the stored records, so the device tests that draw more of them draw the same kinds."""
    D, dets, *_ = golden
    assert PR.records(len(dets), 20261020).tobytes() == dets.tobytes()


def test_estimate_poses_bit_identical(golden):
    D, dets, poses, *_ = golden
    got = D.estimate_poses(dets, PR.TAGSIZE, PR.FX, PR.FY, PR.CX, PR.CY)
    rows = lambda a: a.view(np.uint8).reshape(len(a), -1)  # noqa: E731
    bad = np.flatnonzero(np.any(rows(got) != rows(poses), axis=1))
    assert bad.size == 0, f"{bad.size} poses differ, first at record {bad[:5]}"
    assert np.isinf(poses["err"]).sum() > 0 and np.isfinite(poses["err_other"]).sum() > len(poses) // 2


def test_locate_tags_bit_identical(golden):
    D, dets, _, located, rotation, offset = golden
    got = np.concatenate([D.locate_tags(dets[k:k + 8], PR.TAGSIZE, PR.FX, PR.FY, PR.CX, PR.CY, rotation, offset)
                          for k in range(0, len(dets), 8)])
    assert got.tobytes() == located.tobytes()
