#!/usr/bin/env python3
"""Generates tests/golden/pose_host.npz: seeded detection records (tests/pose_records.py) with what the host pose
functions b200tag_estimate_poses and b200tag_locate_tags return for them.  tests/test_pose_golden.py holds the host
path to these values bit for bit.

The values were recorded before the pose arithmetic moved from csrc/pose.cc into csrc/pose_core.h, which the host and
the device kernel share.  Run it (CPU only) when the host pose functions change on purpose."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

from ros_vision_b200 import build, detector as D  # noqa: E402
import pose_records as PR  # noqa: E402

GOLDEN_POSE = os.path.join(HERE, "pose_host.npz")
COUNT, SEED = 1024, 20261020
ROTATION = PR.rot(0.3, -1.1, 0.7)
OFFSET = np.array([0.25, -0.1, 0.6])


def main():
    build.build_native()
    dets = PR.records(COUNT, SEED)
    poses = D.estimate_poses(dets, PR.TAGSIZE, PR.FX, PR.FY, PR.CX, PR.CY)
    # locate_tags sorts one list by distance: per 8 records, so that the sort and its ties are exercised too
    located = np.concatenate([D.locate_tags(dets[k:k + 8], PR.TAGSIZE, PR.FX, PR.FY, PR.CX, PR.CY, ROTATION, OFFSET)
                              for k in range(0, COUNT, 8)])
    np.savez_compressed(GOLDEN_POSE, dets=dets.view(np.uint8), poses=poses.view(np.uint8), located=located.view(np.uint8),
                        rotation=ROTATION, offset=OFFSET)
    print(GOLDEN_POSE, os.path.getsize(GOLDEN_POSE), "bytes")


if __name__ == "__main__":
    main()
