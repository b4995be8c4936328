#!/usr/bin/env python3
"""Generates tests/golden/reference_stages.npz: the stages tests/test_gpu_reference_live.py compares with upstream
apriltags_cuda's GpuDetector, on that test's seven frames, recorded from the CPU oracle.

The oracle was last run beside upstream's GpuDetector (oracle/_ref/librefgpu.so) at commit ae21773, and every
stage agreed there: bit-exact for the images, the component partition and sizes, the boundary points, the extents and
selection, the angle-sorted points, the prefix moments and the FitQuads, within the test's tolerances for the line-fit
errors, QuadCorners and refined quads.  Neither the oracle nor these frames have changed since, so these are the
values upstream produced, up to those tolerances.  Run it (CPU only) when the oracle changes on purpose, and only
after test_gpu_reference_live has passed against the live upstream library.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

from oracle import pyoracle  # noqa: E402
from helpers import reference_stage_record  # noqa: E402
from test_gpu_reference_live import GOLDEN_STAGES, _frames  # noqa: E402


def main():
    pyoracle.build()
    out = {}
    names = []
    for k, (name, yuyv, w, h, cam, dist) in enumerate(_frames()):
        orc = pyoracle.detect(pyoracle.make_config(w, h, "yuyv", 2, 0.0, camera=cam, dist=dist), yuyv)
        for key, v in reference_stage_record(orc).items():
            out[f"{k}_{key}"] = np.asarray(v)
        names.append(name)
    out["names"] = np.array(names)
    np.savez_compressed(GOLDEN_STAGES, **out)
    print(GOLDEN_STAGES, os.path.getsize(GOLDEN_STAGES), "bytes")


if __name__ == "__main__":
    main()
