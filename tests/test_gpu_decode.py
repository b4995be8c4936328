"""The decode stage (k_decode / decode_family) at every orientation, with bit errors at every max_hamming, per-family
settings, reversed borders, tags cut by the frame edge and the decode options, against the brute-force reference and
the rendered truth (tests/decode_reference.py) and, stage by stage, against the CPU oracle.

Each case runs frame by frame (k_decode<4>, one to four frames) and again as one batch of all its frames (k_decode<1>,
five or more), at quad_decimate 1 and 2.  test_decode_reference_cpu.py runs the same scenes through the oracle."""
import pytest

import decode_reference as R
from parity import compare_all

pytestmark = pytest.mark.gpu

CASES = R.cases()


@pytest.fixture(scope="module")
def D():
    from ros_vision_b200 import detector
    detector.load_library()
    return detector


def _coverage(kind, scenes, tables, frames):
    """Truth checks over (detections, candidate quads) per frame; returns the coverage, or the edge counts."""
    cov, edge = R.Coverage(), (0, 0)
    for sc, (dets, quads, rotation_of) in zip(scenes, frames):
        if kind == "tags":
            R.check_tags(sc, quads, dets, tables, cov, rotation_of)
        else:
            n, n0 = R.check_edge_tags(sc, dets, 0)
            edge = (edge[0] + n, edge[1] + n0)
    return cov, edge


@pytest.mark.parametrize("dec", [1, 2])
@pytest.mark.parametrize("name", list(CASES))
def test_decode(D, oracle, name, dec):
    build, kind = CASES[name]
    scenes, families, tables, opts = build()
    assert len(scenes) >= 2
    orcs = [oracle.detect(oracle.make_config(R.W, R.H, "gray", dec, 0.0, families=families, **opts), sc.gray)
            for sc in scenes]
    # the oracle's own decode rotations (the engine's record does not carry them) and the case's coverage
    ref_cov, ref_edge = _coverage(kind, scenes, tables,
                                  [(o.detections, o.corners, lambda d: int(d["rotation"])) for o in orcs])
    R.check_coverage(name, ref_cov, ref_edge, dec)

    det = D.GpuDetector(R.W, R.H, "gray", quad_decimate=dec, keep_stages=True, families=families,
                        max_batch=max(5, len(scenes)), **opts)
    try:
        runs = {"frame by frame": [], "batch": []}
        for sc, orc in zip(scenes, orcs):
            det.Detect(sc.gray)
            runs["frame by frame"].append((compare_all(det, orc, 0, "gray"), det.FitQuads(0), None))
        frames = [sc.gray for sc in scenes]
        frames = (frames * 5)[:max(5, len(frames))]   # at least five frames: the one-warp kernel
        det.DetectBatch(frames)
        for f, orc in enumerate(orcs):
            runs["batch"].append((compare_all(det, orc, f, "gray"), det.FitQuads(f), None))
    finally:
        det.close()
    for how, res in runs.items():
        cov, edge = _coverage(kind, scenes, tables, res)
        assert (cov.decoded, cov.dropped, cov.ambiguous, cov.corrected) == \
               (ref_cov.decoded, ref_cov.dropped, ref_cov.ambiguous, ref_cov.corrected), how
        assert edge == ref_edge, how
