"""The stages of upstream apriltags_cuda's own GpuDetector pin the CPU oracle and the product.

This is what pins the oracle's front end: every stage upstream exposes through its debug accessors
(apriltag_gpu.h:97-183) is compared with the oracle's restatement on identical YUYV frames -- images and integer
stages bit-exact, component labels up to relabelling, float stages exact or within the stated tolerance (the upstream
build contracts some expressions into FMAs).  The quads upstream hands to quad_decode_index (after its own
RefineEdges) pin the refine stage; decode itself is libapriltag, absent from upstream's tree, and stays unpinned.

Upstream's stages on these frames are stored in tests/golden/reference_stages.npz (digests of the integer stages,
a sample of the line-fit errors, the quad corners in full; see tests/golden/make_reference_stages.py), so the
comparison runs from the repository alone.  When upstream's GpuDetector has been built into
oracle/_ref/librefgpu.so (oracle/build_ref.sh), it also runs live on the same frames and is compared in full.

(A frame without any boundary point cannot be part of this test: upstream hands CUB zero items and aborts in its
CHECK_CUDA at apriltag_gpu.cu:788-802 -- observed on a flat 640x480 frame.  The product and the oracle handle that
case; see test_gpu_parity.py::test_edge_cases.)
"""
import os

import numpy as np
import pytest

from helpers import GOLDEN, canonical_partition, load_golden, match_corner_sets, reference_stage_record

pytestmark = pytest.mark.gpu

GOLDEN_STAGES = os.path.join(GOLDEN, "reference_stages.npz")
CAM = (905.495617, 609.916016, 907.909470, 352.682645)   # gpu_detector_test.cu:63-73
DIST = (0.059238, -0.075154, -0.003801, 0.001113, 0.0)
ERR_REL_TOL = 1e-5        # line-fit errors: f32 expressions, FMA contraction in the upstream build
CORNER_EXACT_TOL = 2e-3   # QuadCorners (float, host code both sides)
REFINE_TOL_PX = 0.05      # north-star corner bar


def _key64(a, b):
    a = np.asarray(a, dtype=np.uint64)
    b = np.asarray(b, dtype=np.uint64)
    return (np.minimum(a, b) << np.uint64(32)) | np.maximum(a, b)


def _frames():
    from ros_vision_b200 import synth
    out = []
    for idx in (0, 1, 7):
        frame, fmt, w, h, dec, sigma, sc = synth.config_frame(2, idx)
        out.append((f"config2[{idx}]", frame, w, h, None, None))
    for name in ("ref_colorimage_crop", "ref_grayimage_crop", "ref_colorimage_notags_crop"):
        meta, img = load_golden(name)
        out.append((name, synth.gray_to_yuyv(img), meta["width"], meta["height"], CAM, DIST))
    sc = synth.make_scene(640, 480, 77, 3, side_range=(50, 140), noise_sigma=2.0)
    out.append(("synthetic640", synth.gray_to_yuyv(sc.gray), 640, 480, None, None))
    return out


def _compare_reference_with_oracle(ref, orc, report):
    """Returns {oracle blob-pair key: reference cluster index} after checking every exposed stage."""
    assert np.array_equal(ref.gray(), orc.gray), "gray"
    assert np.array_equal(ref.decimated(), orc.quad_im), "decimated"
    thresh = ref.thresholded()
    assert np.array_equal(thresh, orc.thresh), "thresholded image (bit-exact)"

    # component labels up to relabelling: the label pairs must form a bijection
    mask = thresh.reshape(-1) != 127
    rl, ol = ref.labels(), orc.labels
    pairs = np.unique(np.stack([rl[mask].astype(np.int64), ol[mask].astype(np.int64)], axis=1), axis=0)
    assert len(pairs) == len(np.unique(rl[mask])) == len(np.unique(ol[mask])), "component partition"
    lut = np.zeros(rl.size, dtype=np.uint32)   # reference label -> oracle label
    lut[pairs[:, 0]] = pairs[:, 1].astype(np.uint32)
    rs = ref.sizes()
    assert np.array_equal(rs[rl[mask]], orc.sizes[ol[mask]]), "component sizes"

    # boundary points: same set, and the same order inside a blob pair
    rp = ref.sorted_points()
    assert len(rp) == len(orc.points), ("number of boundary points", len(rp), len(orc.points))
    rkey = _key64(lut[rp["rep0"]], lut[rp["rep1"]])
    okey = _key64(orc.points["rep0"], orc.points["rep1"])
    order = np.argsort(rkey, kind="stable")
    for fld_r, fld_o in (("x", "x"), ("y", "y"), ("dir", "dir"), ("b2w", "b2w")):
        assert np.array_equal(rp[fld_r][order], orc.points[fld_o]), f"boundary points .{fld_o} (order within blob pair)"
    assert np.array_equal(rkey[order], okey)

    # extents per blob pair
    ext = ref.extents()
    assert len(ext) == len(orc.clusters), "number of blob pairs"
    ekey = rkey[ext["start"]]
    eorder = np.argsort(ekey, kind="stable")
    assert np.array_equal(ekey[eorder], _key64(orc.clusters["rep0"], orc.clusters["rep1"]))
    for fld in ("min_x", "min_y", "max_x", "max_y", "count", "gx_sum", "gy_sum", "pxgx_plus_pygy_sum"):
        assert np.array_equal(ext[fld][eorder].astype(np.int64), orc.clusters[fld].astype(np.int64)), f"extents.{fld}"
    sel = ref.selected_extents()
    assert np.array_equal(sel["count"][eorder] > 0, orc.clusters["selected"] != 0), "SelectBlobs"

    # angle-sorted points, prefix moments, errors per selected blob
    sp = ref.sorted_selected()
    lfp = ref.line_fit_points()
    errs, filt = ref.errors()
    assert len(sp) == len(orc.spoints), "number of selected points"
    worst_err = 0.0
    exact_err = True
    for ci_ref, oc in zip(eorder, orc.clusters):
        if not oc["selected"]:
            continue
        cnt = int(oc["count"])
        r0, o0 = int(sel["start"][ci_ref]), int(oc["sel_start"])
        assert int(sel["count"][ci_ref]) == cnt
        rs_, os_ = sp[r0:r0 + cnt], orc.spoints[o0:o0 + cnt]
        assert np.all(rs_["blob"] == ci_ref)
        for fld in ("theta", "x", "y", "dir"):
            assert np.array_equal(rs_[fld], os_[fld]), f"angle-sorted points .{fld}"
        for fld in ("Mxx", "Myy", "Mxy", "Mx", "My", "W"):
            assert np.array_equal(lfp[fld][r0:r0 + cnt], orc.lfps[fld][o0:o0 + cnt]), f"prefix moment {fld}"
        for got, exp in ((errs[r0:r0 + cnt], orc.errs[o0:o0 + cnt]), (filt[r0:r0 + cnt], orc.filtered_errs[o0:o0 + cnt])):
            scale = max(1.0, float(np.abs(exp).max()))
            d = float(np.abs(got - exp).max()) / scale
            worst_err = max(worst_err, d)
            exact_err &= bool(np.array_equal(got, exp))
    assert worst_err <= ERR_REL_TOL, ("line-fit errors", worst_err)
    report["line_fit_errors_bit_exact"] = exact_err
    report["line_fit_errors_max_rel"] = worst_err

    # fit quads
    fq = ref.fit_quads()
    key_of_ref_cluster = ekey  # indexed by reference cluster index
    okeys = _key64(orc.fitquads["rep0"], orc.fitquads["rep1"])
    lut_fq = {int(k): i for i, k in enumerate(okeys)}
    assert len(fq) == len(orc.fitquads), "number of FitQuads"
    for q in fq:
        o = orc.fitquads[lut_fq[int(key_of_ref_cluster[int(q["blob"])])]]
        assert bool(q["valid"]) == bool(o["valid"]), "FitQuad.valid"
        if q["valid"]:
            assert np.array_equal(q["indices"], o["indices"]), "FitQuad.indices"
            for fld in ("Mx", "My", "W", "Mxx", "Myy", "Mxy", "N"):
                assert np.array_equal(q["moments"][fld], o["moments"][fld]), f"FitQuad.moments.{fld}"

    # quad corners and refined quads
    qc, rq = ref.quad_corners(), ref.refined_quads()
    assert len(qc) == len(orc.corners) == len(rq) == len(orc.refined), "number of QuadCorners"
    ockeys = _key64(orc.corners["rep0"], orc.corners["rep1"])
    lut_qc = {int(k): i for i, k in enumerate(ockeys)}
    worst_c = worst_r = 0.0
    for q, r in zip(qc, rq):
        i = lut_qc[int(key_of_ref_cluster[int(q["blob"])])]
        worst_c = max(worst_c, float(np.abs(q["corners"] - orc.corners["corners"][i]).max()))
        worst_r = max(worst_r, float(np.abs(r["corners"] - orc.refined["corners"][i]).max()))
        assert int(q["reversed_border"]) == int(orc.corners["reversed_border"][i])
    assert worst_c <= CORNER_EXACT_TOL, ("QuadCorners", worst_c)
    assert worst_r <= REFINE_TOL_PX, ("refined quads", worst_r)
    report["quad_corners_max_abs_px"] = worst_c
    report["refined_quads_max_abs_px"] = worst_r
    return rq


def _compare_oracle_with_stored(orc, g, name):
    """The oracle against upstream's stored stages: digests equal, line-fit errors and corners within tolerance."""
    rec = reference_stage_record(orc)
    for key, v in rec.items():
        if key.startswith(("digest_", "num_")):
            assert str(v) == str(g[key]), (name, key)
    assert np.array_equal(rec["err_index"], g["err_index"]), (name, "line-fit error sample")
    for fld, scale in (("err", g["err_absmax"][0]), ("filtered_err", g["err_absmax"][1])):
        d = float(np.abs(rec[fld] - g[fld]).max(initial=0.0)) / max(1.0, float(scale))
        assert d <= ERR_REL_TOL, (name, "line-fit errors", fld, d)
    assert np.array_equal(rec["corner_blob"], g["corner_blob"]), (name, "QuadCorners blobs")
    assert np.array_equal(rec["reversed_border"], g["reversed_border"]), (name, "QuadCorners.reversed_border")
    assert float(np.abs(rec["corners"] - g["corners"]).max(initial=0.0)) <= CORNER_EXACT_TOL, (name, "QuadCorners")
    assert float(np.abs(rec["refined"] - g["refined"]).max(initial=0.0)) <= REFINE_TOL_PX, (name, "refined quads")


def _compare_product(det, thresholded, labels, corners, refined, what):
    """The product against upstream's thresholded image, component partition, QuadCorners and refined quads."""
    assert np.array_equal(det.CopyThresholdedTo(), thresholded), f"product vs {what}: thresholded"
    mask = thresholded.reshape(-1) != 127
    pl = det.CopyUnionMarkersTo()
    pairs = np.unique(np.stack([labels[mask].astype(np.int64), pl[mask].astype(np.int64)], axis=1), axis=0)
    assert len(pairs) == len(np.unique(labels[mask])) == len(np.unique(pl[mask])), f"product vs {what}: components"
    pq = det.FitQuads()
    assert len(pq) == len(corners)
    for q in pq["corners"]:
        assert min(float(np.abs(q - c).max()) for c in corners) <= CORNER_EXACT_TOL, f"product vs {what}: QuadCorners"
    # every detection's corners are one of upstream's refined quads (H maps (+-1,+-1) onto them)
    dets = det.Detections()
    for d in dets:
        best = min(match_corner_sets(d["p"], r) for r in refined)
        assert best <= REFINE_TOL_PX, (f"product detection vs {what} refined quad", best)
    return len(dets)


def test_reference_pins_oracle_and_product(oracle):
    from oracle import pyrefgpu
    from ros_vision_b200 import detector as D
    D.load_library()
    golden = np.load(GOLDEN_STAGES)
    frames = _frames()
    assert [str(n) for n in golden["names"]] == [f[0] for f in frames]
    live = pyrefgpu.available()
    total_quads = total_dets = 0
    for k, (name, yuyv, w, h, cam, dist) in enumerate(frames):
        g = {key[len(f"{k}_"):]: golden[key] for key in golden.files if key.startswith(f"{k}_")}
        orc = oracle.detect(oracle.make_config(w, h, "yuyv", 2, 0.0, camera=cam, dist=dist), yuyv)
        _compare_oracle_with_stored(orc, g, name)
        total_quads += len(g["refined"])

        det = D.GpuDetector(w, h, "yuyv", camera_matrix=cam, distortion_coefficients=dist, keep_stages=True)
        det.Detect(yuyv)
        # the product against upstream's stored stages (its thresholded image and partition are the oracle's, which
        # matched their digests above)
        labels = canonical_partition(orc.labels, orc.thresh.reshape(-1) != 127)
        total_dets += _compare_product(det, orc.thresh, labels, g["corners"], g["refined"], "stored reference")

        if live:   # upstream's GpuDetector itself, every exposed stage
            ref = pyrefgpu.ReferenceGpuDetector(w, h, cam or (1.0, 0.0, 1.0, 0.0), dist or (0.0,) * 5)
            ref.Detect(yuyv)
            report = {}
            rq = _compare_reference_with_oracle(ref, orc, report)
            print(name, report, "quads", len(rq), "detections", len(orc.detections))
            _compare_product(det, ref.thresholded(), ref.labels(), ref.quad_corners()["corners"], rq["corners"],
                             "live reference")
            ref.close()
        det.close()
    assert total_quads > 10 and total_dets > 5
