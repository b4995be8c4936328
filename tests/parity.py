"""Stage-by-stage comparison of the CUDA engine (through the C ABI) with the CPU oracle.

Bars (BASELINE.json north_star): thresholded image, component labels, boundary points, blob
extents, point order, moments, fit quads and quad corners bit-exact; tag ids and hamming
bit-exact; detection corners within 0.05 px and homographies within 1e-4 relative (the refine
stage calls single-precision sin/cos/atan2 from the host libm in the reference and from the
device libm here).
"""
from __future__ import annotations

import numpy as np

from ros_vision_b200 import detector as D

CORNER_TOL_PX = 0.05
H_REL_TOL = 1e-4


def _key64(rep0, rep1):
    return (np.asarray(rep0, dtype=np.uint64) << np.uint64(32)) | np.asarray(rep1, dtype=np.uint64)


def compare_front_end(det: D.GpuDetector, orc, frame=0, fmt="yuyv"):
    if fmt != "gray":
        assert np.array_equal(det.CopyGrayTo(frame), orc.gray), "gray image"
    assert np.array_equal(det.CopyDecimatedTo(frame), orc.quad_im), "quad (decimated/blurred) image"
    assert np.array_equal(det.CopyThresholdedTo(frame), orc.thresh), "thresholded image"
    if det.cfg.keep_stages:
        assert np.array_equal(det.CopyStage(D.STAGE_MINMAX, frame).reshape(orc.minmax.shape), orc.minmax), "tile min/max"
    labels = det.CopyUnionMarkersTo(frame)
    sizes = det.CopyUnionMarkersSizeTo(frame)
    mask = orc.thresh.reshape(-1) != 127
    assert np.array_equal(labels[mask], orc.labels[mask]), "component labels"
    assert np.array_equal(sizes, orc.sizes), "component sizes"
    return labels, sizes


def compare_points_and_blobs(det: D.GpuDetector, orc, frame=0):
    info = det.FrameInfo(frame)
    assert info.status == 0, f"device buffer overflow, status={info.status}"
    assert info.num_points == len(orc.points), (info.num_points, len(orc.points))
    assert info.num_clusters == len(orc.clusters)
    assert info.num_blobs == int(orc.clusters["selected"].sum())
    assert info.num_selected_points == len(orc.spoints)
    clusters = det.CopyStage(D.STAGE_CLUSTERS, frame)
    assert len(clusters) == len(orc.clusters)
    ckey = _key64(clusters["rep0"], clusters["rep1"])
    order = np.argsort(ckey, kind="stable")
    clusters = clusters[order]
    okey = _key64(orc.clusters["rep0"], orc.clusters["rep1"])
    assert np.array_equal(ckey[order], okey), "blob pair keys"
    for a, b in (("min_x", "min_x"), ("min_y", "min_y"), ("max_x", "max_x"), ("max_y", "max_y"), ("count", "count"),
                 ("gx_sum", "gx_sum"), ("gy_sum", "gy_sum"), ("pxgx_plus_pygy_sum", "pxgx_plus_pygy_sum")):
        assert np.array_equal(clusters[a].astype(np.int64), orc.clusters[b].astype(np.int64)), f"extents.{a}"
    assert np.array_equal(clusters["selected"] != 0, orc.clusters["selected"] != 0), "SelectBlobs"
    # boundary points as a set keyed by blob pair
    slot_to_key = {int(s): int(k) for s, k in zip(clusters["slot"], okey)}
    pts = det.CopyStage(D.STAGE_POINTS, frame)
    pkey = np.array([slot_to_key[int(s)] for s in pts["slot"]], dtype=np.uint64) if len(pts) else np.zeros(0, np.uint64)
    got = np.stack([pkey, pts["x"].astype(np.uint64), pts["y"].astype(np.uint64), pts["dir"].astype(np.uint64),
                    pts["black_to_white"].astype(np.uint64)], axis=1) if len(pts) else np.zeros((0, 5), np.uint64)
    ref = np.stack([_key64(orc.points["rep0"], orc.points["rep1"]), orc.points["x"].astype(np.uint64),
                    orc.points["y"].astype(np.uint64), orc.points["dir"].astype(np.uint64),
                    orc.points["b2w"].astype(np.uint64)], axis=1) if len(orc.points) else np.zeros((0, 5), np.uint64)
    got = got[np.lexsort(got.T[::-1])]
    ref = ref[np.lexsort(ref.T[::-1])]
    assert np.array_equal(got, ref), "boundary point set"
    return clusters


def compare_line_fit(det: D.GpuDetector, orc, frame=0):
    """Sorted points, prefix moments, errors, filtered errors -- per blob, bit-exact."""
    blobs = det.CopyStage(D.STAGE_BLOBS, frame)
    keys = det.CopyStage(D.STAGE_SORTED_POINTS, frame)
    lfp = det.CopyStage(D.STAGE_LINE_FIT_POINTS, frame)
    errs = det.CopyStage(D.STAGE_ERRORS, frame)
    filt = det.CopyStage(D.STAGE_FILTERED_ERRORS, frame)
    sel = orc.clusters[orc.clusters["selected"] != 0]
    okey = _key64(sel["rep0"], sel["rep1"])
    # STAGE_BLOBS lists every blob pair within the point-count limits; .selected = passed SelectBlobs
    cand = orc.clusters[(orc.clusters["count"] >= 24) & (orc.clusters["count"] <= 4 * (orc.w + orc.h))]
    assert np.array_equal(np.sort(_key64(blobs["rep0"], blobs["rep1"])), _key64(cand["rep0"], cand["rep1"])), "candidate blob set"
    chosen = blobs[blobs["selected"] != 0]
    bkey = _key64(chosen["rep0"], chosen["rep1"])
    assert np.array_equal(np.sort(bkey), okey), "selected blob set"
    lut = {int(k): i for i, k in enumerate(okey)}
    for b in chosen:
        o = sel[lut[int(_key64(b["rep0"], b["rep1"]))]]
        cnt = int(b["count"])
        assert cnt == int(o["count"])
        for fld in ("min_x", "min_y", "max_x", "max_y", "gx_sum", "gy_sum", "pxgx_plus_pygy_sum"):
            assert int(b[fld]) == int(o[fld]), f"blob extents .{fld}"
        g0, o0 = int(b["offset"]), int(o["sel_start"])
        sp = orc.spoints[o0:o0 + cnt]
        ref_key = ((sp["theta"].astype(np.uint64) << np.uint64(26)) | (sp["dir"].astype(np.uint64) << np.uint64(24)) |
                   (sp["by"].astype(np.uint64) << np.uint64(12)) | sp["bx"].astype(np.uint64))
        assert np.array_equal(keys[g0:g0 + cnt], ref_key), f"angle-sorted points of blob {b['rep0']},{b['rep1']}"
        for fld in ("Mxx", "Myy", "Mxy", "Mx", "My", "W"):
            assert np.array_equal(lfp[fld][g0:g0 + cnt], orc.lfps[fld][o0:o0 + cnt]), f"prefix moment {fld}"
        assert np.array_equal(errs[g0:g0 + cnt].astype(np.float64), orc.errs[o0:o0 + cnt]), "line-fit errors"
        assert np.array_equal(filt[g0:g0 + cnt], orc.filtered_errs[o0:o0 + cnt]), "filtered errors"
    return blobs


def compare_quads(det: D.GpuDetector, orc, blobs, frame=0):
    fq = det.CopyStage(D.STAGE_FIT_QUADS, frame)
    assert len(fq) == len(orc.fitquads), "number of FitQuads"
    gk = _key64(blobs["rep0"][fq["blob_index"]], blobs["rep1"][fq["blob_index"]])
    fq = fq[np.argsort(gk, kind="stable")]
    ok = _key64(orc.fitquads["rep0"], orc.fitquads["rep1"])
    assert np.array_equal(np.sort(gk), ok)
    assert np.array_equal(fq["valid"] != 0, orc.fitquads["valid"] != 0), "FitQuad.valid"
    assert np.array_equal(fq["num_peaks"], orc.fitquads["npeaks"]), "peak counts"
    v = fq["valid"] != 0
    assert np.array_equal(fq["indices"][v], orc.fitquads["indices"][v]), "FitQuad.indices"
    assert np.array_equal(fq["err"][v], orc.fitquads["err"][v]), "FitQuad error"
    for fld in ("Mx", "My", "W", "Mxx", "Myy", "Mxy", "N"):
        assert np.array_equal(fq["moments"][fld][v], orc.fitquads["moments"][fld][v]), f"FitQuad.moments.{fld}"
    quads = det.FitQuads(frame)
    assert len(quads) == len(orc.corners), "number of QuadCorners"
    assert np.array_equal(_key64(quads["rep0"], quads["rep1"]), _key64(orc.corners["rep0"], orc.corners["rep1"]))
    assert np.array_equal(quads["corners"], orc.corners["corners"]), "QuadCorners (bit-exact float)"
    return quads


# decision_margin: the mean of bilinear samples minus the gray-model threshold.  The sample positions move with the
# refined corners (typical difference between device and host single-precision trigonometry: 6.1e-5 px; more on tiny or
# ill-conditioned quads, always below CORNER_TOL_PX), the image gradient is at most 255 grey levels per pixel: the
# tolerance is 255 levels/px times three times the corner difference actually observed on that detection, with a floor
# of 2e-4 px.
MARGIN_FLOOR_PX = 2e-4


def margin_tolerance(corner_diff_px):
    return 255.0 * np.maximum(MARGIN_FLOOR_PX, 3.0 * np.asarray(corner_diff_px))


def _project(H, x, y):
    H = np.asarray(H, dtype=np.float64).reshape(3, 3)
    v = H @ np.array([x, y, 1.0])
    return v[:2] / v[2]


def _dlt(src, dst):
    """Homography with H[2][2] = 1 through four correspondences, float64 (independent of the engine's elimination)."""
    A, b = [], []
    for (x, y), (u, v) in zip(src, dst):
        A.append([x, y, 1, 0, 0, 0, -x * u, -y * u]); b.append(u)
        A.append([0, 0, 0, x, y, 1, -x * v, -y * v]); b.append(v)
    h = np.linalg.solve(np.array(A, dtype=np.float64), np.array(b, dtype=np.float64))
    return np.append(h, 1.0).reshape(3, 3)


TAG_CORNERS = [(-1.0, 1.0), (1.0, 1.0), (1.0, -1.0), (-1.0, -1.0)]  # det->p[i] = H * (tcx, tcy), quad_decode_task


def check_detection_geometry(dets, max_hamming=2):
    """Checks that need no oracle (they pin H, c and p of a detection against each other and against independent
    homography solvers): H is THE homography that maps the tag corners (+-1, +-1) to p; c = H (0, 0).  `max_hamming`:
    the largest any of the detector's families corrects (2 unless a family table says otherwise)."""
    for d in dets:
        H = np.asarray(d["H"], dtype=np.float64).reshape(3, 3)
        assert H[2, 2] != 0 and np.isfinite(H).all()
        Hn = H / H[2, 2]
        scale = max(1.0, np.abs(d["p"]).max())
        assert np.abs(_project(H, 0, 0) - d["c"]).max() <= 1e-9 * scale, "c == H (0, 0)"
        for (x, y), pt in zip(TAG_CORNERS, d["p"]):
            assert np.abs(_project(H, x, y) - pt).max() <= 1e-9 * scale, "p[i] == H (+-1, +-1)"
        # float64 DLT through the detection's own corners: the same matrix (H is fixed by 4 points up to scale)
        ref = _dlt(TAG_CORNERS, d["p"])
        a = np.abs(ref[:2, :2]).max()
        assert np.abs(Hn[:2, :2] - ref[:2, :2]).max() <= 1e-7 * a, "H[0:2,0:2] vs float64 DLT"
        assert np.abs(Hn[:2, 2] - ref[:2, 2]).max() <= 1e-7 * scale, "H[0:2,2] vs float64 DLT"
        assert np.abs(Hn[2, :2] - ref[2, :2]).max() <= 1e-7 * max(np.abs(ref[2, :2]).max(), 1.0 / a), "H[2,0:2] vs float64 DLT"
        try:  # third party: OpenCV's solver (float32 corner input, so 1e-4 relative is what it can confirm)
            import cv2
            cvH = cv2.getPerspectiveTransform(np.array(TAG_CORNERS, dtype=np.float32), np.asarray(d["p"], dtype=np.float32))
            assert np.abs(Hn[:2, :2] - cvH[:2, :2]).max() <= H_REL_TOL * a, "H vs cv2.getPerspectiveTransform"
            assert np.abs(Hn[:2, 2] - cvH[:2, 2]).max() <= 1e-3, "H translation vs cv2.getPerspectiveTransform"
            assert np.abs(Hn[2, :2] - cvH[2, :2]).max() <= H_REL_TOL * max(np.abs(cvH[2, :2]).max(), 1.0 / a), "H[2,:] vs cv2"
        except ImportError:
            pass
        assert 0 <= int(d["hamming"]) <= max_hamming and float(d["decision_margin"]) >= 0.0
    ids = [int(x) for x in dets["id"]]
    assert ids == sorted(ids), "detections are sorted by id (apriltag_detect.cu:662)"


def compare_homography(got_H, ref_H, corner_tol=CORNER_TOL_PX):
    """north_star: homographies within 1e-4 relative.  Both matrices are scaled to H[2][2] = 1, then
      * the whole matrix: Frobenius norm of the difference <= 1e-4 of the reference's norm;
      * element-wise, each block against ITS OWN scale, so that the small perspective terms are really checked:
        the 2x2 block |dH| <= 1e-4 * max|block|, the translation column within the corner tolerance,
        the perspective row |dH| <= 1e-4 * max|row| + what a `corner_tol` corner change can produce (tol / a^2);
      * projected tag corners and centre within the corner tolerance."""
    g = np.asarray(got_H, dtype=np.float64).reshape(3, 3)
    r = np.asarray(ref_H, dtype=np.float64).reshape(3, 3)
    g, r = g / g[2, 2], r / r[2, 2]
    assert np.linalg.norm(g - r) <= H_REL_TOL * np.linalg.norm(r), "homography (Frobenius)"
    a = np.abs(r[:2, :2]).max()
    assert np.abs(g[:2, :2] - r[:2, :2]).max() <= H_REL_TOL * a, "homography 2x2 block"
    assert np.abs(g[:2, 2] - r[:2, 2]).max() <= corner_tol, "homography translation"
    assert np.abs(g[2, :2] - r[2, :2]).max() <= H_REL_TOL * np.abs(r[2, :2]).max() + corner_tol / (a * a), "homography perspective row"
    for x, y in TAG_CORNERS + [(0.0, 0.0)]:
        assert np.abs(_project(g, x, y) - _project(r, x, y)).max() <= corner_tol, "projected tag corner"


def compare_detections(det: D.GpuDetector, orc, frame=0):
    got = det.Detections(frame)
    ref = orc.detections
    assert [int(x) for x in got["id"]] == [int(x) for x in ref["id"]], "tag ids"
    assert np.array_equal(got["hamming"], ref["hamming"]), "hamming"
    families = getattr(det, "families", ["tag36h11"])
    if "family" in got.dtype.names and "family" in ref.dtype.names:
        # the engine numbers the families as its caller listed them; the oracle by its built-in table when it was
        # given names only, else by the caller's list too (pyoracle.make_config)
        from oracle.pyoracle import FAMILY_NAMES
        mine = [f if isinstance(f, str) else f.get("name") for f in families]
        theirs = FAMILY_NAMES if all(isinstance(f, str) for f in families) else mine
        assert [mine[int(i)] for i in got["family"]] == [theirs[int(i)] for i in ref["family"]], "tag family"
    if len(ref):
        assert np.abs(got["p"] - ref["p"]).max() <= CORNER_TOL_PX, "corners"
        assert np.abs(got["c"] - ref["c"]).max() <= CORNER_TOL_PX, "centres"
        for g, r in zip(got, ref):
            compare_homography(g["H"], r["H"])
        dp = np.abs(got["p"] - ref["p"]).reshape(len(ref), -1).max(axis=1)
        dm = np.abs(got["decision_margin"].astype(np.float64) - ref["decision_margin"].astype(np.float64))
        assert (dm <= margin_tolerance(dp)).all(), f"decision margin: diff {dm.tolist()} at corner diff {dp.tolist()}"
    max_hamming = max(2 if isinstance(f, str) else int(f.get("max_hamming", 2)) for f in families)
    check_detection_geometry(got, max_hamming)
    check_detection_geometry(ref, max_hamming)
    return got


def compare_all(det: D.GpuDetector, orc, frame=0, fmt="yuyv"):
    compare_front_end(det, orc, frame, fmt)
    compare_points_and_blobs(det, orc, frame)
    blobs = compare_line_fit(det, orc, frame)
    compare_quads(det, orc, blobs, frame)
    return compare_detections(det, orc, frame)
