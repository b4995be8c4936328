"""Shared helpers for the parity tests."""
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_png_gray(path):
    import cv2
    im = cv2.imread(path, cv2.IMREAD_UNCHANGED)
    assert im is not None and im.ndim == 2, path
    return np.ascontiguousarray(im)


def load_golden(name):
    with open(os.path.join(GOLDEN, name + ".json")) as f:
        meta = json.load(f)
    img = load_png_gray(os.path.join(GOLDEN, meta["image"]))
    assert img.shape == (meta["height"], meta["width"])
    return meta, img


def match_corner_sets(a, b):
    """Max distance between two 4-corner sets under the best cyclic shift / reversal."""
    a = np.asarray(a, dtype=np.float64).reshape(4, 2)
    b = np.asarray(b, dtype=np.float64).reshape(4, 2)
    best = np.inf
    for rev in (False, True):
        bb = b[::-1] if rev else b
        for s in range(4):
            d = np.abs(a - np.roll(bb, s, axis=0)).max()
            best = min(best, d)
    return best


def canonical_partition(labels, mask):
    """Relabel `labels` (flat) by first occurrence over mask==True pixels; others -> -1."""
    labels = np.asarray(labels).reshape(-1)
    mask = np.asarray(mask).reshape(-1)
    out = np.full(labels.shape, -1, dtype=np.int64)
    vals = labels[mask]
    _, first_idx, inv = np.unique(vals, return_index=True, return_inverse=True)
    order = np.argsort(np.argsort(first_idx))
    out[mask] = order[inv]
    return out


def stage_digest(*cols):
    return hashlib.sha256(np.stack([np.asarray(c, dtype=np.int64).reshape(-1) for c in cols], axis=1).tobytes()).hexdigest()


def reference_stage_record(orc, err_samples=256):
    """The stages test_gpu_reference_live compares with upstream GpuDetector, in a form a golden file can hold: SHA-256
    digests of the integer stages (component labels relabelled by first occurrence, so every labelling of the same
    partition has the same digest), a seeded sample of the line-fit errors, and the quad corners in full."""
    mask = orc.thresh.reshape(-1) != 127
    ol = orc.labels.reshape(-1)
    part = canonical_partition(ol, mask)
    u, first = np.unique(ol[mask], return_index=True)
    canon_u = part[mask][first]

    def canon(rep):
        pos = np.searchsorted(u, rep)
        assert np.array_equal(u[np.minimum(pos, len(u) - 1)], rep), "blob representative outside the partition"
        return canon_u[pos]

    pt, cl, sp, lf, fq, qc = orc.points, orc.clusters, orc.spoints, orc.lfps, orc.fitquads, orc.corners
    valid = fq["valid"] != 0
    mom = fq["moments"]
    rng = np.random.default_rng(len(orc.errs))
    idx = np.sort(rng.choice(len(orc.errs), size=min(err_samples, len(orc.errs)), replace=False))
    return {
        "digest_gray": stage_digest(orc.gray),
        "digest_decimated": stage_digest(orc.quad_im),
        "digest_thresholded": stage_digest(orc.thresh),
        "digest_partition": stage_digest(part[mask]),
        "digest_sizes": stage_digest(orc.sizes[ol[mask]]),
        "digest_points": stage_digest(canon(pt["rep0"]), canon(pt["rep1"]), pt["x"], pt["y"], pt["dir"], pt["b2w"]),
        "digest_extents": stage_digest(canon(cl["rep0"]), canon(cl["rep1"]), *(cl[f] for f in (
            "min_x", "min_y", "max_x", "max_y", "count", "gx_sum", "gy_sum", "pxgx_plus_pygy_sum")), cl["selected"] != 0),
        "digest_sorted_selected": stage_digest(sp["theta"], sp["x"], sp["y"], sp["dir"]),
        "digest_prefix_moments": stage_digest(*(lf[f] for f in ("Mxx", "Myy", "Mxy", "Mx", "My", "W"))),
        "digest_fit_quads": stage_digest(canon(fq["rep0"]), canon(fq["rep1"]), valid,
                                    *(np.where(valid, fq["indices"][:, j], 0) for j in range(4)),
                                    *(np.where(valid, mom[f][:, j], 0) for f in ("Mx", "My", "W", "Mxx", "Myy", "Mxy", "N")
                                      for j in range(4))),
        "num_points": len(pt), "num_blob_pairs": len(cl), "num_selected_points": len(sp), "num_fit_quads": len(fq),
        "err_index": idx, "err": orc.errs[idx], "filtered_err": orc.filtered_errs[idx],
        "err_absmax": np.array([np.abs(orc.errs).max(initial=0.0), np.abs(orc.filtered_errs).max(initial=0.0)]),
        "corner_blob": np.stack([canon(qc["rep0"]), canon(qc["rep1"])], axis=1).reshape(-1, 2),
        "corners": qc["corners"], "reversed_border": qc["reversed_border"], "refined": orc.refined["corners"],
    }
