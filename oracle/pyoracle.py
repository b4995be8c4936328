"""TEST INFRASTRUCTURE: ctypes binding of oracle/liboracle.so.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this module; the product (ros_vision_b200/) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

FMT = {"gray": 0, "yuyv": 1, "bgr": 2}

STAGE_THRESHOLD, STAGE_LABELS, STAGE_POINTS, STAGE_BLOBS, STAGE_LINEFIT, STAGE_QUADS, STAGE_DECODE = range(1, 8)


class OrcConfig(C.Structure):
    _fields_ = [
        ("width", C.c_int), ("height", C.c_int), ("format", C.c_int), ("quad_decimate", C.c_int),
        ("quad_sigma", C.c_float), ("refine_edges", C.c_int), ("decode_sharpening", C.c_double),
        ("min_cluster_pixels", C.c_int), ("max_nmaxima", C.c_int), ("cos_critical_rad", C.c_float),
        ("max_line_fit_mse", C.c_float), ("min_white_black_diff", C.c_int),
        ("fx", C.c_double), ("cx", C.c_double), ("fy", C.c_double), ("cy", C.c_double),
        ("k1", C.c_double), ("k2", C.c_double), ("p1", C.c_double), ("p2", C.c_double), ("k3", C.c_double),
        ("max_stage", C.c_int), ("family_mask", C.c_uint32), ("families", C.c_void_p), ("nfamilies", C.c_int),
    ]


class OrcFamily(C.Structure):
    _fields_ = [
        ("name", C.c_char_p), ("nbits", C.c_int), ("ncodes", C.c_int), ("width_at_border", C.c_int),
        ("total_width", C.c_int), ("reversed_border", C.c_int), ("h", C.c_int), ("codes", C.POINTER(C.c_uint64)),
        ("bit_x", C.POINTER(C.c_int32)), ("bit_y", C.POINTER(C.c_int32)), ("max_hamming", C.c_int),
    ]


POINT_DT = np.dtype([("rep0", "<u4"), ("rep1", "<u4"), ("x", "<u2"), ("y", "<u2"), ("bx", "<u2"), ("by", "<u2"),
                     ("dir", "u1"), ("b2w", "u1"), ("pad", "u1", (2,))])
CLUSTER_DT = np.dtype([("rep0", "<u4"), ("rep1", "<u4"), ("min_x", "<u2"), ("min_y", "<u2"), ("max_x", "<u2"),
                       ("max_y", "<u2"), ("start", "<u4"), ("count", "<u4"), ("gx_sum", "<i4"), ("gy_sum", "<i4"),
                       ("pxgx_plus_pygy_sum", "<i8"), ("selected", "<i4"), ("sel_start", "<u4")])
SPOINT_DT = np.dtype([("blob", "<u4"), ("theta", "<u4"), ("x", "<u2"), ("y", "<u2"), ("bx", "<u2"), ("by", "<u2"),
                      ("dir", "u1"), ("pad", "u1", (3,))])
LFP_DT = np.dtype([("Mxx", "<i8"), ("Myy", "<i8"), ("Mxy", "<i8"), ("Mx", "<i8"), ("My", "<i8"), ("W", "<i8")])
MOMENTS_DT = np.dtype([("Mx", "<i8"), ("My", "<i8"), ("W", "<i8"), ("Mxx", "<i8"), ("Myy", "<i8"), ("Mxy", "<i8"),
                       ("N", "<i4"), ("pad", "<i4")])
FITQUAD_DT = np.dtype([("blob", "<u4"), ("rep0", "<u4"), ("rep1", "<u4"), ("valid", "<i4"), ("npeaks", "<i4"),
                       ("indices", "<u4", (4,)), ("pad0", "<u4"), ("moments", MOMENTS_DT, (4,)), ("err", "<f8")])
CORNERS_DT = np.dtype([("corners", "<f4", (4, 2)), ("reversed_border", "<i4"), ("blob", "<u4"), ("rep0", "<u4"),
                       ("rep1", "<u4")])
DET_DT = np.dtype([("id", "<i4"), ("hamming", "<i4"), ("decision_margin", "<f4"), ("rotation", "<i4"),
                   ("H", "<f8", (9,)), ("c", "<f8", (2,)), ("p", "<f8", (4, 2)), ("rep0", "<u4"), ("rep1", "<u4"),
                   ("family", "<i4"), ("pad", "<i4")])


class OrcResult(C.Structure):
    _fields_ = [
        ("W", C.c_int), ("H", C.c_int), ("w", C.c_int), ("h", C.c_int),
        ("gray", C.c_void_p), ("quad_im", C.c_void_p), ("minmax", C.c_void_p), ("thresh", C.c_void_p),
        ("labels", C.c_void_p), ("sizes", C.c_void_p),
        ("num_points", C.c_int), ("points", C.c_void_p),
        ("num_clusters", C.c_int), ("clusters", C.c_void_p),
        ("num_selected_points", C.c_int), ("spoints", C.c_void_p), ("lfps", C.c_void_p),
        ("errs", C.c_void_p), ("filtered_errs", C.c_void_p), ("is_peak", C.c_void_p),
        ("num_fitquads", C.c_int), ("fitquads", C.c_void_p),
        ("num_corners", C.c_int), ("corners", C.c_void_p),
        ("num_detections", C.c_int), ("detections", C.c_void_p),
        ("refined", C.c_void_p),
    ]


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("apriltag_oracle.c", "classic_detector.c", "apriltag_oracle.h", "oracle_internal.h",
                                             "cuda_math_emul.h", "tag_families.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s", "liboracle.so"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(so):
            build()
        L = C.CDLL(so)
        L.orc_default_config.argtypes = [C.POINTER(OrcConfig), C.c_int, C.c_int, C.c_int]
        L.orc_detect.argtypes = [C.POINTER(OrcConfig), C.c_void_p]
        L.orc_detect.restype = C.POINTER(OrcResult)
        L.orc_free_result.argtypes = [C.POINTER(OrcResult)]
        L.orc_emul_atan2f.argtypes = [C.c_float, C.c_float]
        L.orc_emul_atan2f.restype = C.c_float
        L.orc_emul_hypotf.argtypes = [C.c_float, C.c_float]
        L.orc_emul_hypotf.restype = C.c_float
        L.orc_undistort.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(OrcConfig)]
        L.orc_undistort.restype = C.c_int
        L.orc_redistort.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(OrcConfig)]
        L.orc_homography_compute.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_homography_compute.restype = C.c_int
        L.orc_tag36h11_code.argtypes = [C.c_int]
        L.orc_tag36h11_code.restype = C.c_uint64
        L.orc_decode_codeword.argtypes = [C.c_uint64, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.orc_decode_codeword.restype = C.c_int
        L.orc_decode_codeword_family.argtypes = [C.POINTER(OrcFamily), C.c_uint64, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.orc_decode_codeword_family.restype = C.c_int
        L.orc_family_get.argtypes = [C.c_int]
        L.orc_family_get.restype = C.POINTER(OrcFamily)
        L.orc_classic_detect.argtypes = [C.POINTER(OrcConfig), C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.orc_classic_detect.restype = C.c_int
        L.orc_family_index.argtypes = [C.c_char_p]
        L.orc_family_index.restype = C.c_int
        _LIB = L
    return _LIB


FAMILY_NAMES = ("tag36h11", "tag25h9", "tag16h5")   # bit positions of OrcConfig.family_mask


def family_mask(families) -> int:
    if isinstance(families, str):
        families = [families]
    return sum(1 << FAMILY_NAMES.index(f) for f in families)


def family_table(family) -> OrcFamily:
    """An orc_family from a built-in name or from a dict in the layout GpuDetector takes (ros_vision_b200.tag_families
    entries + optional "reversed_border", "max_hamming", "name").  The arrays it points to live on the returned object."""
    if isinstance(family, str):
        i = lib().orc_family_index(family.encode())
        if i < 0:
            raise ValueError(f"no built-in tag family {family!r}")
        return lib().orc_family_get(i).contents
    fam = OrcFamily()
    fam._keep = (f"{family.get('name', 'custom')}".encode(), (C.c_uint64 * len(family["codes"]))(*family["codes"]),
                 (C.c_int32 * family["nbits"])(*family["bit_x"]), (C.c_int32 * family["nbits"])(*family["bit_y"]))
    fam.name, fam.codes, fam.bit_x, fam.bit_y = fam._keep
    fam.nbits, fam.ncodes = family["nbits"], len(family["codes"])
    fam.width_at_border, fam.total_width = family["width_at_border"], family["total_width"]
    fam.reversed_border, fam.max_hamming = int(family.get("reversed_border", 0)), int(family.get("max_hamming", 2))
    fam.h = int(family.get("min_hamming", 0))
    return fam


def decode_codeword(family, word: int, max_hamming: int):
    """quick_decode_codeword of the oracle for `family` (name or dict) at `max_hamming`: (id, hamming, rotation) or
    None."""
    table = family_table(family)
    fam = OrcFamily.from_buffer_copy(table)   # (the copy points into `table`'s arrays, alive until we return)
    fam.max_hamming = int(max_hamming)
    h, r = C.c_int(), C.c_int()
    i = lib().orc_decode_codeword_family(C.byref(fam), C.c_uint64(word), C.byref(h), C.byref(r))
    return None if i < 0 else (i, h.value, r.value)


def make_config(width, height, fmt="yuyv", quad_decimate=2, quad_sigma=0.0, refine_edges=True, camera=None,
                dist=None, max_stage=STAGE_DECODE, families=("tag36h11",), **qtp) -> OrcConfig:
    """`families` as GpuDetector takes them: built-in names select the oracle's tables by family_mask (detections
    carry the built-in index); a list with any dict becomes the configuration's own family list, in that order
    (detections carry the index into it)."""
    cfg = OrcConfig()
    lib().orc_default_config(C.byref(cfg), width, height, FMT[fmt])
    cfg.quad_decimate = int(quad_decimate)
    cfg.quad_sigma = float(quad_sigma)
    cfg.refine_edges = int(bool(refine_edges))
    cfg.max_stage = max_stage
    if isinstance(families, (str, dict)):
        families = [families]
    if all(isinstance(f, str) for f in families):
        cfg.family_mask = family_mask(families)
    else:
        tables = [family_table(f) for f in families]
        arr = (OrcFamily * len(tables))(*tables)
        cfg._keep = (tables, arr)
        cfg.families, cfg.nfamilies = C.addressof(arr), len(tables)
    if camera is not None:
        cfg.fx, cfg.cx, cfg.fy, cfg.cy = camera
    if dist is not None:
        cfg.k1, cfg.k2, cfg.p1, cfg.p2, cfg.k3 = dist
    for k, v in qtp.items():
        setattr(cfg, k, v)
    return cfg


def _arr(ptr, dtype, count):
    if not ptr or count == 0:
        return np.zeros((0,), dtype=dtype)
    nbytes = np.dtype(dtype).itemsize * count
    buf = (C.c_char * nbytes).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype, count=count).copy()


class Result:
    """Host copy of every stage the oracle produced."""

    def __init__(self, r: OrcResult):
        self.W, self.H, self.w, self.h = r.W, r.H, r.w, r.h
        N, n = self.W * self.H, self.w * self.h
        self.gray = _arr(r.gray, np.uint8, N).reshape(self.H, self.W)
        self.quad_im = _arr(r.quad_im, np.uint8, n).reshape(self.h, self.w)
        self.minmax = _arr(r.minmax, np.uint8, (self.w // 4) * (self.h // 4) * 2).reshape(self.h // 4, self.w // 4, 2)
        self.thresh = _arr(r.thresh, np.uint8, n).reshape(self.h, self.w)
        self.labels = _arr(r.labels, np.uint32, n if r.labels else 0)
        self.sizes = _arr(r.sizes, np.uint32, n if r.sizes else 0)
        self.points = _arr(r.points, POINT_DT, r.num_points)
        self.clusters = _arr(r.clusters, CLUSTER_DT, r.num_clusters)
        ns = r.num_selected_points
        self.spoints = _arr(r.spoints, SPOINT_DT, ns if r.spoints else 0)
        self.lfps = _arr(r.lfps, LFP_DT, ns if r.lfps else 0)
        self.errs = _arr(r.errs, np.float64, ns if r.errs else 0)
        self.filtered_errs = _arr(r.filtered_errs, np.float64, ns if r.filtered_errs else 0)
        self.is_peak = _arr(r.is_peak, np.uint8, ns if r.is_peak else 0)
        self.fitquads = _arr(r.fitquads, FITQUAD_DT, r.num_fitquads)
        self.corners = _arr(r.corners, CORNERS_DT, r.num_corners)
        self.detections = _arr(r.detections, DET_DT, r.num_detections)
        self.refined = _arr(r.refined, CORNERS_DT, r.num_corners if r.refined else 0)


def detect(cfg: OrcConfig, image: np.ndarray) -> Result:
    image = np.ascontiguousarray(image, dtype=np.uint8)
    bpp = {0: 1, 1: 2, 2: 3}[cfg.format]
    assert image.size == cfg.width * cfg.height * bpp, (image.shape, cfg.width, cfg.height, cfg.format)
    p = lib().orc_detect(C.byref(cfg), image.ctypes.data_as(C.c_void_p))
    if not p:
        raise ValueError("oracle rejected the configuration")
    try:
        return Result(p.contents)
    finally:
        lib().orc_free_result(p)


def detect_raw(cfg: OrcConfig, image: np.ndarray) -> int:
    """Runs the oracle and returns only the detection count (used for timing; no stage copies)."""
    p = lib().orc_detect(C.byref(cfg), image.ctypes.data_as(C.c_void_p))
    n = p.contents.num_detections
    lib().orc_free_result(p)
    return n


def classic_detect(cfg: OrcConfig, gray: np.ndarray, cap: int = 1024):
    """The classic CPU detector (libapriltag apriltag_detector_detect restated, oracle/classic_detector.c) on a gray
    frame.  Returns (detections as DET_DT array, number of candidate quads)."""
    gray = np.ascontiguousarray(gray, dtype=np.uint8)
    assert gray.size == cfg.width * cfg.height, (gray.shape, cfg.width, cfg.height)
    out = np.zeros(cap, dtype=DET_DT)
    nq = C.c_int()
    n = lib().orc_classic_detect(C.byref(cfg), gray.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), cap, C.byref(nq))
    if n < 0:
        raise ValueError("classic detector rejected the configuration")
    return out[:min(n, cap)].copy(), nq.value


def classic_detect_raw(cfg: OrcConfig, gray: np.ndarray) -> int:
    """Detection count only (timing)."""
    return lib().orc_classic_detect(C.byref(cfg), gray.ctypes.data_as(C.c_void_p), None, 0, None)
