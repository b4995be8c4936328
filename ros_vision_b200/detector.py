"""Python host side of the B200 AprilTag engine: a ctypes mirror of the reference's
`frc971::apriltag::GpuDetector` (src/apriltags_cuda/include/apriltags_cuda/apriltag_gpu.h:77-359)
over the C ABI in include/b200tag.h.

Method names follow the reference class (Detect, Detections, FitQuads, CopyGrayTo, ...).
There is no CPU fallback: if libb200tag.so is missing or no CUDA device is present the
constructor raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200tag.so")

FMT = {"gray": 0, "yuyv": 1, "bgr": 2}
BYTES_PER_PIXEL = {"gray": 1, "yuyv": 2, "bgr": 3}

(STAGE_GRAY, STAGE_QUAD_IMAGE, STAGE_THRESHOLD, STAGE_LABELS, STAGE_SIZES, STAGE_POINTS, STAGE_BLOBS,
 STAGE_SORTED_POINTS, STAGE_LINE_FIT_POINTS, STAGE_ERRORS, STAGE_FILTERED_ERRORS, STAGE_FIT_QUADS, STAGE_QUADS,
 STAGE_RAW_DETECTIONS, STAGE_MINMAX, STAGE_CLUSTERS) = range(16)

ST_POINTS_OVERFLOW, ST_HASH_OVERFLOW, ST_BLOBS_OVERFLOW, ST_QUADS_OVERFLOW, ST_DETS_OVERFLOW, ST_JPEG_TRUNCATED = 1, 2, 4, 8, 16, 32


class B200TagError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("format", C.c_int32),
        ("quad_decimate", C.c_int32), ("quad_sigma", C.c_float), ("refine_edges", C.c_int32),
        ("decode_sharpening", C.c_double), ("min_cluster_pixels", C.c_int32), ("max_nmaxima", C.c_int32),
        ("cos_critical_rad", C.c_float), ("max_line_fit_mse", C.c_float), ("min_white_black_diff", C.c_int32),
        ("fx", C.c_double), ("cx", C.c_double), ("fy", C.c_double), ("cy", C.c_double),
        ("k1", C.c_double), ("k2", C.c_double), ("p1", C.c_double), ("p2", C.c_double), ("k3", C.c_double),
        ("max_batch", C.c_int32), ("device", C.c_int32), ("keep_stages", C.c_int32),
        ("max_points", C.c_uint32), ("max_blobs", C.c_uint32), ("max_detections", C.c_uint32),
        ("test_flags", C.c_int32), ("reserved", C.c_int32 * 7),
    ]


class FrameInfo(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("status", "num_points", "num_clusters", "num_blobs", "num_selected_points",
                                          "num_fit_quads", "num_quads", "num_detections")]


DETECTION_DT = np.dtype([("id", "<i4"), ("hamming", "<i4"), ("decision_margin", "<f4"), ("frame", "<i4"),
                         ("family", "<i4"), ("reserved", "<i4"), ("H", "<f8", (9,)), ("c", "<f8", (2,)), ("p", "<f8", (4, 2))])


class Family(C.Structure):
    """b200tag_family: the fields of libapriltag's apriltag_family_t that detection reads."""
    _fields_ = [("name", C.c_char_p), ("nbits", C.c_uint32), ("ncodes", C.c_uint32), ("codes", C.POINTER(C.c_uint64)),
                ("bit_x", C.POINTER(C.c_uint32)), ("bit_y", C.POINTER(C.c_uint32)), ("width_at_border", C.c_int32),
                ("total_width", C.c_int32), ("reversed_border", C.c_int32), ("max_hamming", C.c_int32)]
QUAD_DT = np.dtype([("corners", "<f4", (4, 2)), ("reversed_border", "<i4"), ("blob_index", "<u4"), ("rep0", "<u4"),
                    ("rep1", "<u4")])
POINT_DT = np.dtype([("slot", "<u4"), ("x", "<u2"), ("y", "<u2"), ("dir", "u1"), ("black_to_white", "u1"),
                     ("pad", "u1", (2,))])
BLOB_DT = np.dtype([("rep0", "<u4"), ("rep1", "<u4"), ("min_x", "<u4"), ("min_y", "<u4"), ("max_x", "<u4"),
                    ("max_y", "<u4"), ("count", "<u4"), ("offset", "<u4"), ("gx_sum", "<i4"), ("gy_sum", "<i4"),
                    ("pxgx_plus_pygy_sum", "<i8"), ("slot", "<u4"), ("selected", "<i4")])
LFP_DT = np.dtype([("Mxx", "<i8"), ("Myy", "<i8"), ("Mxy", "<i8"), ("Mx", "<i8"), ("My", "<i8"), ("W", "<i8")])
MOMENTS_DT = np.dtype([("Mx", "<i8"), ("My", "<i8"), ("W", "<i8"), ("Mxx", "<i8"), ("Myy", "<i8"), ("Mxy", "<i8"),
                       ("N", "<i4"), ("pad", "<i4")])
FIT_QUAD_DT = np.dtype([("blob_index", "<u4"), ("valid", "<i4"), ("num_peaks", "<i4"), ("indices", "<u4", (4,)),
                        ("pad", "<u4"), ("moments", MOMENTS_DT, (4,)), ("err", "<f8")])

_STAGE_DTYPES = {
    STAGE_GRAY: np.uint8, STAGE_QUAD_IMAGE: np.uint8, STAGE_THRESHOLD: np.uint8, STAGE_LABELS: np.uint32,
    STAGE_SIZES: np.uint32, STAGE_POINTS: POINT_DT, STAGE_BLOBS: BLOB_DT, STAGE_SORTED_POINTS: np.uint64,
    STAGE_LINE_FIT_POINTS: LFP_DT, STAGE_ERRORS: np.float32, STAGE_FILTERED_ERRORS: np.float64,
    STAGE_FIT_QUADS: FIT_QUAD_DT, STAGE_QUADS: QUAD_DT, STAGE_RAW_DETECTIONS: DETECTION_DT, STAGE_MINMAX: np.uint8,
    STAGE_CLUSTERS: BLOB_DT,
}

POSE_DT = np.dtype([("R", "<f8", (3, 3)), ("t", "<f8", (3,)), ("err", "<f8"), ("err_other", "<f8")])
TAG_POSITION_DT = np.dtype([("index", "<i4"), ("id", "<i4"), ("camera", "<f8", (3,)), ("robot", "<f8", (3,)),
                            ("distance", "<f8"), ("err", "<f8")])  # b200tag_tag_position
POSE_METHODS = {"oi": 0, "ippe": 1}  # B200TAG_POSE_ORTHOGONAL_ITERATION, B200TAG_POSE_IPPE
FIELD_TAG_DT = np.dtype([("family", "<i4"), ("id", "<i4"), ("R", "<f8", (3, 3)), ("t", "<f8", (3,))])  # b200tag_field_tag
FIELD_POSE_DT = np.dtype([("num_tags", "<i4"), ("iterations", "<i4"), ("reserved", "<i4", (2,)), ("camera_R", "<f8", (3, 3)),
                          ("camera_t", "<f8", (3,)), ("robot_R", "<f8", (3, 3)), ("robot_t", "<f8", (3,)), ("rms", "<f8"),
                          ("rms_other", "<f8")])  # b200tag_field_pose
COVARIANCE_DT = np.dtype([("C", "<f8", (6, 6))])  # b200tag_covariance: xi = (rx, ry, rz, tx, ty, tz), rad and m
FIELD_COVARIANCE_DT = np.dtype([("camera", "<f8", (6, 6)), ("robot", "<f8", (6, 6))])  # b200tag_field_covariance
FLOOR_POSE_DT = np.dtype([("num_tags", "<i4"), ("iterations", "<i4"), ("mode", "<i4"), ("reserved", "<i4"), ("x", "<f8"),
                          ("y", "<f8"), ("cos_heading", "<f8"), ("sin_heading", "<f8"), ("heading", "<f8"), ("rms", "<f8"),
                          ("rms_other", "<f8")])  # b200tag_floor_pose; mode 0 free, 1 prior, 2 fixed
FLOOR_MODES = {0: "free", 1: "prior", 2: "fixed"}

_lib = None


def load_library():
    """Loads libb200tag.so; raises B200TagError (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200TagError(f"{LIB_PATH} not built: run `python -m ros_vision_b200.build` (nvcc, sm_100a). "
                           "This engine has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, sz = C.c_void_p, C.c_int, C.c_size_t
    L.b200tag_default_config.argtypes = [C.POINTER(Config), i32, i32, i32]
    L.b200tag_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.b200tag_create_families.argtypes = [C.POINTER(Config), C.POINTER(Family), i32, C.POINTER(vp)]
    L.b200tag_builtin_family.argtypes = [C.c_char_p]
    L.b200tag_builtin_family.restype = C.POINTER(Family)
    L.b200tag_debug_reconcile.argtypes = [vp, i32]
    L.b200tag_destroy.argtypes = [vp]
    L.b200tag_destroy.restype = None
    L.b200tag_detect.argtypes = [vp, vp]
    L.b200tag_detect_batch.argtypes = [vp, C.POINTER(vp), i32]
    L.b200tag_detect_device.argtypes = [vp, vp, sz, i32]
    L.b200tag_enqueue_device.argtypes = [vp, vp, sz, i32]
    L.b200tag_enqueue_host.argtypes = [vp, C.POINTER(vp), i32]
    L.b200tag_enqueue_host_block.argtypes = [vp, vp, sz, i32]
    L.b200tag_enqueue_mjpg.argtypes = [vp, C.POINTER(vp), C.POINTER(sz), i32]
    L.b200tag_detect_mjpg.argtypes = [vp, C.POINTER(vp), C.POINTER(sz), i32]
    L.b200tag_mjpg_backend.argtypes = [vp]
    L.b200tag_mjpg_parallel_frames.argtypes = [vp, i32]
    L.b200tag_debug_jpeg_model.argtypes = [vp, sz, vp, sz, C.POINTER(i32)]
    L.b200tag_jpeg_probe.argtypes = [vp, sz, C.POINTER(C.c_int32), vp, sz, C.POINTER(sz)]
    L.b200tag_mjpg_backend.restype = C.c_char_p
    L.b200tag_finish.argtypes = [vp]
    L.b200tag_stream.argtypes = [vp]
    L.b200tag_stream.restype = vp
    L.b200tag_detections.argtypes = [vp, i32, C.POINTER(i32)]
    L.b200tag_detections.restype = vp
    L.b200tag_quads.argtypes = [vp, i32, C.POINTER(i32)]
    L.b200tag_quads.restype = vp
    L.b200tag_frame_info_get.argtypes = [vp, i32, C.POINTER(FrameInfo)]
    L.b200tag_copy_stage.argtypes = [vp, i32, i32, vp, sz, C.POINTER(sz)]
    L.b200tag_set_camera.argtypes = [vp] + [C.c_double] * 4
    L.b200tag_set_distortion.argtypes = [vp] + [C.c_double] * 5
    L.b200tag_undistort.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double)] + [C.c_double] * 9
    L.b200tag_alloc_pinned.argtypes = [sz]
    L.b200tag_alloc_pinned.restype = vp
    L.b200tag_alloc_pinned_wc.argtypes = [sz]
    L.b200tag_alloc_pinned_wc.restype = vp
    L.b200tag_free_pinned.argtypes = [vp]
    L.b200tag_free_pinned.restype = None
    L.b200tag_kernels_per_batch.argtypes = [vp]
    L.b200tag_profile_device.argtypes = [vp, vp, sz, i32, i32, C.POINTER(C.c_char_p), C.POINTER(C.c_float), i32,
                                         C.POINTER(i32)]
    L.b200tag_debug_math.argtypes = [i32, vp, vp, vp, i32]
    L.b200tag_error_string.argtypes = [i32]
    L.b200tag_error_string.restype = C.c_char_p
    L.b200tag_last_error.argtypes = [vp]
    L.b200tag_last_error.restype = C.c_char_p
    L.b200tag_estimate_poses.argtypes = [vp, i32] + [C.c_double] * 5 + [vp]
    L.b200tag_locate_tags.argtypes = [vp, i32] + [C.c_double] * 5 + [vp, vp, vp]
    L.b200tag_set_pose_estimation.argtypes = [vp] + [C.c_double] * 5 + [vp, vp]
    L.b200tag_poses.argtypes = [vp, i32, C.POINTER(i32)]
    L.b200tag_poses.restype = vp
    L.b200tag_tag_positions.argtypes = [vp, i32, C.POINTER(i32)]
    L.b200tag_tag_positions.restype = vp
    L.b200tag_debug_estimate_poses_device.argtypes = [vp, i32] + [C.c_double] * 5 + [vp]
    L.b200tag_estimate_poses_ippe.argtypes = [vp, i32] + [C.c_double] * 5 + [vp]
    L.b200tag_debug_estimate_poses_ippe_device.argtypes = [vp, i32] + [C.c_double] * 5 + [vp]
    L.b200tag_set_pose_method.argtypes = [vp, i32]
    L.b200tag_estimate_field_pose.argtypes = [vp, i32, vp, i32] + [C.c_double] * 5 + [vp, vp, vp]
    L.b200tag_debug_estimate_field_pose_device.argtypes = [vp, i32, vp, i32] + [C.c_double] * 5 + [vp, vp, vp]
    L.b200tag_set_field_layout.argtypes = [vp, vp, i32]
    L.b200tag_field_pose_get.argtypes = [vp, i32]
    L.b200tag_field_pose_get.restype = vp
    L.b200tag_undistort_points.argtypes = [vp, i32] + [C.c_double] * 4 + [vp, vp]
    L.b200tag_estimate_poses_distorted.argtypes = [vp, i32, i32] + [C.c_double] * 5 + [vp, vp]
    L.b200tag_debug_estimate_poses_distorted_device.argtypes = [i32, vp, i32] + [C.c_double] * 5 + [vp, vp]
    L.b200tag_estimate_field_pose_distorted.argtypes = [vp, i32, vp, i32] + [C.c_double] * 5 + [vp, vp, vp, vp]
    L.b200tag_debug_estimate_field_pose_distorted_device.argtypes = [vp, i32, vp, i32] + [C.c_double] * 5 + [vp, vp, vp, vp]
    L.b200tag_set_pose_distortion.argtypes = [vp, vp]
    L.b200tag_estimate_pose_covariances.argtypes = [vp, vp, i32] + [C.c_double] * 5 + [vp, C.c_double, vp]
    L.b200tag_debug_pose_covariances_device.argtypes = [vp, vp, i32] + [C.c_double] * 5 + [vp, C.c_double, vp]
    L.b200tag_estimate_field_pose_covariance.argtypes = [vp, i32, vp, i32] + [C.c_double] * 5 + [vp, vp, vp, C.c_double, vp, vp]
    L.b200tag_debug_field_pose_covariance_device.argtypes = [vp, i32, vp, i32] + [C.c_double] * 5 + [vp, vp, vp, C.c_double, vp, vp]
    L.b200tag_set_pose_covariance.argtypes = [vp, C.c_double]
    L.b200tag_pose_covariances.argtypes = [vp, i32, C.POINTER(i32)]
    L.b200tag_pose_covariances.restype = vp
    L.b200tag_field_covariance_get.argtypes = [vp, i32]
    L.b200tag_field_covariance_get.restype = vp
    L.b200tag_estimate_floor_pose.argtypes = [vp, i32, vp, i32] + [C.c_double] * 5 + [vp, vp, vp] + [C.c_double] * 3 + [vp, vp]
    L.b200tag_debug_floor_pose_device.argtypes = L.b200tag_estimate_floor_pose.argtypes
    L.b200tag_set_floor_pose.argtypes = [vp, C.c_double]
    L.b200tag_set_robot_headings.argtypes = [vp, vp, i32]
    L.b200tag_floor_pose_get.argtypes = [vp, i32]
    L.b200tag_floor_pose_get.restype = vp
    L.b200tag_floor_covariance_get.argtypes = [vp, i32]
    L.b200tag_floor_covariance_get.restype = vp
    L.b200tag_version.restype = i32
    _lib = L
    return L


def default_config(width: int, height: int, fmt: str = "yuyv") -> Config:
    cfg = Config()
    rc = load_library().b200tag_default_config(C.byref(cfg), width, height, FMT[fmt])
    if rc:
        raise B200TagError("b200tag_default_config failed")
    return cfg


def jpeg_model_decode(jpeg: bytes, width: int, height: int):
    """Test hook: the host model of the parallel JPEG decode kernels -> (luminance plane, synchronisation rounds)."""
    lib = load_library()
    buf = np.frombuffer(jpeg, dtype=np.uint8)
    out = np.zeros((height, width), dtype=np.uint8)
    rounds = C.c_int32(0)
    rc = lib.b200tag_debug_jpeg_model(buf.ctypes.data_as(C.c_void_p), buf.size, out.ctypes.data_as(C.c_void_p), out.size, C.byref(rounds))
    if rc:
        raise ValueError(f"b200tag_debug_jpeg_model: {rc}")
    return out, rounds.value


def _pose_method(method: str) -> int:
    if method not in POSE_METHODS:
        raise ValueError(f"unknown pose method {method!r}: expected one of {sorted(POSE_METHODS)}")
    return POSE_METHODS[method]


def _distortion(distortion):
    """The `dist` argument of the C ABI: None, or 5 float64 coefficients (k1, k2, p1, p2, k3)."""
    if distortion is None:
        return None
    d = np.ascontiguousarray(distortion, dtype=np.float64).reshape(-1)
    if d.size != 5:
        raise ValueError(f"distortion needs 5 coefficients (k1, k2, p1, p2, k3), got {d.size}")
    return d


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def undistort_points(points, fx: float, fy: float, cx: float, cy: float, distortion) -> np.ndarray:
    """Ideal pinhole pixels of distorted pixels `points` (..., 2) under the 5-coefficient Brown-Conrady model
    `distortion` = (k1, k2, p1, p2, k3) of OpenCV's projectPoints, inverted exactly (b200tag_undistort_points); NaN where
    a point cannot be undistorted (past the fold of a strong barrel model)."""
    lib = load_library()
    pts = np.ascontiguousarray(points, dtype=np.float64)
    flat = pts.reshape(-1, 2)
    out = np.zeros_like(flat)
    rc = lib.b200tag_undistort_points(_ptr(flat) if len(flat) else None, len(flat), float(fx), float(fy), float(cx),
                                      float(cy), _ptr(_distortion(distortion)), _ptr(out) if len(flat) else None)
    if rc:
        raise B200TagError(f"b200tag_undistort_points: {lib.b200tag_error_string(rc).decode()}")
    return out.reshape(pts.shape)


def estimate_poses(detections: np.ndarray, tagsize: float, fx: float, fy: float, cx: float, cy: float,
                   method: str = "oi", distortion=None) -> np.ndarray:
    """estimate_tag_pose for every detection (the node's step after Detect, apriltags_cuda_detector.cu:425-462):
    returns POSE_DT records (R, t in the camera frame, object-space error).  Pure host math in libb200tag.so.
    method="ippe" computes the closed-form IPPE pose instead (b200tag_estimate_poses_ippe, OpenCV's SOLVEPNP_IPPE_SQUARE
    candidates, the one with the smaller object-space error returned).  With `distortion` = (k1, k2, p1, p2, k3) the
    corners are undistorted first (b200tag_estimate_poses_distorted)."""
    lib = load_library()
    m = _pose_method(method)
    dist = _distortion(distortion)
    dets = np.ascontiguousarray(detections, dtype=DETECTION_DT)
    out = np.zeros(len(dets), dtype=POSE_DT)
    if len(dets):
        args = (float(tagsize), float(fx), float(fy), float(cx), float(cy))
        if dist is None:
            fn = {0: "b200tag_estimate_poses", 1: "b200tag_estimate_poses_ippe"}[m]
            rc = getattr(lib, fn)(_ptr(dets), len(dets), *args, _ptr(out))
        else:
            fn = "b200tag_estimate_poses_distorted"
            rc = lib.b200tag_estimate_poses_distorted(_ptr(dets), len(dets), m, *args, _ptr(dist), _ptr(out))
        if rc:
            raise B200TagError(f"{fn}: {lib.b200tag_error_string(rc).decode()}")
    return out


def locate_tags(detections: np.ndarray, tagsize: float, fx: float, fy: float, cx: float, cy: float,
                rotation=None, offset=None) -> np.ndarray:
    """The node's per-frame step behind Detect (apriltags_cuda_detector.cu:421-462,595-599): pose of every detection, tag
    position in the camera frame and -- through the camera's extrinsic `rotation` (3x3) and `offset` (3) -- in the robot
    frame, distance from the camera; TAG_POSITION_DT records, closest first."""
    lib = load_library()
    dets = np.ascontiguousarray(detections, dtype=DETECTION_DT)
    out = np.zeros(len(dets), dtype=TAG_POSITION_DT)
    rot = None if rotation is None else np.ascontiguousarray(rotation, dtype=np.float64).reshape(9)
    off = None if offset is None else np.ascontiguousarray(offset, dtype=np.float64).reshape(3)
    rc = lib.b200tag_locate_tags(dets.ctypes.data_as(C.c_void_p) if len(dets) else None, len(dets), float(tagsize), float(fx),
                                 float(fy), float(cx), float(cy), None if rot is None else rot.ctypes.data_as(C.c_void_p),
                                 None if off is None else off.ctypes.data_as(C.c_void_p),
                                 out.ctypes.data_as(C.c_void_p) if len(dets) else None)
    if rc:
        raise B200TagError(f"b200tag_locate_tags: {lib.b200tag_error_string(rc).decode()}")
    return out


def estimate_poses_device(detections: np.ndarray, tagsize: float, fx: float, fy: float, cx: float, cy: float,
                          method: str = "oi", distortion=None) -> np.ndarray:
    """Test hook: estimate_poses computed by the device pose kernel of `method` (the one GpuDetector.SetPoseEstimation
    enables) on the current CUDA device."""
    lib = load_library()
    m = _pose_method(method)
    dist = _distortion(distortion)
    dets = np.ascontiguousarray(detections, dtype=DETECTION_DT)
    out = np.zeros(len(dets), dtype=POSE_DT)
    args = (_ptr(dets) if len(dets) else None, len(dets), float(tagsize), float(fx), float(fy), float(cx), float(cy))
    if dist is None:
        fn = {0: "b200tag_debug_estimate_poses_device", 1: "b200tag_debug_estimate_poses_ippe_device"}[m]
        rc = getattr(lib, fn)(*args, _ptr(out) if len(dets) else None)
    else:
        fn = "b200tag_debug_estimate_poses_distorted_device"
        rc = lib.b200tag_debug_estimate_poses_distorted_device(m, *args, _ptr(dist), _ptr(out) if len(dets) else None)
    if rc:
        raise B200TagError(f"{fn}: {lib.b200tag_error_string(rc).decode()}")
    return out


def _field_call(fn, fn_distorted, detections, layout, tagsize, fx, fy, cx, cy, rotation, offset, distortion) -> np.ndarray:
    lib = load_library()
    dist = _distortion(distortion)
    dets = np.ascontiguousarray(detections, dtype=DETECTION_DT)
    lay = np.ascontiguousarray(np.zeros(0, dtype=FIELD_TAG_DT) if layout is None else layout, dtype=FIELD_TAG_DT)
    rot = None if rotation is None else np.ascontiguousarray(rotation, dtype=np.float64).reshape(9)
    off = None if offset is None else np.ascontiguousarray(offset, dtype=np.float64).reshape(3)
    out = np.zeros(1, dtype=FIELD_POSE_DT)
    args = [dets.ctypes.data_as(C.c_void_p) if len(dets) else None, len(dets),
            lay.ctypes.data_as(C.c_void_p) if len(lay) else None, len(lay), float(tagsize), float(fx), float(fy),
            float(cx), float(cy)]
    if dist is not None:
        fn = fn_distorted
        args.append(_ptr(dist))
    rc = getattr(lib, fn)(*args, _ptr(rot), _ptr(off), _ptr(out))
    if rc:
        raise B200TagError(f"{fn}: {lib.b200tag_error_string(rc).decode()}")
    return out[0]


def estimate_field_pose(detections: np.ndarray, layout: np.ndarray, tagsize: float, fx: float, fy: float, cx: float,
                        cy: float, rotation=None, offset=None, distortion=None) -> np.ndarray:
    """One camera (and robot) pose in the field from every detection of a layout tag (b200tag_estimate_field_pose): a
    FIELD_POSE_DT record.  `layout` holds FIELD_TAG_DT records (X_field = R X_tag + t); `detections` may be reconciled
    or raw.  rotation / offset are the camera's extrinsics, as for locate_tags.  With `distortion` = (k1, k2, p1, p2,
    k3) the used tags' corners are undistorted first and rms is measured in the ideal image
    (b200tag_estimate_field_pose_distorted).  Pure host math in libb200tag.so."""
    return _field_call("b200tag_estimate_field_pose", "b200tag_estimate_field_pose_distorted", detections, layout, tagsize,
                       fx, fy, cx, cy, rotation, offset, distortion)


def estimate_field_pose_device(detections: np.ndarray, layout: np.ndarray, tagsize: float, fx: float, fy: float,
                               cx: float, cy: float, rotation=None, offset=None, distortion=None) -> np.ndarray:
    """Test hook: estimate_field_pose computed by the device kernel GpuDetector.SetFieldLayout enables."""
    return _field_call("b200tag_debug_estimate_field_pose_device", "b200tag_debug_estimate_field_pose_distorted_device",
                       detections, layout, tagsize, fx, fy, cx, cy, rotation, offset, distortion)


def _pose_covariances(fn, detections, poses, tagsize, fx, fy, cx, cy, sigma, distortion) -> np.ndarray:
    lib = load_library()
    dist = _distortion(distortion)
    dets = np.ascontiguousarray(detections, dtype=DETECTION_DT)
    ps = np.ascontiguousarray(poses, dtype=POSE_DT)
    if len(ps) != len(dets):
        raise ValueError(f"{len(dets)} detections but {len(ps)} poses")
    out = np.zeros(len(dets), dtype=COVARIANCE_DT)
    n = len(dets)
    rc = getattr(lib, fn)(_ptr(dets) if n else None, _ptr(ps) if n else None, n, float(tagsize), float(fx), float(fy),
                          float(cx), float(cy), _ptr(dist), float(sigma), _ptr(out) if n else None)
    if rc:
        raise B200TagError(f"{fn}: {lib.b200tag_error_string(rc).decode()}")
    return out


def estimate_pose_covariances(detections: np.ndarray, poses: np.ndarray, tagsize: float, fx: float, fy: float, cx: float,
                              cy: float, sigma: float, distortion=None) -> np.ndarray:
    """The covariance of every tag pose (b200tag_estimate_pose_covariances): COVARIANCE_DT records parallel to `poses`
    (POSE_DT, from estimate_poses with either method and the same `distortion`).  C is the 6x6 covariance of the pose's
    (rx, ry, rz, tx, ty, tz) in the camera frame for corner noise of `sigma` px per coordinate; all inf on failure."""
    return _pose_covariances("b200tag_estimate_pose_covariances", detections, poses, tagsize, fx, fy, cx, cy, sigma,
                             distortion)


def estimate_pose_covariances_device(detections, poses, tagsize, fx, fy, cx, cy, sigma, distortion=None) -> np.ndarray:
    """Test hook: estimate_pose_covariances computed by the device kernel k_pose_cov."""
    return _pose_covariances("b200tag_debug_pose_covariances_device", detections, poses, tagsize, fx, fy, cx, cy, sigma,
                             distortion)


def _field_covariance_call(fn, detections, layout, tagsize, fx, fy, cx, cy, sigma, rotation, offset, distortion):
    lib = load_library()
    dist = _distortion(distortion)
    dets = np.ascontiguousarray(detections, dtype=DETECTION_DT)
    lay = np.ascontiguousarray(np.zeros(0, dtype=FIELD_TAG_DT) if layout is None else layout, dtype=FIELD_TAG_DT)
    rot = None if rotation is None else np.ascontiguousarray(rotation, dtype=np.float64).reshape(9)
    off = None if offset is None else np.ascontiguousarray(offset, dtype=np.float64).reshape(3)
    pose = np.zeros(1, dtype=FIELD_POSE_DT)
    cov = np.zeros(1, dtype=FIELD_COVARIANCE_DT)
    rc = getattr(lib, fn)(_ptr(dets) if len(dets) else None, len(dets), _ptr(lay) if len(lay) else None, len(lay),
                          float(tagsize), float(fx), float(fy), float(cx), float(cy), _ptr(dist), _ptr(rot), _ptr(off),
                          float(sigma), _ptr(pose), _ptr(cov))
    if rc:
        raise B200TagError(f"{fn}: {lib.b200tag_error_string(rc).decode()}")
    return pose[0], cov[0]


def estimate_field_pose_covariance(detections: np.ndarray, layout: np.ndarray, tagsize: float, fx: float, fy: float,
                                   cx: float, cy: float, sigma: float, rotation=None, offset=None, distortion=None):
    """estimate_field_pose and the covariance of its result (b200tag_estimate_field_pose_covariance): (FIELD_POSE_DT
    record, FIELD_COVARIANCE_DT record).  The pose is bit-identical to estimate_field_pose's; `camera` and `robot` are
    the 6x6 covariances of (rx, ry, rz, tx, ty, tz) of camera_R / camera_t and robot_R / robot_t in the field frame, for
    corner noise of `sigma` px per coordinate.  pose2d_stddevs(cov["robot"]) gives a pose estimator's (x, y, heading)
    standard deviations."""
    return _field_covariance_call("b200tag_estimate_field_pose_covariance", detections, layout, tagsize, fx, fy, cx, cy,
                                  sigma, rotation, offset, distortion)


def estimate_field_pose_covariance_device(detections, layout, tagsize, fx, fy, cx, cy, sigma, rotation=None, offset=None,
                                          distortion=None):
    """Test hook: estimate_field_pose_covariance computed by k_field_pose's variant with the covariance."""
    return _field_covariance_call("b200tag_debug_field_pose_covariance_device", detections, layout, tagsize, fx, fy, cx,
                                  cy, sigma, rotation, offset, distortion)


def _floor_call(fn, detections, layout, tagsize, fx, fy, cx, cy, rotation, offset, heading, heading_weight, distortion,
                sigma):
    lib = load_library()
    dist = _distortion(distortion)
    dets = np.ascontiguousarray(detections, dtype=DETECTION_DT)
    lay = np.ascontiguousarray(np.zeros(0, dtype=FIELD_TAG_DT) if layout is None else layout, dtype=FIELD_TAG_DT)
    rot = None if rotation is None else np.ascontiguousarray(rotation, dtype=np.float64).reshape(9)
    off = None if offset is None else np.ascontiguousarray(offset, dtype=np.float64).reshape(3)
    out = np.zeros(1, dtype=FLOOR_POSE_DT)
    cov = np.zeros((3, 3), dtype=np.float64)
    rc = getattr(lib, fn)(_ptr(dets) if len(dets) else None, len(dets), _ptr(lay) if len(lay) else None, len(lay),
                          float(tagsize), float(fx), float(fy), float(cx), float(cy), _ptr(dist), _ptr(rot), _ptr(off),
                          float(heading), float(heading_weight), float(sigma), _ptr(out), _ptr(cov) if sigma > 0 else None)
    if rc:
        raise B200TagError(f"{fn}: {lib.b200tag_error_string(rc).decode()}")
    return out[0], (cov if sigma > 0 else None)


def estimate_floor_pose(detections: np.ndarray, layout: np.ndarray, tagsize: float, fx: float, fy: float, cx: float,
                        cy: float, rotation=None, offset=None, heading=float("nan"), heading_weight=float("inf"),
                        distortion=None, sigma=0.0):
    """The robot's (x, y, heading) on a flat floor (b200tag_estimate_floor_pose): (FLOOR_POSE_DT record, 3x3 covariance
    of (x, y, heading) in the field frame or None when sigma is 0).  Correspondences as estimate_field_pose; rotation /
    offset are the camera's extrinsics with the robot frame's origin on the floor.  `heading` (rad, counter-clockwise
    from field +x) is the gyro's: NaN solves for it (free), a finite heading with heading_weight = inf fixes it, and
    with 0 < heading_weight < inf adds it as a prior of heading_weight px per unit of 2 tan(delta / 2) (corner noise
    over gyro noise in rad).  Pure host math in libb200tag.so."""
    return _floor_call("b200tag_estimate_floor_pose", detections, layout, tagsize, fx, fy, cx, cy, rotation, offset,
                       heading, heading_weight, distortion, sigma)


def estimate_floor_pose_device(detections: np.ndarray, layout: np.ndarray, tagsize: float, fx: float, fy: float,
                               cx: float, cy: float, rotation=None, offset=None, heading=float("nan"),
                               heading_weight=float("inf"), distortion=None, sigma=0.0):
    """Test hook: estimate_floor_pose computed by the device kernels GpuDetector.SetFloorPose enables."""
    return _floor_call("b200tag_debug_floor_pose_device", detections, layout, tagsize, fx, fy, cx, cy, rotation, offset,
                       heading, heading_weight, distortion, sigma)


def pose2d_stddevs(cov) -> tuple:
    """(sigma_x, sigma_y, sigma_yaw) of a robot Pose2d, in m, m and rad, as WPILib's addVisionMeasurement takes them:
    from a 6x6 field-frame pose covariance (e.g. the `robot` field of FIELD_COVARIANCE_DT) sqrt(C[3][3]),
    sqrt(C[4][4]) and sqrt(C[2][2]); from the 3x3 (x, y, heading) covariance of a floor pose the square roots of its
    diagonal."""
    C = np.asarray(cov, dtype=np.float64)
    if C.size == 9:
        C3 = C.reshape(3, 3)
        return float(np.sqrt(C3[0, 0])), float(np.sqrt(C3[1, 1])), float(np.sqrt(C3[2, 2]))
    C6 = C.reshape(6, 6)
    return float(np.sqrt(C6[3, 3])), float(np.sqrt(C6[4, 4])), float(np.sqrt(C6[2, 2]))


def _records(ptr, n, dtype) -> np.ndarray:
    if not ptr or n == 0:
        return np.zeros((0,), dtype=dtype)
    buf = (C.c_char * (dtype.itemsize * n)).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype, count=n).copy()


class PinnedBuffer:
    """Page-locked host staging memory (numpy view), for the host->device leg of Detect."""

    def __init__(self, nbytes: int, write_combined: bool = False):
        self._lib = load_library()
        self.ptr = (self._lib.b200tag_alloc_pinned_wc if write_combined else self._lib.b200tag_alloc_pinned)(nbytes)
        if not self.ptr:
            raise B200TagError("b200tag_alloc_pinned failed")
        self.nbytes = nbytes
        self.array = np.frombuffer((C.c_uint8 * nbytes).from_address(self.ptr), dtype=np.uint8)

    def close(self):
        if self.ptr:
            self.array = None
            self._lib.b200tag_free_pinned(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GpuDetector:
    """Mirror of frc971::apriltag::GpuDetector.

    GpuDetector(width, height, tag_detector..., camera_matrix, distortion_coefficients)
    (apriltag_gpu.h:84-85): the apriltag_detector_t fields the reference reads are keyword
    arguments here (quad_decimate, quad_sigma, refine_edges, qtp fields).
    """

    def __init__(self, width, height, fmt="yuyv", quad_decimate=2, quad_sigma=0.0, refine_edges=True,
                 camera_matrix=None, distortion_coefficients=None, max_batch=1, device=-1, keep_stages=False,
                 max_points=0, max_blobs=0, max_detections=0, test_flags=0, families=("tag36h11",), **qtp):
        self._lib = load_library()
        cfg = default_config(width, height, fmt)
        cfg.quad_decimate = int(quad_decimate)
        cfg.quad_sigma = float(quad_sigma)
        cfg.refine_edges = int(bool(refine_edges))
        cfg.max_batch = int(max_batch)
        cfg.device = int(device)
        cfg.keep_stages = int(bool(keep_stages))
        cfg.test_flags = int(test_flags)
        cfg.max_points, cfg.max_blobs, cfg.max_detections = int(max_points), int(max_blobs), int(max_detections)
        if camera_matrix is not None:
            cfg.fx, cfg.cx, cfg.fy, cfg.cy = camera_matrix  # CameraMatrix field order, apriltag_gpu.h:61-66
        if distortion_coefficients is not None:
            cfg.k1, cfg.k2, cfg.p1, cfg.p2, cfg.k3 = distortion_coefficients
        for k, v in qtp.items():
            if not hasattr(cfg, k):
                raise TypeError(f"unknown detector parameter {k!r}")
            setattr(cfg, k, v)
        self.cfg = cfg
        self.width, self.height, self.fmt = width, height, fmt
        self.frame_bytes = width * height * BYTES_PER_PIXEL[fmt]
        self.max_batch = int(max_batch)
        h = C.c_void_p()
        # tag families (apriltag_detector_add_family): names of built-in tables or dicts in the layout of
        # ros_vision_b200.tag_families.FAMILIES entries (+ optional "reversed_border", "max_hamming", "name")
        if isinstance(families, (str, dict)):
            families = [families]
        self.families = list(families)
        fams = (Family * len(self.families))()
        keep = []
        for i, f in enumerate(self.families):
            if isinstance(f, str):
                b = self._lib.b200tag_builtin_family(f.encode())
                if not b:
                    raise ValueError(f"no built-in tag family {f!r}")
                fams[i] = b.contents
            else:
                codes = (C.c_uint64 * len(f["codes"]))(*f["codes"])
                bx = (C.c_uint32 * f["nbits"])(*[v & 0xffffffff for v in f["bit_x"]])
                by = (C.c_uint32 * f["nbits"])(*[v & 0xffffffff for v in f["bit_y"]])
                keep.append((codes, bx, by))
                fams[i] = Family(f.get("name", "custom").encode(), f["nbits"], len(f["codes"]), codes, bx, by, f["width_at_border"],
                                 f["total_width"], int(f.get("reversed_border", 0)), int(f.get("max_hamming", 2)))
        rc = self._lib.b200tag_create_families(C.byref(cfg), fams, len(self.families), C.byref(h))
        if rc:
            msg = self._lib.b200tag_last_error(None).decode()
            raise B200TagError(f"b200tag_create: {self._lib.b200tag_error_string(rc).decode()}: {msg}")
        self._h = h
        self.last_count = 0

    # -- lifecycle -----------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.b200tag_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what, allow_overflow=False):
        if rc == 0 or (allow_overflow and rc == -4):
            return rc
        raise B200TagError(f"{what}: {self._lib.b200tag_error_string(rc).decode()}: "
                           f"{self._lib.b200tag_last_error(self._h).decode()}")

    # -- detection -----------------------------------------------------------------------------
    def Detect(self, image) -> None:
        """GpuDetector::Detect(const uint8_t*): one host frame, synchronous (apriltag_gpu.h:89)."""
        self.DetectBatch([image])

    def DetectBatch(self, images, allow_overflow=False) -> int:
        arrs = [np.ascontiguousarray(im, dtype=np.uint8) for im in images]
        for a in arrs:
            if a.size != self.frame_bytes:
                raise ValueError(f"frame has {a.size} bytes, expected {self.frame_bytes}")
        ptrs = (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
        rc = self._lib.b200tag_detect_batch(self._h, ptrs, len(arrs))
        self.last_count = len(arrs)
        return self._check(rc, "b200tag_detect_batch", allow_overflow)

    def DetectPointers(self, host_ptrs, allow_overflow=False) -> int:
        """Same as DetectBatch for raw host addresses (e.g. PinnedBuffer.ptr)."""
        ptrs = (C.c_void_p * len(host_ptrs))(*host_ptrs)
        rc = self._lib.b200tag_detect_batch(self._h, ptrs, len(host_ptrs))
        self.last_count = len(host_ptrs)
        return self._check(rc, "b200tag_detect_batch", allow_overflow)

    def EnqueuePointers(self, host_ptrs) -> None:
        ptrs = (C.c_void_p * len(host_ptrs))(*host_ptrs)
        self._check(self._lib.b200tag_enqueue_host(self._h, ptrs, len(host_ptrs)), "b200tag_enqueue_host")
        self.last_count = len(host_ptrs)

    def EnqueueHostBlock(self, host_ptr: int, count: int, stride: int = 0) -> None:
        """`count` frames of one host allocation (pinned ring buffer), one host->device copy."""
        self._check(self._lib.b200tag_enqueue_host_block(self._h, C.c_void_p(host_ptr), stride, count),
                    "b200tag_enqueue_host_block")
        self.last_count = count

    def EnqueueMjpg(self, jpegs) -> None:
        """Camera wire format: `jpegs` = JPEG bitstreams (bytes / uint8 arrays) of width x height; nvJPEG decodes their
        luminance planes on the detector's stream and the gray pipeline runs behind it (detector created with fmt="gray")."""
        arrs = [np.frombuffer(j, dtype=np.uint8) if isinstance(j, (bytes, bytearray, memoryview)) else np.ascontiguousarray(j, dtype=np.uint8)
                for j in jpegs]
        ptrs = (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
        sizes = (C.c_size_t * len(arrs))(*[a.size for a in arrs])
        self._mjpg_keep = (arrs, ptrs, sizes)  # the bitstreams stay alive until Finish
        self._check(self._lib.b200tag_enqueue_mjpg(self._h, ptrs, sizes, len(arrs)), "b200tag_enqueue_mjpg")
        self.last_count = len(arrs)

    def DetectMjpg(self, jpegs, allow_overflow=False) -> int:
        self.EnqueueMjpg(jpegs)
        return self.Finish(allow_overflow)

    def MjpgParallelFrames(self) -> int:
        """Frames of the last MJPG batch decoded by the parallel kernels (the rest took the sequential kernel)."""
        return int(self._lib.b200tag_mjpg_parallel_frames(self._h, self.last_count))

    @property
    def mjpg_backend(self) -> str:
        return (self._lib.b200tag_mjpg_backend(self._h) or b"").decode()

    def DetectDevice(self, device_ptr: int, count: int = 1, stride: int = 0, allow_overflow=False) -> int:
        rc = self._lib.b200tag_detect_device(self._h, C.c_void_p(device_ptr), stride, count)
        self.last_count = count
        return self._check(rc, "b200tag_detect_device", allow_overflow)

    def EnqueueDevice(self, device_ptr: int, count: int = 1, stride: int = 0) -> None:
        self._check(self._lib.b200tag_enqueue_device(self._h, C.c_void_p(device_ptr), stride, count),
                    "b200tag_enqueue_device")
        self.last_count = count

    def Finish(self, allow_overflow=False) -> int:
        return self._check(self._lib.b200tag_finish(self._h), "b200tag_finish", allow_overflow)

    @property
    def stream(self) -> int:
        return int(self._lib.b200tag_stream(self._h) or 0)

    # -- results -------------------------------------------------------------------------------
    def Detections(self, frame: int = 0) -> np.ndarray:
        """GpuDetector::Detections(): reconciled detections sorted by id (apriltag_gpu.h:93)."""
        n = C.c_int()
        p = self._lib.b200tag_detections(self._h, frame, C.byref(n))
        if not p or n.value == 0:
            return np.zeros((0,), dtype=DETECTION_DT)
        buf = (C.c_char * (DETECTION_DT.itemsize * n.value)).from_address(p)
        return np.frombuffer(buf, dtype=DETECTION_DT, count=n.value).copy()

    def FitQuads(self, frame: int = 0) -> np.ndarray:
        """GpuDetector::FitQuads(): QuadCorners of the last frame (apriltag_gpu.h:91)."""
        n = C.c_int()
        p = self._lib.b200tag_quads(self._h, frame, C.byref(n))
        if not p or n.value == 0:
            return np.zeros((0,), dtype=QUAD_DT)
        buf = (C.c_char * (QUAD_DT.itemsize * n.value)).from_address(p)
        return np.frombuffer(buf, dtype=QUAD_DT, count=n.value).copy()

    def SetPoseEstimation(self, tagsize, fx, fy, cx, cy, rotation=None, offset=None, method="oi", distortion=None) -> None:
        """The node's pose step on the GPU: from the next Detect on, a kernel at the end of the detection graph estimates
        every detection's pose (Poses) and its robot-frame record (TagPositions), with the arguments of locate_tags.
        tagsize = 0 turns it off.  method="ippe" runs the closed-form IPPE pose (estimate_poses(..., method="ippe"))
        instead of libapriltag's orthogonal iteration.  `distortion` = (k1, k2, p1, p2, k3) undistorts the corners
        before the pose and field pose steps, as estimate_poses(..., distortion=...) does; None turns that off."""
        m = _pose_method(method)
        dist = _distortion(distortion)
        rot = None if rotation is None else np.ascontiguousarray(rotation, dtype=np.float64).reshape(9)
        off = None if offset is None else np.ascontiguousarray(offset, dtype=np.float64).reshape(3)
        self._check(self._lib.b200tag_set_pose_estimation(self._h, float(tagsize), float(fx), float(fy), float(cx), float(cy),
                                                          None if rot is None else rot.ctypes.data_as(C.c_void_p),
                                                          None if off is None else off.ctypes.data_as(C.c_void_p)),
                    "b200tag_set_pose_estimation")
        self._check(self._lib.b200tag_set_pose_method(self._h, m), "b200tag_set_pose_method")
        self._check(self._lib.b200tag_set_pose_distortion(self._h, _ptr(dist)), "b200tag_set_pose_distortion")

    def Poses(self, frame: int = 0) -> np.ndarray:
        """POSE_DT records parallel to Detections(frame); empty when the last call ran without the pose step."""
        n = C.c_int()
        return _records(self._lib.b200tag_poses(self._h, frame, C.byref(n)), n.value, POSE_DT)

    def TagPositions(self, frame: int = 0) -> np.ndarray:
        """TAG_POSITION_DT records of frame `frame`, closest first, as locate_tags(Detections(frame), ...) returns them."""
        n = C.c_int()
        return _records(self._lib.b200tag_tag_positions(self._h, frame, C.byref(n)), n.value, TAG_POSITION_DT)

    def SetPoseCovariance(self, sigma: float) -> None:
        """From the next Detect on, the covariance of every pose (PoseCovariances) and of the field pose
        (FieldCovariance) for corner noise of `sigma` px per coordinate, as estimate_pose_covariances and
        estimate_field_pose_covariance compute them.  0 turns it off."""
        self._check(self._lib.b200tag_set_pose_covariance(self._h, float(sigma)), "b200tag_set_pose_covariance")

    def PoseCovariances(self, frame: int = 0) -> np.ndarray:
        """COVARIANCE_DT records parallel to Poses(frame); empty when the last call ran without the covariance."""
        n = C.c_int()
        return _records(self._lib.b200tag_pose_covariances(self._h, frame, C.byref(n)), n.value, COVARIANCE_DT)

    def FieldCovariance(self, frame: int = 0):
        """The FIELD_COVARIANCE_DT record of FieldPose(frame); None when the last call ran without it."""
        p = self._lib.b200tag_field_covariance_get(self._h, frame)
        return None if not p else _records(p, 1, FIELD_COVARIANCE_DT)[0]

    def SetFieldLayout(self, layout) -> None:
        """From the next Detect on, while the pose step is on, one field pose per frame from every visible tag of
        `layout` (FIELD_TAG_DT records, e.g. field_layout.from_wpilib), with SetPoseEstimation's tagsize, intrinsics and
        extrinsics (FieldPose).  None or an empty layout turns it off."""
        lay = np.ascontiguousarray(np.zeros(0, dtype=FIELD_TAG_DT) if layout is None else layout, dtype=FIELD_TAG_DT)
        self._check(self._lib.b200tag_set_field_layout(self._h, lay.ctypes.data_as(C.c_void_p) if len(lay) else None,
                                                       len(lay)), "b200tag_set_field_layout")

    def FieldPose(self, frame: int = 0):
        """The FIELD_POSE_DT record of frame `frame`, as estimate_field_pose(Detections(frame), ...) returns it; None when
        the last call ran without the field step."""
        p = self._lib.b200tag_field_pose_get(self._h, frame)
        return None if not p else _records(p, 1, FIELD_POSE_DT)[0]

    def SetFloorPose(self, heading_weight) -> None:
        """From the next Detect on, whenever the field step runs, the robot's floor pose per frame (FloorPose) with
        estimate_floor_pose's model, from the field step's corners.  heading_weight > 0 (inf: the gyro heading is
        fixed) turns it on, 0 off; SetPoseCovariance's sigma adds FloorCovariance."""
        self._check(self._lib.b200tag_set_floor_pose(self._h, float(heading_weight)), "b200tag_set_floor_pose")

    def SetRobotHeadings(self, headings) -> None:
        """Gyro headings (rad) for the next Detect / Enqueue call only, one per frame; frames past the list or NaN run
        in free mode, and so does every frame of a call without a preceding SetRobotHeadings."""
        h = np.ascontiguousarray(np.zeros(0) if headings is None else headings, dtype=np.float64).reshape(-1)
        self._check(self._lib.b200tag_set_robot_headings(self._h, _ptr(h) if len(h) else None, len(h)),
                    "b200tag_set_robot_headings")

    def FloorPose(self, frame: int = 0):
        """The FLOOR_POSE_DT record of frame `frame`, as estimate_floor_pose(Detections(frame), ...) returns it; None
        when the last call ran without the floor step."""
        p = self._lib.b200tag_floor_pose_get(self._h, frame)
        return None if not p else _records(p, 1, FLOOR_POSE_DT)[0]

    def FloorCovariance(self, frame: int = 0):
        """The 3x3 covariance of FloorPose(frame)'s (x, y, heading); None when the last call ran without it."""
        p = self._lib.b200tag_floor_covariance_get(self._h, frame)
        return None if not p else np.frombuffer((C.c_char * 72).from_address(p), dtype=np.float64).reshape(3, 3).copy()

    def ReinitializeDetections(self) -> None:
        """apriltag_gpu.cu:202-220 frees and re-creates the zarray; results here are plain arrays."""

    def FrameInfo(self, frame: int = 0) -> FrameInfo:
        info = FrameInfo()
        self._check(self._lib.b200tag_frame_info_get(self._h, frame, C.byref(info)), "b200tag_frame_info_get")
        return info

    def CopyStage(self, stage: int, frame: int = 0) -> np.ndarray:
        nbytes = C.c_size_t()
        self._check(self._lib.b200tag_copy_stage(self._h, frame, stage, None, 0, C.byref(nbytes)), "b200tag_copy_stage")
        dt = np.dtype(_STAGE_DTYPES[stage])
        out = np.zeros((nbytes.value // dt.itemsize,), dtype=dt)
        if nbytes.value:
            self._check(self._lib.b200tag_copy_stage(self._h, frame, stage, out.ctypes.data_as(C.c_void_p), out.nbytes,
                                                     C.byref(nbytes)), "b200tag_copy_stage")
        return out

    # the reference's debug accessors, apriltag_gpu.h:98-183
    def CopyGrayTo(self, frame=0):
        return self.CopyStage(STAGE_GRAY, frame).reshape(self.height, self.width)

    def CopyDecimatedTo(self, frame=0):
        f = self.cfg.quad_decimate
        return self.CopyStage(STAGE_QUAD_IMAGE, frame).reshape(self.height // f, self.width // f)

    def CopyThresholdedTo(self, frame=0):
        f = self.cfg.quad_decimate
        return self.CopyStage(STAGE_THRESHOLD, frame).reshape(self.height // f, self.width // f)

    def CopyUnionMarkersTo(self, frame=0):
        return self.CopyStage(STAGE_LABELS, frame)

    def CopyUnionMarkersSizeTo(self, frame=0):
        return self.CopyStage(STAGE_SIZES, frame)

    def SetCameraMatrix(self, fx, cx, fy, cy):
        self._check(self._lib.b200tag_set_camera(self._h, fx, cx, fy, cy), "b200tag_set_camera")

    def SetDistortionCoefficients(self, k1, k2, p1, p2, k3):
        self._check(self._lib.b200tag_set_distortion(self._h, k1, k2, p1, p2, k3), "b200tag_set_distortion")

    @staticmethod
    def UnDistort(u, v, camera_matrix, distortion_coefficients):
        """GpuDetector::UnDistort (apriltag_gpu.h:199-200). Returns (u, v, converged)."""
        cu, cv = C.c_double(u), C.c_double(v)
        ok = load_library().b200tag_undistort(C.byref(cu), C.byref(cv), *camera_matrix, *distortion_coefficients)
        return cu.value, cv.value, bool(ok)

    # -- measurement helpers -------------------------------------------------------------------
    def kernels_per_batch(self) -> int:
        return int(self._lib.b200tag_kernels_per_batch(self._h))

    def ProfileDevice(self, device_ptr: int, count: int, iters: int = 5, stride: int = 0):
        cap = 64
        names = (C.c_char_p * cap)()
        ms = (C.c_float * cap)()
        n = C.c_int()
        self._check(self._lib.b200tag_profile_device(self._h, C.c_void_p(device_ptr), stride, count, iters, names, ms,
                                                     cap, C.byref(n)), "b200tag_profile_device")
        self.last_count = count
        return [(names[i].decode(), float(ms[i])) for i in range(min(n.value, cap))]
