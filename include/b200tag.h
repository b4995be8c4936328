/*
 * b200tag -- C ABI of the B200-native AprilTag detection engine.
 *
 * This is the drop-in boundary for the hot path of Team766/ros_vision's
 * `apriltags_cuda` package: everything frc971::apriltag::GpuDetector does per
 * frame (reference: src/apriltags_cuda/include/apriltags_cuda/apriltag_gpu.h:77-359,
 * src/apriltags_cuda/src/apriltag_gpu.cu:725-1166, src/apriltags_cuda/src/apriltag_detect.cu).
 * The C++ class with the reference's own name and members is layered on these
 * entry points in include/apriltags_cuda/apriltag_gpu.h; INTEGRATION.md shows how
 * the ROS 2 node links it.
 *
 * Plain C types only: pointers, sizes, PODs.  All functions return 0 on success
 * or a negative B200TAG_E_* code; b200tag_error_string() describes it.  There is
 * no CPU fallback: without a CUDA device b200tag_create fails with
 * B200TAG_E_NO_DEVICE.
 */
#ifndef B200TAG_H_
#define B200TAG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200TAG_ABI_VERSION 2

/* Input pixel formats.  The reference accepts YUYV only (apriltag_gpu.h:89); the
 * node converts bgr8 -> YUYV on the CPU first (apriltags_cuda_detector.cu:399-401),
 * which B200TAG_FMT_BGR8 makes unnecessary. */
enum { B200TAG_FMT_GRAY8 = 0, B200TAG_FMT_YUYV = 1, B200TAG_FMT_BGR8 = 2 };

enum {
  B200TAG_OK = 0,
  B200TAG_E_INVALID = -1,    /* bad argument / unsupported configuration */
  B200TAG_E_NO_DEVICE = -2,  /* no usable CUDA device */
  B200TAG_E_CUDA = -3,       /* a CUDA call failed (see b200tag_last_error) */
  B200TAG_E_OVERFLOW = -4,   /* a fixed-capacity device buffer overflowed on this frame */
  B200TAG_E_NOMEM = -5,
};

/* Bits of b200tag_frame_info.status (non-zero => results for that frame are incomplete). */
enum {
  B200TAG_ST_POINTS_OVERFLOW = 1u << 0,
  B200TAG_ST_HASH_OVERFLOW = 1u << 1,
  B200TAG_ST_BLOBS_OVERFLOW = 1u << 2,
  B200TAG_ST_QUADS_OVERFLOW = 1u << 3,
  B200TAG_ST_DETS_OVERFLOW = 1u << 4,
  B200TAG_ST_JPEG_TRUNCATED = 1u << 5, /* MJPG input: the bitstream does not end with an EOI marker (a cut-off frame: the
                                          missing part of the image decodes as flat gray).  Does not fail the call. */
};

/* b200tag_config.test_flags: results must be identical with and without them. */
enum {
  B200TAG_TEST_DIRECT_HASH = 1,   /* k_boundary: every point bypasses the CTA-local blob-pair table */
  B200TAG_TEST_BITONIC_SORT = 2,  /* fit kernels: angle sort by the bitonic network instead of the bucket sort */
  B200TAG_TEST_SMALL_CHUNKS = 4,  /* k_boundary: a tile's points go through the blob-pair grouping 96 at a time (the path of
                                     tiles with more than two points per pixel) */
};

/* Mirrors the fields of apriltag_detector_t / apriltag_quad_thresh_params that the
 * reference reads (apriltag_gpu.cu:166-181,737,884,1084-1086; apriltag_detect.cu:229,
 * 244,455,580) plus CameraMatrix / DistCoeffs (apriltag_gpu.h:61-74). */
typedef struct b200tag_config {
  int32_t abi_version;    /* B200TAG_ABI_VERSION */
  int32_t width, height;  /* full-resolution frame; width/quad_decimate and height/quad_decimate
                             must be multiples of 4 (the reference requires W%8==0, H%8==0 at decimate 2) */
  int32_t format;         /* B200TAG_FMT_* */
  int32_t quad_decimate;  /* integer >= 1 (the reference: exactly 2, apriltag_gpu.cu:166) */
  float quad_sigma;       /* Gaussian blur of the quad image; 0 = off (ignored by the reference) */
  int32_t refine_edges;
  double decode_sharpening;
  int32_t min_cluster_pixels;
  int32_t max_nmaxima;    /* must be 10 (line_fit_filter.cu:1205) */
  float cos_critical_rad;
  float max_line_fit_mse;
  int32_t min_white_black_diff;
  double fx, cx, fy, cy;      /* CameraMatrix */
  double k1, k2, p1, p2, k3;  /* DistCoeffs */
  int32_t max_batch;      /* frames per call that buffers are sized for (>= 1) */
  int32_t device;         /* CUDA device ordinal, -1 = current device */
  int32_t keep_stages;    /* 1 = also keep debug-only stage arrays (filtered min/max, fit quads) */
  uint32_t max_points;    /* capacity of the boundary-point list per frame; 0 = default (2 * quad pixels) */
  uint32_t max_blobs;     /* capacity of the candidate-blob list per frame; 0 = default */
  uint32_t max_detections;/* per frame; 0 = default (256) */
  int32_t test_flags;     /* B200TAG_TEST_*: force the rarely taken fallback paths (tests only), 0 in production */
  int32_t reserved[7];
} b200tag_config;

/* apriltag_detection_t (libapriltag apriltag.h) flattened: id, hamming, decision_margin,
 * H (row-major 3x3), centre, corners. */
typedef struct b200tag_detection {
  int32_t id;
  int32_t hamming;
  float decision_margin;
  int32_t frame;  /* index within the batch */
  int32_t family; /* index into the families the detector was created with (apriltag_detection_t.family) */
  int32_t reserved;
  double H[9];
  double c[2];
  double p[4][2];
} b200tag_detection;

/* frc971::apriltag::QuadCorners (apriltag_gpu.h:55-59). */
typedef struct b200tag_quad {
  float corners[4][2];
  int32_t reversed_border;
  uint32_t blob_index;
  uint32_t rep0, rep1; /* the two component labels bounding the blob */
} b200tag_quad;

typedef struct b200tag_frame_info {
  uint32_t status; /* B200TAG_ST_* */
  uint32_t num_points;
  uint32_t num_clusters;
  uint32_t num_blobs;
  uint32_t num_selected_points;
  uint32_t num_fit_quads;
  uint32_t num_quads;
  uint32_t num_detections; /* before host-side reconcile */
} b200tag_frame_info;

/* Stage selectors for b200tag_copy_stage: the reference's Copy*To debug accessors
 * (apriltag_gpu.h:98-183), generalised. */
enum {
  B200TAG_STAGE_GRAY = 0,        /* uint8[W*H]                      CopyGrayTo (GRAY8 detectors: host / JPEG frames only) */
  B200TAG_STAGE_QUAD_IMAGE = 1,  /* uint8[w*h]                      CopyDecimatedTo */
  B200TAG_STAGE_THRESHOLD = 2,   /* uint8[w*h]                      CopyThresholdedTo */
  B200TAG_STAGE_LABELS = 3,      /* uint32[w*h]                     CopyUnionMarkersTo */
  B200TAG_STAGE_SIZES = 4,       /* uint32[w*h]                     CopyUnionMarkersSizeTo */
  B200TAG_STAGE_POINTS = 5,      /* b200tag_point[num_points]       CopyCompressedUnionMarkerPairTo */
  B200TAG_STAGE_BLOBS = 6,       /* b200tag_blob[candidates]: every blob pair within the point-count limits;
                                    .selected tells whether it also passed SelectBlobs      CopySelectedExtents */
  B200TAG_STAGE_SORTED_POINTS = 7,/* uint64[...] indexed by b200tag_blob.offset             CopySortedSelectedBlobs */
  B200TAG_STAGE_LINE_FIT_POINTS = 8, /* b200tag_lfp[...]            CopyLineFitPoints */
  B200TAG_STAGE_ERRORS = 9,      /* float[num_selected_points]      CopyErrors */
  B200TAG_STAGE_FILTERED_ERRORS = 10, /* double[...]                CopyFilteredErrors */
  B200TAG_STAGE_FIT_QUADS = 11,  /* b200tag_fit_quad[num_fit_quads] CopyFitQuads */
  B200TAG_STAGE_QUADS = 12,      /* b200tag_quad[num_quads]         FitQuads() */
  B200TAG_STAGE_RAW_DETECTIONS = 13, /* b200tag_detection[num_detections] before reconcile */
  B200TAG_STAGE_MINMAX = 14,     /* uint8[(w/4)*(h/4)*2] filtered tile min,max */
  B200TAG_STAGE_CLUSTERS = 15,   /* b200tag_blob[num_clusters] every blob pair, selected or not (keep_stages) */
};

typedef struct b200tag_point { /* one boundary point; QuadBoundaryPoint (points.h:25-161) unpacked */
  uint32_t slot;  /* cluster slot (engine-internal id of the blob pair) */
  uint16_t x, y;  /* half-pixel coordinates 2*base + d */
  uint8_t dir, black_to_white, pad[2];
} b200tag_point;

typedef struct b200tag_blob { /* MinMaxExtents (line_fit_filter.h:14-59) + selection */
  uint32_t rep0, rep1;
  uint32_t min_x, min_y, max_x, max_y;
  uint32_t count;
  uint32_t offset; /* first point of this blob in the sorted-point arrays (candidate blobs) */
  int32_t gx_sum, gy_sum;
  int64_t pxgx_plus_pygy_sum;
  uint32_t slot;
  int32_t selected;
} b200tag_blob;

typedef struct b200tag_lfp { /* LineFitPoint (line_fit_filter.h:61-83), inclusive per-blob prefix sums */
  int64_t Mxx, Myy, Mxy, Mx, My, W;
} b200tag_lfp;

typedef struct b200tag_moments { /* LineFitMoments (line_fit_filter.h:85-94) */
  int64_t Mx, My, W, Mxx, Myy, Mxy;
  int32_t N, pad;
} b200tag_moments;

typedef struct b200tag_fit_quad { /* FitQuad (line_fit_filter.h:130-135) */
  uint32_t blob_index;
  int32_t valid;
  int32_t num_peaks;
  uint32_t indices[4];
  uint32_t pad;
  b200tag_moments moments[4];
  double err;
} b200tag_fit_quad;

typedef struct b200tag_detector b200tag_detector;

/* A tag family: the fields of libapriltag's apriltag_family_t that detection reads (apriltag_gpu.cu:169-177 for
 * width_at_border / reversed_border; quad_decode_index for the rest).  The reference accepts the eight families of
 * apriltag_utils.cu:10-27; here any family of at most 64 bits and total_width <= 12 is accepted, several at once as
 * long as they share one border polarity (the reference's own precondition, apriltag_detect.cu:108).  bit_x / bit_y
 * are apriltag_family_t's uint32_t arrays (negative coordinates of the tagStandard / tagCircle families wrap, as in
 * libapriltag).  The arrays are copied by b200tag_create_families. */
typedef struct b200tag_family {
  const char *name;
  uint32_t nbits, ncodes;
  const uint64_t *codes;
  const uint32_t *bit_x, *bit_y;
  int32_t width_at_border, total_width;
  int32_t reversed_border;
  int32_t max_hamming; /* bits corrected (apriltag_detector_add_family_bits; the node's add_family uses 2), 0..3 */
} b200tag_family;

/* Built-in tables: "tag36h11", "tag25h9", "tag16h5" (AprilTag 3 layouts, max_hamming 2); NULL for other names. */
const b200tag_family *b200tag_builtin_family(const char *name);

/* Fills `cfg` with libapriltag's apriltag_detector_create() defaults as the node sets them
 * (apriltags_cuda_detector.cu:142-147): decimate 2, sigma 0, refine_edges on. */
int b200tag_default_config(b200tag_config *cfg, int width, int height, int format);

/* GpuDetector::GpuDetector (apriltag_gpu.cu:111-188): allocates every device buffer up front. */
int b200tag_create(const b200tag_config *cfg, b200tag_detector **out);
/* The same with the caller's tag families (apriltag_detector_add_family, apriltags_cuda_detector.cu:139-140);
 * b200tag_create == one family, the built-in tag36h11 the node configures.  B200TAG_E_INVALID for an empty list, more
 * than 8 families, mixed border polarities or a family outside the limits above. */
int b200tag_create_families(const b200tag_config *cfg, const b200tag_family *families, int nfamilies, b200tag_detector **out);
/* GpuDetector::~GpuDetector (apriltag_gpu.cu:190-200). */
void b200tag_destroy(b200tag_detector *det);

/* GpuDetector::Detect (apriltag_gpu.cu:725): `host_image` is one tightly packed frame in
 * cfg.format (pageable or pinned); returns with detections ready. */
int b200tag_detect(b200tag_detector *det, const uint8_t *host_image);
/* `count` <= cfg.max_batch frames, each from its own host buffer. */
int b200tag_detect_batch(b200tag_detector *det, const uint8_t *const *host_images, int count);
/* Frames already resident in device memory, `count` frames `frame_stride_bytes` apart
 * (0 = tightly packed).  Runs on the detector's stream and returns when results are on the host. */
int b200tag_detect_device(b200tag_detector *det, const void *device_images, size_t frame_stride_bytes, int count);

/* Asynchronous halves of b200tag_detect_device, for callers that time or overlap on the GPU:
 * enqueue puts all device work + the result copy on the detector's stream, finish waits for it
 * and builds the detection lists.  `stream_out` (optional) receives the cudaStream_t. */
int b200tag_enqueue_device(b200tag_detector *det, const void *device_images, size_t frame_stride_bytes, int count);
int b200tag_enqueue_host(b200tag_detector *det, const uint8_t *const *host_images, int count);
/* `count` frames of ONE host allocation, `frame_stride_bytes` apart (0 = back to back), e.g. a pinned camera ring
 * buffer: they cross PCIe in a single copy instead of one per frame. */
int b200tag_enqueue_host_block(b200tag_detector *det, const uint8_t *host_frames, size_t frame_stride_bytes, int count);
/* Camera wire format (SURVEY section 8 row f2; reference: camera_publisher.cpp:198,336 decodes the cameras' MJPG stream
 * to bgr8 with OpenCV on the CPU, apriltags_cuda_detector.cu:399-401 then converts bgr8 -> YUYV).  `count` JPEG
 * bitstreams in host memory, each width x height of a detector created for B200TAG_FMT_GRAY8: their luminance planes
 * are decoded on the detector's stream into its input staging buffer and the detection pipeline runs behind that.
 * Baseline JPEG (8-bit, Huffman, one interleaved scan, gray or YCbCr with full-resolution luminance, with or without
 * DHT segments / restart markers -- what UVC cameras send) goes through the detector's own decode kernel
 * (csrc/kernels_jpeg.cu); other JPEG kinds (progressive, ...) through nvJPEG (libnvjpeg.so.12 of the CUDA toolkit,
 * loaded on first use).  enqueue + b200tag_finish, or the synchronous b200tag_detect_mjpg.  B200TAG_E_INVALID for a
 * bitstream that cannot be parsed or is of the wrong size.  b200tag_mjpg_backend names the decoder of the last batch
 * ("native", or nvJPEG's "gpu" / "hardware" / "hybrid" / "default"; "" before the first call).
 * b200tag_jpeg_probe (host only) parses the headers: info = {width, height, blocks per MCU, luminance blocks per MCU
 * horizontally, vertically, restart interval, offset of the entropy-coded data, MCUs}, `dht_out` the Huffman tables in
 * use (per table: present flag, 16 counts, values; tables K.3-K.6 of ITU-T T.81 when the stream has none); returns 1
 * for a JPEG the native kernel does not handle. */
int b200tag_enqueue_mjpg(b200tag_detector *det, const uint8_t *const *jpegs, const size_t *sizes, int count);
int b200tag_detect_mjpg(b200tag_detector *det, const uint8_t *const *jpegs, const size_t *sizes, int count);
const char *b200tag_mjpg_backend(const b200tag_detector *det);
int b200tag_jpeg_probe(const uint8_t *jpeg, size_t size, int32_t info[8], uint8_t *dht_out, size_t dht_cap, size_t *dht_len);
/* How many of the first `count` frames of the last MJPG batch the parallel decode kernels handled (the rest -- streams
 * with restart markers, or whose synchronisation was not proven within the fixed number of rounds -- went through the
 * sequential warp-per-frame kernel).  Synchronises the stream. */
int b200tag_mjpg_parallel_frames(b200tag_detector *det, int count);
/* Test hook: host model of the parallel JPEG decode kernels (same entropy-decoding core and arithmetic, threads replaced
 * by loops), so the scheme can be checked without a GPU.  Not on any detection path.  0 = plane written to `out`;
 * 1 = a stream the parallel path does not take (restart markers, non-baseline); `rounds` = synchronisation rounds. */
int b200tag_debug_jpeg_model(const uint8_t *jpeg, size_t size, uint8_t *out, size_t out_cap, int *rounds);
int b200tag_finish(b200tag_detector *det);
void *b200tag_stream(b200tag_detector *det);

/* GpuDetector::Detections(): detections of frame `frame` of the last call, after reconcile,
 * sorted by id.  The array is owned by the detector and valid until the next detect call. */
const b200tag_detection *b200tag_detections(const b200tag_detector *det, int frame, int *count);
/* GpuDetector::FitQuads(). */
const b200tag_quad *b200tag_quads(const b200tag_detector *det, int frame, int *count);
int b200tag_frame_info_get(const b200tag_detector *det, int frame, b200tag_frame_info *info);

/* Copies one intermediate stage of frame `frame` to `dst` (host).  `out_bytes` receives the
 * stage size; returns B200TAG_E_INVALID if cap_bytes is too small. */
int b200tag_copy_stage(b200tag_detector *det, int frame, int stage, void *dst, size_t cap_bytes, size_t *out_bytes);

/* SetCameraMatrix / SetDistortionCoefficients (apriltag_gpu.h:189-195). */
int b200tag_set_camera(b200tag_detector *det, double fx, double cx, double fy, double cy);
int b200tag_set_distortion(b200tag_detector *det, double k1, double k2, double p1, double p2, double k3);

/* GpuDetector::UnDistort (apriltag_gpu.h:199-200, apriltag_detect.cu:335-402). Pure host helper. */
int b200tag_undistort(double *u, double *v, double fx, double cx, double fy, double cy, double k1, double k2,
                      double p1, double p2, double k3);

/* Pose of a tag in the camera frame (x right, y down, z forward): X_cam = R * X_tag + t, tag corners at
 * (+-tagsize/2, +-tagsize/2, 0).  The step the node runs on every detection right after Detect
 * (libapriltag estimate_tag_pose, called at apriltags_cuda_detector.cu:433): initial pose from the homography,
 * orthogonal iteration, the second local minimum of the object-space error, the better of the two returned.
 * Restated from the published algorithm -- libapriltag is not vendored in the reference tree. */
typedef struct b200tag_pose {
  double R[9];       /* row-major 3x3 rotation */
  double t[3];
  double err;        /* object-space error of the returned pose (estimate_tag_pose's return value) */
  double err_other;  /* error of the other local minimum, HUGE_VAL if there is none */
} b200tag_pose;
int b200tag_estimate_pose(const b200tag_detection *det, double tagsize, double fx, double fy, double cx, double cy,
                          b200tag_pose *out);
int b200tag_estimate_poses(const b200tag_detection *dets, int count, double tagsize, double fx, double fy, double cx,
                           double cy, b200tag_pose *out);

/* Pose methods.  ORTHOGONAL_ITERATION is the algorithm above (libapriltag's estimate_tag_pose, the default
 * everywhere).  IPPE is Infinitesimal Plane-based Pose Estimation (Collins & Bartoli 2014) for a square tag, the two
 * candidates OpenCV's solvePnPGeneric(..., SOLVEPNP_IPPE_SQUARE) returns: closed form from the homography of the
 * detection's corners p (not H), without iteration.  It solves the image-plane problem rather than minimising the
 * object-space error, so with pixel noise its pose differs from OI's by about the pose's own uncertainty.  The returned
 * candidate is the one with the smaller object-space error, and err / err_other are object-space errors as for OI.
 * A quad for which no candidate can be formed gives R = I, t = 0 and err = err_other = HUGE_VAL. */
enum { B200TAG_POSE_ORTHOGONAL_ITERATION = 0, B200TAG_POSE_IPPE = 1 };
/* b200tag_estimate_poses with IPPE; the same arguments and checks. */
int b200tag_estimate_poses_ippe(const b200tag_detection *dets, int count, double tagsize, double fx, double fy, double cx,
                                double cy, b200tag_pose *out);

/* The rest of the node's per-frame step (apriltags_cuda_detector.cu:421-462,595-599): every detection's pose, the tag
 * position in the camera frame (the pose's t), in the robot frame (rotation * t + offset, transformCameraToRobot) and
 * its Euclidean distance from the camera; the records come back closest first, as the node publishes them (ties
 * keep the detections' order).  `rotation` is a row-major 3x3 matrix and `offset` a 3-vector, the camera's
 * "extrinsics" entry; NULL means identity / zero (the node's defaults, :36-37). */
typedef struct b200tag_tag_position {
  int index;          /* position of the detection in the input list */
  int id;
  double camera[3];   /* tag origin in the camera frame */
  double robot[3];    /* the same point in the robot frame */
  double distance;    /* |camera| */
  double err;         /* object-space error of the pose (estimate_tag_pose's return value) */
} b200tag_tag_position;
int b200tag_locate_tags(const b200tag_detection *dets, int count, double tagsize, double fx, double fy, double cx,
                        double cy, const double *rotation, const double *offset, b200tag_tag_position *out);

/* The same step on the device, inside every detect call: a kernel at the end of the detection graph estimates the pose
 * of every detection, and the results come back with the detections.  Off by default; a detector that never turns it
 * on launches, allocates and returns exactly what it would without it.
 * b200tag_set_pose_estimation turns it on (tagsize > 0) or off (tagsize == 0), with the same arguments and meaning as
 * b200tag_locate_tags; rotation / offset may be NULL.  B200TAG_E_INVALID (state unchanged) unless tagsize >= 0 and fx,
 * fy are non-zero.  Takes effect from the next detect call; adds one kernel to b200tag_kernels_per_batch. */
int b200tag_set_pose_estimation(b200tag_detector *det, double tagsize, double fx, double fy, double cx, double cy,
                                const double *rotation, const double *offset);
/* The method the device pose step runs from the next detect call: B200TAG_POSE_ORTHOGONAL_ITERATION (the default) or
 * B200TAG_POSE_IPPE, whose poses are bit-identical to b200tag_estimate_poses_ippe's.  Independent of
 * b200tag_set_pose_estimation, which alone turns the step on and off.  B200TAG_E_INVALID (state unchanged) for any
 * other value. */
int b200tag_set_pose_method(b200tag_detector *det, int method);
/* Poses of frame `frame` of the last call, parallel to b200tag_detections(det, frame): element i is the pose of
 * detection i.  NULL and *count = 0 when the last call ran without the pose step.  Owned by the detector, valid until
 * the next detect call. */
const b200tag_pose *b200tag_poses(const b200tag_detector *det, int frame, int *count);
/* The same detections as b200tag_locate_tags returns them (closest first, .index into b200tag_detections). */
const b200tag_tag_position *b200tag_tag_positions(const b200tag_detector *det, int frame, int *count);
/* Test hook, as b200tag_debug_math: the device pose kernel on caller-supplied records (current device); arguments and
 * results as b200tag_estimate_poses. */
int b200tag_debug_estimate_poses_device(const b200tag_detection *dets, int count, double tagsize, double fx, double fy,
                                        double cx, double cy, b200tag_pose *out);
/* The same for the device IPPE kernel; results as b200tag_estimate_poses_ippe. */
int b200tag_debug_estimate_poses_ippe_device(const b200tag_detection *dets, int count, double tagsize, double fx,
                                             double fy, double cx, double cy, b200tag_pose *out);

/* Field pose from every visible layout tag (a multi-tag solve): one camera pose per frame, fitted to the corners of all
 * tags of a field layout in view by least-squares pixel reprojection error.
 *
 * Tag frame: the one of b200tag_pose.  Detection corner p[i] is tag point P_i = (-s, s, 0), (s, s, 0), (s, -s, 0),
 * (-s, -s, 0), s = tagsize / 2; x points right and y down as the tag is read, z into the tag, so an upright tag seen
 * head-on has R = I.
 *
 * Layout: b200tag_field_tag places one tag's frame in the field, X_field = R * X_tag + t (R row-major, a rotation).
 * Every layout tag has the pose step's tagsize.
 *
 * Which detections take part: per layout (family, id) at most one, the one reconcile prefers (lower hamming, then the
 * larger decision_margin, then the smaller corners in reconcile's order).  Reconcile only removes the loser of a pair,
 * so that detection survives it: a raw device list and the reconciled list give the same pose.  A tag whose IPPE pose
 * cannot be formed is left out.  Correspondences are ordered by layout index, then corner 0..3.
 *
 * Solve: both IPPE candidates of every used tag, composed with its layout entry, are seeds, scored by the summed
 * squared pixel error over all corners (a seed putting any corner at Z <= 0 scores HUGE_VAL); the best is refined by
 * Levenberg-Marquardt on that error (pinhole model, Cayley rotation update, at most 20 iterations).  With exactly one
 * tag both candidates are refined and the better returned.  Only + - * /, sqrt, fabs and fmax, with every sum taken in
 * one fixed order, so host and device results are bit-identical. */
typedef struct b200tag_field_tag {
  int32_t family, id;  /* index into the detector's families, tag id */
  double R[9];         /* row-major: X_field = R * X_tag + t */
  double t[3];
} b200tag_field_tag;

typedef struct b200tag_field_pose {
  int32_t num_tags;     /* layout tags the solve used */
  int32_t iterations;   /* Levenberg-Marquardt iterations run (accepted and rejected steps) */
  int32_t reserved[2];
  double camera_R[9];   /* the camera in the field: X_field = camera_R * X_cam + camera_t */
  double camera_t[3];
  double robot_R[9];    /* the robot in the field, through the extrinsics X_robot = rotation * X_cam + offset:
                           robot_R = camera_R * rotation^T, robot_t = camera_t - robot_R * offset */
  double robot_t[3];
  double rms;           /* RMS pixel reprojection error over the corners used; HUGE_VAL when no seed has every corner
                           in front of the camera */
  double rms_other;     /* one tag only: the same for the other IPPE candidate after the same refinement; else HUGE_VAL */
} b200tag_field_pose;   /* num_tags == 0 (no usable layout tag): R = I, t = 0, rms = rms_other = HUGE_VAL */

#define B200TAG_MAX_FIELD_TAGS 1024

/* One frame on the host.  `dets` as b200tag_detections or a raw list; rotation / offset may be NULL (identity / zero).
 * B200TAG_E_INVALID for bad arguments (tagsize > 0, fx, fy non-zero) or a bad layout: NULL with nlayout > 0, more than
 * B200TAG_MAX_FIELD_TAGS tags, a duplicate (family, id), R not a rotation within 1e-6 (R R^T = I, det R > 0), a
 * non-finite value. */
int b200tag_estimate_field_pose(const b200tag_detection *dets, int count, const b200tag_field_tag *layout, int nlayout,
                                double tagsize, double fx, double fy, double cx, double cy, const double *rotation,
                                const double *offset, b200tag_field_pose *out);
/* The same solve on the device, inside every detect call, one kernel after the pose step: from the next detect call,
 * whenever the pose step is on (b200tag_set_pose_estimation, with either method) and the layout is not empty, with the
 * pose step's tagsize, intrinsics and extrinsics.  count == 0 turns it off.  The layout is copied to the device on the
 * detector's stream (a batch in flight keeps the old one).  Besides the checks of b200tag_estimate_field_pose,
 * B200TAG_E_INVALID for a family outside the detector's families or an id outside the family's codes; the state is
 * unchanged on any error.  Adds one kernel to b200tag_kernels_per_batch while it runs. */
int b200tag_set_field_layout(b200tag_detector *det, const b200tag_field_tag *layout, int count);
/* The field pose of frame `frame` of the last call; NULL when that call ran without the step.  Owned by the detector,
 * valid until the next detect call. */
const b200tag_field_pose *b200tag_field_pose_get(const b200tag_detector *det, int frame);
/* Test hook: the device kernel on one caller-supplied (raw) list; arguments and result as b200tag_estimate_field_pose. */
int b200tag_debug_estimate_field_pose_device(const b200tag_detection *dets, int count, const b200tag_field_tag *layout,
                                             int nlayout, double tagsize, double fx, double fy, double cx, double cy,
                                             const double *rotation, const double *offset, b200tag_field_pose *out);

/* Pinned host staging memory, so b200tag_detect* can overlap H2D with compute. */
void *b200tag_alloc_pinned(size_t bytes);
/* Write-combined pinned memory: for buffers the CPU (or a capture driver) only ever WRITES, such as a camera ring
 * buffer; the DMA engine reads it without snooping the CPU caches, which matters when several GPUs pull frames from
 * the same host at once.  CPU reads from it are slow.  Free with b200tag_free_pinned. */
void *b200tag_alloc_pinned_wc(size_t bytes);
void b200tag_free_pinned(void *p);

/* Number of this library's kernels launched per frame batch (for benchmarks' gpu_launches). */
int b200tag_kernels_per_batch(const b200tag_detector *det);
/* Per-kernel device time of the last b200tag_profile_device call (ms); names are static strings. */
int b200tag_profile_device(b200tag_detector *det, const void *device_images, size_t frame_stride_bytes, int count,
                           int iters, const char **names, float *ms, int cap, int *n);

/* Test hook: reconcile_detections (libapriltag; apriltag_detect.cu:660) as the engine runs it on the host after every
 * frame, on a caller-supplied list: overlapping detections of the same family and id are reduced to the one with the
 * lower hamming distance, then the larger decision margin; the survivors are sorted by id.  Returns their number. */
int b200tag_debug_reconcile(b200tag_detection *dets, int count);

/* Test hook: out[i] = atan2f(a[i], b[i]) (op 0) or hypotf(a[i], b[i]) (op 1) evaluated on the device. */
int b200tag_debug_math(int op, const float *a, const float *b, float *out, int n);

const char *b200tag_error_string(int code);
const char *b200tag_last_error(const b200tag_detector *det);
int b200tag_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B200TAG_H_ */
