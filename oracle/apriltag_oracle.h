/*
 * TEST INFRASTRUCTURE -- CPU oracle for the AprilTag detection hot path.
 *
 * A plain-C restatement of the algorithm implemented by the reference's
 * frc971::apriltag::GpuDetector::Detect (src/apriltags_cuda/src/apriltag_gpu.cu:725-1166
 * and the files it calls).  It exists only to check the CUDA engine in
 * ros_vision_b200/: only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may load it.  The product never links it.
 *
 * Parity status (see DESIGN.md "Oracle"):
 *   - front end through QuadCorners: follows in-tree reference sources line by
 *     line (citations on every function in apriltag_oracle.c); pinned by the
 *     reference's own known answers (tests/golden) and, on the GPU box, by the
 *     reference's kernels compiled from /root/reference into oracle/_ref.
 *   - decode / reconcile (quad_decode_index, reconcile_detections) live in the
 *     un-vendored libapriltag fork github.com/cgpadwick/apriltag tag 3.3.0
 *     (src/external/CMakeLists.txt:86-95); restated from the published AprilTag 3
 *     algorithm.  For decision_margin and H: PARITY UNPINNED (no reference
 *     test asserts them); ids and corners are pinned by gpu_detector_test.cu's
 *     known answers.  The codeword lookup (id, hamming, rotation at max_hamming
 *     0..3, lowest id when two codes are within reach), the rotation applied to H
 *     and the corner order are pinned by a brute-force reference and rendered
 *     ground truth (tests/test_decode_reference_cpu.py): every orientation,
 *     0..4 flipped cells, reversed borders.
 */
#ifndef APRILTAG_ORACLE_H_
#define APRILTAG_ORACLE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { ORC_FMT_GRAY8 = 0, ORC_FMT_YUYV = 1, ORC_FMT_BGR8 = 2 };

typedef struct {
  int width, height;      /* full-resolution frame */
  int format;             /* ORC_FMT_* */
  int quad_decimate;      /* integer factor >= 1 (reference supports only 2) */
  float quad_sigma;       /* 0 = off; >0 blur, <0 sharpen (upstream semantics) */
  int refine_edges;
  double decode_sharpening;
  int min_cluster_pixels; /* qtp */
  int max_nmaxima;        /* must be 10 */
  float cos_critical_rad;
  float max_line_fit_mse;
  int min_white_black_diff;
  double fx, cx, fy, cy;      /* CameraMatrix, apriltag_gpu.h:61-66 */
  double k1, k2, p1, p2, k3;  /* DistCoeffs, apriltag_gpu.h:68-74 */
  int max_stage;          /* stop after this stage (ORC_STAGE_*), for timing/tests */
  uint32_t family_mask;   /* bit i = built-in family i (orc_family_get); 0 means tag36h11 only */
  /* The caller's families, as b200tag_family lists them (codes, bit_x / bit_y, widths, reversed_border,
   * max_hamming).  When nfamilies > 0 they replace family_mask and detections carry an index into this list. */
  const struct orc_family *families;
  int nfamilies;
} orc_config;

/* apriltag_family_t (libapriltag apriltag.h), the fields the detector reads, and the bits_corrected the family was
 * added with (apriltag_detector_add_family_bits). */
typedef struct orc_family {
  const char *name;
  int nbits, ncodes;
  int width_at_border, total_width;
  int reversed_border;
  int h; /* minimum Hamming distance */
  const uint64_t *codes;
  const int32_t *bit_x, *bit_y;
  int max_hamming; /* 0..3; the built-in families use 2 */
} orc_family;
#define ORC_NUM_FAMILIES 3 /* 0 tag36h11, 1 tag25h9, 2 tag16h5 */
const orc_family *orc_family_get(int index);
int orc_family_index(const char *name);

enum {
  ORC_STAGE_THRESHOLD = 1,
  ORC_STAGE_LABELS = 2,
  ORC_STAGE_POINTS = 3,
  ORC_STAGE_BLOBS = 4,
  ORC_STAGE_LINEFIT = 5,
  ORC_STAGE_QUADS = 6,
  ORC_STAGE_DECODE = 7,
};

/* One boundary point (QuadBoundaryPoint, points.h:25-161), unpacked. */
typedef struct {
  uint32_t rep0, rep1; /* min / max component label */
  uint16_t x, y;       /* half-pixel coordinates: 2*base + d */
  uint16_t bx, by;     /* base pixel in the quad image */
  uint8_t dir;         /* 0:(1,0) 1:(1,1) 2:(0,1) 3:(-1,1) */
  uint8_t b2w;         /* black_to_white */
  uint8_t pad[2];
} orc_point;

/* Per blob-pair extents (MinMaxExtents, line_fit_filter.h:14-59). */
typedef struct {
  uint32_t rep0, rep1;
  uint16_t min_x, min_y, max_x, max_y;
  uint32_t start; /* first point in the key-sorted point list */
  uint32_t count;
  int32_t gx_sum, gy_sum;
  int64_t pxgx_plus_pygy_sum;
  int32_t selected;     /* passes SelectBlobs */
  uint32_t sel_start;   /* offset among selected points */
} orc_cluster;

/* A selected point after the angle sort (IndexPoint, points.h:169-279). */
typedef struct {
  uint32_t blob;  /* index into clusters[] */
  uint32_t theta; /* llrintf((atan2f+pi)*8e6) */
  uint16_t x, y, bx, by;
  uint8_t dir, pad[3];
} orc_spoint;

/* Inclusive per-blob prefix moments (LineFitPoint, line_fit_filter.h:61-83). */
typedef struct {
  int64_t Mxx, Myy, Mxy, Mx, My, W;
} orc_lfp;

typedef struct {
  int64_t Mx, My, W, Mxx, Myy, Mxy;
  int32_t N, pad;
} orc_moments;

/* FitQuad, line_fit_filter.h:130-135. */
typedef struct {
  uint32_t blob; /* index into clusters[] */
  uint32_t rep0, rep1;
  int32_t valid;
  int32_t npeaks;
  uint32_t indices[4];
  orc_moments moments[4];
  double err;
} orc_fitquad;

/* QuadCorners, apriltag_gpu.h:55-59 (corners in full-resolution pixels). */
typedef struct {
  float corners[4][2];
  int32_t reversed_border;
  uint32_t blob;
  uint32_t rep0, rep1;
} orc_quadcorners;

/* apriltag_detection_t as produced by quad_decode_index (libapriltag). */
typedef struct {
  int32_t id, hamming;
  float decision_margin;
  int32_t rotation;
  double H[9];
  double c[2];
  double p[4][2];
  uint32_t rep0, rep1;
  int32_t family; /* index into the built-in families */
  int32_t pad;
} orc_detection;

typedef struct {
  int W, H, w, h;
  uint8_t *gray;     /* W*H */
  uint8_t *quad_im;  /* w*h  decimated (and blurred) */
  uint8_t *minmax;   /* (w/4)*(h/4)*2 filtered tile min,max */
  uint8_t *thresh;   /* w*h  in {0,127,255} */
  uint32_t *labels;  /* w*h  smallest pixel index of the component; 127-pixels: own index */
  uint32_t *sizes;   /* w*h  pixel count at the root index, 0 elsewhere */
  int num_points;
  orc_point *points;       /* sorted by (rep0, rep1, dir, by, bx) */
  int num_clusters;
  orc_cluster *clusters;   /* sorted by (rep0, rep1) */
  int num_selected_points;
  orc_spoint *spoints;     /* sorted by (blob, theta, dir, by, bx) */
  orc_lfp *lfps;           /* num_selected_points */
  double *errs;            /* num_selected_points */
  double *filtered_errs;   /* num_selected_points */
  uint8_t *is_peak;        /* num_selected_points */
  int num_fitquads;
  orc_fitquad *fitquads;   /* one per selected blob having >= 1 peak, cluster order */
  int num_corners;
  orc_quadcorners *corners;
  int num_detections;
  orc_detection *detections; /* after reconcile, sorted by id */
  orc_quadcorners *refined;  /* num_corners: corners[] after RefineEdges (apriltag_detect.cu:405-564) */
} orc_result;

void orc_default_config(orc_config *cfg, int width, int height, int format);
/* Runs the detector on one frame.  Returns NULL on a bad configuration. */
orc_result *orc_detect(const orc_config *cfg, const uint8_t *image);
void orc_free_result(orc_result *r);

/* Exposed pieces (unit tests). */
float orc_emul_atan2f(float y, float x);
float orc_emul_hypotf(float a, float b);
int orc_undistort(double *u, double *v, const orc_config *cfg);
void orc_redistort(double *x, double *y, const orc_config *cfg);
int orc_homography_compute(const double corr[4][4], double H[9]);
uint64_t orc_tag36h11_code(int id);
/* quick-decode: returns id or -1; hamming/rotation via out params.  orc_decode_codeword is tag36h11 at
 * max_hamming 2; orc_decode_codeword_family takes the family's own max_hamming. */
int orc_decode_codeword(uint64_t rcode, int *hamming, int *rotation);
int orc_decode_codeword_family(const orc_family *fam, uint64_t rcode, int *hamming, int *rotation);

/* The classic CPU detector (libapriltag apriltag_detector_detect, the reference's second detection path:
 * test/gpu_detector_test.cu:104-157) restated in classic_detector.c.  `image` is a gray frame of cfg->width x
 * cfg->height (cfg->format is ignored).  Writes up to `cap` detections (after reconcile, sorted by id) and returns
 * their number; `nquads` (optional) receives the number of candidate quads. */
int orc_classic_detect(const orc_config *cfg, const uint8_t *gray, orc_detection *out, int cap, int *nquads);

#ifdef __cplusplus
}
#endif
#endif
