// Host side of the C ABI (include/b200tag.h): device-buffer arena, stream, launch sequence,
// result hand-off.  Mirrors the life cycle of frc971::apriltag::GpuDetector
// (reference: src/apriltags_cuda/src/apriltag_gpu.cu:111-220,725-1166) without any of its seven
// mid-frame host synchronisations: every data-dependent size stays in device counters.
#include <cuda_runtime.h>
#include <dlfcn.h>
// nvJPEG is optional: it only serves JPEG kinds the detector's own decode kernels do not take (progressive, 12-bit,
// arithmetic coding) and the comparison arm of tools/bench_mjpg.py.  Without its header the library builds all the
// same and such streams are refused with B200TAG_E_INVALID.
#if defined(__has_include)
#if __has_include(<nvjpeg.h>) && !defined(B200TAG_NO_NVJPEG)
#include <nvjpeg.h>
#define B200TAG_HAVE_NVJPEG 1
#endif
#endif

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/b200tag.h"
#include "dev_types.h"
#include "jpeg.h"
#include "jpeg_core.h"
#include "kernels.h"
#include "pose_core.h"

#include "tag_families_data.h"

using namespace b200tag;

// nvJPEG, bound at first use (b200tag_enqueue_mjpg): the library is part of the CUDA toolkit, but a detector that is
// never handed JPEG frames should not need it.
#ifdef B200TAG_HAVE_NVJPEG
struct MjpgDecoder {
  void *lib = nullptr;
  nvjpegHandle_t handle = nullptr;
  nvjpegJpegState_t state = nullptr;
  int backend = -1;       // nvjpegBackend_t the handle was created with
  int batch = 0;          // batch size of the last nvjpegDecodeBatchedInitialize
  decltype(&nvjpegCreateEx) create = nullptr;
  decltype(&nvjpegDestroy) destroy = nullptr;
  decltype(&nvjpegJpegStateCreate) state_create = nullptr;
  decltype(&nvjpegJpegStateDestroy) state_destroy = nullptr;
  decltype(&nvjpegGetImageInfo) image_info = nullptr;
  decltype(&nvjpegDecodeBatchedInitialize) batched_init = nullptr;
  decltype(&nvjpegDecodeBatched) batched = nullptr;
};
#else
struct MjpgDecoder {
  void *lib = nullptr;
  void *handle = nullptr;
  int backend = -1;
};
#endif

// The detector's own JPEG luminance decoder (kernels_jpeg.cu): one pinned host block and its device twin hold, per
// batch, the frame descriptors, the Huffman table sets and the entropy-coded segments; one copy moves all of it.
struct NativeJpeg {
  uint8_t *h_block = nullptr;  // pinned
  uint8_t *d_block = nullptr;
  size_t cap = 0;
  uint8_t *d_ws = nullptr;     // workspace of the parallel kernels, sized with `cap`
  int16_t *d_coef = nullptr;   // coefficient buffer (fixed size, all zero between batches)
  uint32_t *d_rst = nullptr;   // restart-interval starts, one slot per 8x8 block of a frame
  int16_t *d_dcs = nullptr;    // DC values, one per 8x8 block of a frame
  size_t coef_stride = 0;
  bool init = false;
  std::vector<JpegParsed> parsed;
  bool last_native = false;    // the last MJPG batch went through this decoder (else nvJPEG)
  const uint32_t *d_proven = nullptr;  // per frame of the last batch: decoded by the parallel kernels
  bool last_parallel = false;
};

struct b200tag_detector {
  b200tag_config cfg;
  FrameParams fp;
  int device = 0;
  cudaStream_t stream = nullptr;
  SideStreams side;  // concurrent blob-tier kernels
  // CUDA graphs of the whole launch sequence, keyed by (input pointer, stride, frame count)
  struct GraphEntry {
    const void *images;
    size_t stride;
    int count;
    int launches;
    cudaGraphExec_t exec;
  };
  std::vector<GraphEntry> graphs;
  bool use_graphs = true;
  void *arena = nullptr;
  size_t arena_bytes = 0;
  uint8_t *d_in = nullptr;  // internal input staging (frames copied from the host)
  size_t in_bytes = 0;      // bytes per frame of input
  // host-visible results
  Counters *h_counters = nullptr;          // pinned, max_batch
  b200tag_detection *h_dets = nullptr;     // pinned + mapped, max_batch * det_cap (kernels write here)
  b200tag_detection *d_dets_alias = nullptr;
  std::vector<std::vector<b200tag_detection>> dets;  // after reconcile
  std::vector<std::vector<b200tag_quad>> quads;
  std::vector<bool> quads_valid;
  int last_count = 0;
  const uint8_t *last_images = nullptr;  // input of the last enqueue (d_in for host / JPEG frames)
  size_t last_stride = 0;
  bool pending = false;
  int kernels_per_batch = 0;
  std::string err;
  KernelTimer timer;
  MjpgDecoder mjpg;
  NativeJpeg jpeg;
  std::vector<uint32_t> host_status;  // per frame of the last batch: status bits raised on the host (B200TAG_ST_JPEG_TRUNCATED)
  void *d_families = nullptr;  // DevFamily[nfamilies] followed by the code tables
  int min_width_at_border = 8;
  bool normal_border = true, reversed_border = false;
  // the pose step (b200tag_set_pose_estimation): on while tagsize > 0
  struct PoseSettings {
    double tagsize = 0, fx = 0, fy = 0, cx = 0, cy = 0;
    double rotation[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, offset[3] = {0, 0, 0};
    int method = B200TAG_POSE_ORTHOGONAL_ITERATION;  // b200tag_set_pose_method
    double dist[5] = {0, 0, 0, 0, 0};                 // b200tag_set_pose_distortion; all zero: none
    double sigma = 0;                                 // b200tag_set_pose_covariance; 0: no covariances
  };
  PoseSettings pose, last_pose;                // current; what the last enqueue ran with
  b200tag_pose *h_poses = nullptr;             // pinned + mapped, parallel to h_dets; allocated when first turned on
  b200tag_pose *d_poses_alias = nullptr;
  std::vector<std::vector<b200tag_pose>> poses;                   // parallel to dets
  std::vector<std::vector<b200tag_tag_position>> positions;       // closest first
  std::vector<uint32_t> family_ncodes;                            // codes per family, for the layout checks
  // the field pose step (b200tag_set_field_layout): on while the pose step is on and field_n > 0
  int field_n = 0;
  bool last_field = false;                     // the last enqueue ran the step
  b200tag_field_tag *d_field_layout = nullptr; // device, B200TAG_MAX_FIELD_TAGS entries; allocated when first set
  pose::FieldKey *d_field_keys = nullptr;      // device, the layout's sorted keys
  void *d_field_scratch = nullptr;             // device, per frame field_scratch_stride pose::FieldTagData
  uint32_t field_scratch_stride = 0;
  b200tag_field_pose *h_field = nullptr;       // pinned + mapped, max_batch entries
  b200tag_field_pose *d_field_alias = nullptr;
  std::vector<b200tag_field_pose> field_poses; // per frame of the last call
  // the covariances (b200tag_set_pose_covariance): pinned + mapped, allocated when first turned on
  b200tag_covariance *h_cov = nullptr;         // parallel to h_dets
  b200tag_covariance *d_cov_alias = nullptr;
  b200tag_field_covariance *h_field_cov = nullptr;  // max_batch entries
  b200tag_field_covariance *d_field_cov_alias = nullptr;
  std::vector<std::vector<b200tag_covariance>> covs;  // parallel to dets
  std::vector<b200tag_field_covariance> field_covs;   // per frame of the last call
  // the floor pose step (b200tag_set_floor_pose): on while the field step runs and floor_weight > 0
  double floor_weight = 0;
  bool last_floor = false;                     // the last enqueue ran the step
  b200tag_floor_pose *h_floor = nullptr;       // pinned + mapped, max_batch entries; allocated when first turned on
  b200tag_floor_pose *d_floor_alias = nullptr;
  double *h_floor_cov = nullptr;               // pinned + mapped, 9 per frame
  double *d_floor_cov_alias = nullptr;
  double *h_gyro = nullptr;                    // pinned + mapped, (cos, sin) per frame, NaN: no heading; written by
  double *d_gyro_alias = nullptr;              // enqueue_impl, when no batch is in flight
  std::vector<double> next_gyro;               // b200tag_set_robot_headings: (cos, sin) per frame for the next call
  bool next_gyro_set = false;
  std::vector<b200tag_floor_pose> floor_poses; // per frame of the last call
  std::vector<double> floor_covs;              // 9 per frame of the last call
};

namespace b200tag {
// test hook: evaluates the device libm routines the hot path depends on (atan2f / hypotf)
__global__ void k_debug_math(int op, const float *a, const float *b, float *out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = op == 0 ? atan2f(a[i], b[i]) : hypotf(a[i], b[i]);
}
}  // namespace b200tag

namespace {

thread_local std::string g_create_error;

#define CK(call)                                                                                  \
  do {                                                                                            \
    cudaError_t e_ = (call);                                                                      \
    if (e_ != cudaSuccess) {                                                                      \
      char buf_[512];                                                                             \
      snprintf(buf_, sizeof(buf_), "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      det->err = buf_;                                                                            \
      return B200TAG_E_CUDA;                                                                      \
    }                                                                                             \
  } while (0)

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// The current CUDA device is per host thread.  Every entry point that touches CUDA runs on the detector's own
// device and puts the caller's back on exit, so a detector can be driven from any thread (a ROS executor) and
// detectors on different GPUs can live in one process.
struct DeviceGuard {
  int prev = -1, dev = -1;
  explicit DeviceGuard(int device) : dev(device) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (dev >= 0 && prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    if (dev >= 0 && prev >= 0 && prev != dev) cudaSetDevice(prev);
  }
  DeviceGuard(const DeviceGuard &) = delete;
  DeviceGuard &operator=(const DeviceGuard &) = delete;
};

struct ArenaPlan {
  size_t off = 0;
  size_t take(size_t bytes) {
    const size_t o = off;
    off = align_up(off + bytes, 256);
    return o;
  }
};

int blur_kernel(float quad_sigma, uint8_t *k) {  // image_u8_gaussian_blur's kernel (libapriltag, recalled)
  const float sigma = fabsf(quad_sigma);
  int ksz = static_cast<int>(4 * sigma);
  if ((ksz & 1) == 0) ksz++;
  if (ksz <= 1) return 0;
  if (ksz > 31) ksz = 31;
  double dk[32], acc = 0;
  for (int i = 0; i < ksz; i++) {
    const int x = -ksz / 2 + i;
    const double q = x / sigma;
    dk[i] = exp(-.5 * q * q);
    acc += dk[i];
  }
  for (int i = 0; i < ksz; i++) k[i] = static_cast<uint8_t>(dk[i] / acc * 255);
  return ksz;
}

// reconcile_detections (libapriltag; declared at apriltag_detect.cu:31-32, called at :660) ------
bool seg_intersect(const double *a0, const double *a1, const double *b0, const double *b1) {
  const double d1x = a1[0] - a0[0], d1y = a1[1] - a0[1];
  const double d2x = b1[0] - b0[0], d2y = b1[1] - b0[1];
  const double den = d1x * d2y - d1y * d2x;
  if (den == 0) return false;
  const double t = ((b0[0] - a0[0]) * d2y - (b0[1] - a0[1]) * d2x) / den;
  const double u = ((b0[0] - a0[0]) * d1y - (b0[1] - a0[1]) * d1x) / den;
  return t >= 0 && t <= 1 && u >= 0 && u <= 1;
}
bool poly_contains(const double p[4][2], const double *q) {
  bool c = false;
  for (int i = 0, j = 3; i < 4; j = i++) {
    if (((p[i][1] > q[1]) != (p[j][1] > q[1])) &&
        (q[0] < (p[j][0] - p[i][0]) * (q[1] - p[i][1]) / (p[j][1] - p[i][1]) + p[i][0]))
      c = !c;
  }
  return c;
}
bool polys_overlap(const double a[4][2], const double b[4][2]) {
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++)
      if (seg_intersect(a[i], a[(i + 1) & 3], b[j], b[(j + 1) & 3])) return true;
  double ca[2] = {0, 0}, cb[2] = {0, 0};
  for (int i = 0; i < 4; i++) {
    ca[0] += a[i][0] / 4; ca[1] += a[i][1] / 4;
    cb[0] += b[i][0] / 4; cb[1] += b[i][1] / 4;
  }
  return poly_contains(a, cb) || poly_contains(b, ca);
}
int prefer_smaller(int pref, double q0, double q1) {
  if (pref) return pref;
  if (q0 < q1) return -1;
  if (q1 < q0) return 1;
  return 0;
}
bool det_less(const b200tag_detection &a, const b200tag_detection &b) {  // detection_compare_function + tie-break
  if (a.id != b.id) return a.id < b.id;
  if (a.c[0] != b.c[0]) return a.c[0] < b.c[0];
  if (a.c[1] != b.c[1]) return a.c[1] < b.c[1];
  if (a.family != b.family) return a.family < b.family;
  return a.hamming < b.hamming;
}
// A detection with the pose the device computed for it: reconcile moves both together.
struct DetPose {
  b200tag_detection det;
  b200tag_pose pose;
};
// The same with the pose's covariance (b200tag_set_pose_covariance).
struct DetPoseCov {
  b200tag_detection det;
  b200tag_pose pose;
  b200tag_covariance cov;
};
const b200tag_detection &rec(const b200tag_detection &d) { return d; }
const b200tag_detection &rec(const DetPose &d) { return d.det; }
const b200tag_detection &rec(const DetPoseCov &d) { return d.det; }

template <class T>
void reconcile(std::vector<T> &v) {
  // device append order is arbitrary: fix it first
  std::sort(v.begin(), v.end(), [](const T &a, const T &b) { return det_less(rec(a), rec(b)); });
  auto d = [&v](int i) -> const b200tag_detection & { return rec(v[i]); };
  int n = static_cast<int>(v.size());
  for (int i0 = 0; i0 < n; i0++) {
    for (int i1 = i0 + 1; i1 < n; i1++) {
      if (d(i0).id != d(i1).id || d(i0).family != d(i1).family) continue;
      if (!polys_overlap(d(i0).p, d(i1).p)) continue;
      int pref = 0;
      pref = prefer_smaller(pref, d(i0).hamming, d(i1).hamming);
      pref = prefer_smaller(pref, -d(i0).decision_margin, -d(i1).decision_margin);
      for (int i = 0; i < 4; i++) {
        pref = prefer_smaller(pref, d(i0).p[i][0], d(i1).p[i][0]);
        pref = prefer_smaller(pref, d(i0).p[i][1], d(i1).p[i][1]);
      }
      if (pref < 0) {
        v[i1] = v[n - 1];
        n--;
        i1--;
      } else {
        v[i0] = v[n - 1];
        n--;
        i0--;
        break;
      }
    }
  }
  v.resize(n);
  std::sort(v.begin(), v.end(), [](const T &a, const T &b) { return det_less(rec(a), rec(b)); });
}

int validate(const b200tag_config &c, std::string *why) {
  auto bad = [&](const char *m) { *why = m; return B200TAG_E_INVALID; };
  if (c.abi_version != B200TAG_ABI_VERSION) return bad("abi_version mismatch");
  if (c.width <= 0 || c.height <= 0) return bad("width/height must be positive");
  if (c.format < B200TAG_FMT_GRAY8 || c.format > B200TAG_FMT_BGR8) return bad("unknown format");
  if (c.quad_decimate < 1 || c.quad_decimate > 8) return bad("quad_decimate must be an integer in [1, 8]");
  if (c.width % c.quad_decimate || c.height % c.quad_decimate) return bad("frame size must be divisible by quad_decimate");
  const int w = c.width / c.quad_decimate, h = c.height / c.quad_decimate;
  if (w % 4 || h % 4 || w < 8 || h < 8) return bad("quad image dimensions must be multiples of 4 (threshold.cu:156-157)");
  if (w > 4096 || h > 4096) return bad("quad image larger than 4096x4096 (12-bit point coordinates)");
  if (c.format == B200TAG_FMT_YUYV && (c.width % 8)) return bad("YUYV frames need width % 8 == 0");
  if (c.max_nmaxima != 10) return bad("max_nmaxima must be 10 (line_fit_filter.cu:1205)");
  if (c.max_batch < 1 || c.max_batch > 4096) return bad("max_batch out of range");
  return 0;
}

void build_params(b200tag_detector *det) {
  const b200tag_config &c = det->cfg;
  FrameParams &p = det->fp;
  memset(&p, 0, sizeof(p));
  p.W = c.width; p.H = c.height; p.f = c.quad_decimate;
  p.w = c.width / p.f; p.h = c.height / p.f;
  p.fmt = c.format;
  p.tiles_x = p.w / 4; p.tiles_y = p.h / 4;
  p.inv_w = static_cast<uint32_t>(((1ull << 32) + p.w - 1) / p.w);
  p.blur_ksz = c.quad_sigma != 0 ? blur_kernel(c.quad_sigma, p.blur_k) : 0;
  p.sharpen = c.quad_sigma < 0;
  p.min_white_black_diff = c.min_white_black_diff;
  p.min_cluster_pixels = static_cast<uint32_t>(std::max(24, c.min_cluster_pixels));  // apriltag_gpu.cu:529
  p.max_cluster_pixels = static_cast<uint32_t>(4 * (p.w + p.h));                      // :871 in quad-image units
  int mtw = det->min_width_at_border;  // min over the families; apriltag_gpu.cu:169-181
  mtw = static_cast<int>(static_cast<float>(mtw) / static_cast<float>(p.f));
  if (mtw < 3) mtw = 3;
  p.min_tag_width = mtw;
  p.normal_border = det->normal_border; p.reversed_border = det->reversed_border;
  p.cos_critical_rad = c.cos_critical_rad;
  p.max_line_fit_mse = c.max_line_fit_mse;
  p.refine_edges = c.refine_edges;
  p.decode_sharpening = c.decode_sharpening;
  p.fx = c.fx; p.cx = c.cx; p.fy = c.fy; p.cy = c.cy;
  p.k1 = c.k1; p.k2 = c.k2; p.p1 = c.p1; p.p2 = c.p2; p.k3 = c.k3;
  p.keep_stages = c.keep_stages;
  p.test_flags = c.test_flags;
}

int finish_impl(b200tag_detector *det) {
  if (!det->pending) return 0;
  CK(cudaStreamSynchronize(det->stream));
  det->pending = false;
  int rc = 0;
  for (int f = 0; f < det->last_count; f++) {
    const Counters &c = det->h_counters[f];
    const uint32_t nd = std::min(c.num_detections, det->fp.det_cap);
    const b200tag_detection *src = det->h_dets + static_cast<size_t>(f) * det->fp.det_cap;
    if (det->last_pose.tagsize > 0 && det->last_pose.sigma > 0) {
      const size_t o = static_cast<size_t>(f) * det->fp.det_cap;
      std::vector<DetPoseCov> all(nd);
      for (uint32_t i = 0; i < nd; i++) all[i] = DetPoseCov{src[i], det->h_poses[o + i], det->h_cov[o + i]};
      reconcile(all);
      det->dets[f].resize(all.size());
      det->poses[f].resize(all.size());
      det->covs[f].resize(all.size());
      for (size_t i = 0; i < all.size(); i++) {
        det->dets[f][i] = all[i].det;
        det->poses[f][i] = all[i].pose;
        det->covs[f][i] = all[i].cov;
      }
      det->positions[f].resize(all.size());
      locate_from_poses(det->dets[f].data(), det->poses[f].data(), static_cast<int>(all.size()), det->last_pose.rotation,
                        det->last_pose.offset, det->positions[f].data());
    } else if (det->last_pose.tagsize > 0) {
      const b200tag_pose *ps = det->h_poses + static_cast<size_t>(f) * det->fp.det_cap;
      std::vector<DetPose> both(nd);
      for (uint32_t i = 0; i < nd; i++) both[i] = DetPose{src[i], ps[i]};
      reconcile(both);
      det->dets[f].resize(both.size());
      det->poses[f].resize(both.size());
      for (size_t i = 0; i < both.size(); i++) {
        det->dets[f][i] = both[i].det;
        det->poses[f][i] = both[i].pose;
      }
      det->positions[f].resize(both.size());
      locate_from_poses(det->dets[f].data(), det->poses[f].data(), static_cast<int>(both.size()), det->last_pose.rotation,
                        det->last_pose.offset, det->positions[f].data());
    } else {
      det->dets[f].assign(src, src + nd);
      reconcile(det->dets[f]);
      det->poses[f].clear();
      det->positions[f].clear();
    }
    if (det->last_field) det->field_poses[f] = det->h_field[f];
    if (det->last_field && det->last_pose.sigma > 0) det->field_covs[f] = det->h_field_cov[f];
    if (det->last_floor) {
      b200tag_floor_pose &fp = det->floor_poses[f];
      fp = det->h_floor[f];
      fp.heading = std::atan2(fp.sin_heading, fp.cos_heading);
      if (det->last_pose.sigma > 0) memcpy(&det->floor_covs[9 * static_cast<size_t>(f)], det->h_floor_cov + 9 * static_cast<size_t>(f), 9 * sizeof(double));
    }
    det->quads_valid[f] = false;
    if (c.status) rc = B200TAG_E_OVERFLOW;
  }
  if (rc) det->err = "a fixed-capacity device buffer overflowed; see b200tag_frame_info.status";
  return rc;
}

void drop_graphs(b200tag_detector *det) {
  for (auto &g : det->graphs) cudaGraphExecDestroy(g.exec);
  det->graphs.clear();
}

// memset of the counters, every kernel, result counters to the host -- on det->stream (side streams fork/join inside)
int record_sequence(b200tag_detector *det, const void *device_images, size_t stride, int count, KernelTimer *kt, int *launches_out) {
  FrameParams p = det->fp;
  p.in = static_cast<const uint8_t *>(device_images);
  p.in_stride = stride ? stride : det->in_bytes;
  if (det->cfg.format == B200TAG_FMT_GRAY8) {
    p.gray = const_cast<uint8_t *>(p.in);
    p.gray_stride = p.in_stride;
  }
  CK(cudaMemsetAsync(p.counters, 0, sizeof(Counters) * count, det->stream));
  Launcher ln{det->stream, kt};
  launch_frontend(p, count, ln);
  launch_blobs(p, count, ln, kt ? nullptr : &det->side);  // per-kernel timing runs serially
  launch_decode(p, count, ln);
  if (det->pose.tagsize > 0) {
    const auto &ps = det->pose;
    PoseLaunch pl{det->d_dets_alias, det->d_poses_alias, p.counters, p.det_cap, 0, ps.tagsize, ps.fx, ps.fy, ps.cx, ps.cy,
                  ps.method, {}};
    memcpy(pl.dist, ps.dist, sizeof(pl.dist));
    launch_pose(pl, count, ln);
    if (ps.sigma > 0) launch_pose_cov(pl, det->d_cov_alias, ps.sigma, count, ln);
    if (det->field_n > 0) {
      FieldLaunch fl{det->d_dets_alias, p.counters, p.det_cap, 0, det->d_field_layout, det->d_field_keys, det->field_n,
                     static_cast<pose::FieldTagData *>(det->d_field_scratch), det->field_scratch_stride,
                     ps.tagsize, ps.fx, ps.fy, ps.cx, ps.cy, {}, {}, det->d_field_alias, {}};
      memcpy(fl.rotation, ps.rotation, sizeof(fl.rotation));
      memcpy(fl.offset, ps.offset, sizeof(fl.offset));
      memcpy(fl.dist, ps.dist, sizeof(fl.dist));
      fl.cov = det->d_field_cov_alias;
      fl.sigma = ps.sigma;
      launch_field_pose(fl, count, ln);
      if (det->floor_weight > 0) {
        FloorLaunch gl{fl.scratch, fl.scratch_stride, det->d_field_alias, det->d_gyro_alias, det->floor_weight,
                       ps.fx, ps.fy, ps.cx, ps.cy, {}, {}, {}, det->d_floor_alias, det->d_floor_cov_alias, ps.sigma};
        memcpy(gl.rotation, ps.rotation, sizeof(gl.rotation));
        memcpy(gl.offset, ps.offset, sizeof(gl.offset));
        memcpy(gl.dist, ps.dist, sizeof(gl.dist));
        launch_floor_pose(gl, count, ln);
      }
    }
  }
  *launches_out = ln.count;
  CK(cudaMemcpyAsync(det->h_counters, p.counters, sizeof(Counters) * count, cudaMemcpyDeviceToHost, det->stream));
  return 0;
}

// The launch sequence of a (input buffer, frame count) pair never changes, so it is captured once into a CUDA
// graph and replayed: one graph launch instead of 15 stream operations per batch (what matters for the
// single-frame latency path, where the kernels are short).
int enqueue_impl(b200tag_detector *det, const void *device_images, size_t stride, int count, KernelTimer *kt, bool keep_host_status = false) {
  if (!keep_host_status) det->host_status.assign(static_cast<size_t>(count), 0u);
  // the headings of b200tag_set_robot_headings belong to this call only; every caller has finished the previous batch,
  // so no kernel reads h_gyro while it is written
  const bool floor = det->pose.tagsize > 0 && det->field_n > 0 && det->floor_weight > 0;
  if (floor)
    for (int f = 0; f < count; f++) {
      const bool given = det->next_gyro_set && 2 * static_cast<size_t>(f) < det->next_gyro.size();
      det->h_gyro[2 * f] = given ? det->next_gyro[2 * f] : NAN;
      det->h_gyro[2 * f + 1] = given ? det->next_gyro[2 * f + 1] : NAN;
    }
  det->next_gyro_set = false;
  det->last_images = static_cast<const uint8_t *>(device_images);
  det->last_stride = stride ? stride : det->in_bytes;
  int launches = 0;
  bool done = false;
  if (!kt && det->use_graphs) {
    for (auto &g : det->graphs) {
      if (g.images == device_images && g.stride == stride && g.count == count) {
        CK(cudaGraphLaunch(g.exec, det->stream));
        launches = g.launches;
        done = true;
        break;
      }
    }
    if (!done && det->graphs.size() < 16) {
      cudaGraph_t graph = nullptr;
      CK(cudaStreamBeginCapture(det->stream, cudaStreamCaptureModeThreadLocal));
      const int rc = record_sequence(det, device_images, stride, count, nullptr, &launches);
      const cudaError_t ce = cudaStreamEndCapture(det->stream, &graph);
      cudaGraphExec_t exec = nullptr;
      if (rc == 0 && ce == cudaSuccess && graph && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) {
        det->graphs.push_back({device_images, stride, count, launches, exec});
        cudaGraphDestroy(graph);
        CK(cudaGraphLaunch(exec, det->stream));
        done = true;
      } else {  // capture not possible here: fall back to plain stream launches from now on
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        det->use_graphs = false;
      }
    }
  }
  if (!done) {
    if (int rc = record_sequence(det, device_images, stride, count, kt, &launches)) return rc;
  }
  det->kernels_per_batch = launches;
  CK(cudaGetLastError());
  det->last_pose = det->pose;
  det->last_field = det->pose.tagsize > 0 && det->field_n > 0;
  det->last_floor = floor;
  det->last_count = count;
  det->pending = true;
  return 0;
}

}  // namespace

extern "C" {

int b200tag_version(void) { return B200TAG_ABI_VERSION; }

const char *b200tag_error_string(int code) {
  switch (code) {
    case B200TAG_OK: return "ok";
    case B200TAG_E_INVALID: return "invalid argument or unsupported configuration";
    case B200TAG_E_NO_DEVICE: return "no usable CUDA device (this engine has no CPU fallback)";
    case B200TAG_E_CUDA: return "CUDA error";
    case B200TAG_E_OVERFLOW: return "device buffer overflow on this frame";
    case B200TAG_E_NOMEM: return "out of memory";
    default: return "unknown error";
  }
}

const char *b200tag_last_error(const b200tag_detector *det) { return det ? det->err.c_str() : g_create_error.c_str(); }

int b200tag_default_config(b200tag_config *cfg, int width, int height, int format) {
  if (!cfg) return B200TAG_E_INVALID;
  memset(cfg, 0, sizeof(*cfg));
  cfg->abi_version = B200TAG_ABI_VERSION;
  cfg->width = width;
  cfg->height = height;
  cfg->format = format;
  cfg->quad_decimate = 2;
  cfg->quad_sigma = 0.0f;
  cfg->refine_edges = 1;
  cfg->decode_sharpening = 0.25;
  cfg->min_cluster_pixels = 5;
  cfg->max_nmaxima = 10;
  cfg->cos_critical_rad = cosf(static_cast<float>(10 * 3.14159265358979323846 / 180));
  cfg->max_line_fit_mse = 10.0f;
  cfg->min_white_black_diff = 5;
  cfg->fx = 1.0; cfg->fy = 1.0; cfg->cx = 0.0; cfg->cy = 0.0;
  cfg->max_batch = 1;
  cfg->device = -1;
  cfg->keep_stages = 0;
  return 0;
}

namespace {
struct Builtin {
  b200tag_family fam;
  std::vector<uint32_t> bx, by;
};
const Builtin *builtin_families() {
  static Builtin table[3];
  static bool ready = [] {
    auto fill = [](Builtin &b, const char *name, uint32_t nbits, uint32_t ncodes, const uint64_t *codes, const int32_t *bx, const int32_t *by,
                   int wb, int tw) {
      b.bx.assign(bx, bx + nbits);
      b.by.assign(by, by + nbits);
      b.fam = b200tag_family{name, nbits, ncodes, codes, b.bx.data(), b.by.data(), wb, tw, 0, 2};
    };
    fill(table[0], "tag36h11", b200_tag36h11_NBITS, b200_tag36h11_NCODES, b200_tag36h11_codes, b200_tag36h11_bit_x, b200_tag36h11_bit_y,
         b200_tag36h11_WIDTH_AT_BORDER, b200_tag36h11_TOTAL_WIDTH);
    fill(table[1], "tag25h9", b200_tag25h9_NBITS, b200_tag25h9_NCODES, b200_tag25h9_codes, b200_tag25h9_bit_x, b200_tag25h9_bit_y,
         b200_tag25h9_WIDTH_AT_BORDER, b200_tag25h9_TOTAL_WIDTH);
    fill(table[2], "tag16h5", b200_tag16h5_NBITS, b200_tag16h5_NCODES, b200_tag16h5_codes, b200_tag16h5_bit_x, b200_tag16h5_bit_y,
         b200_tag16h5_WIDTH_AT_BORDER, b200_tag16h5_TOTAL_WIDTH);
    return true;
  }();
  (void)ready;
  return table;
}

// Validates the caller's families (apriltag_gpu.cu:169-177, apriltag_detect.cu:108) and builds the device tables.
int install_families(b200tag_detector *det, const b200tag_family *fams, int n) {
  if (!fams || n < 1 || n > kMaxFamilies) {
    det->err = "between 1 and 8 tag families are required";
    return B200TAG_E_INVALID;
  }
  bool normal = false, reversed = false;
  int min_wb = 1000000;
  size_t total_codes = 0;
  for (int i = 0; i < n; i++) {
    const b200tag_family &f = fams[i];
    if (f.nbits < 1 || f.nbits > static_cast<uint32_t>(kMaxFamilyBits) || f.ncodes < 1 || !f.codes || !f.bit_x || !f.bit_y ||
        f.width_at_border < 1 || f.width_at_border > 8 || f.total_width < f.width_at_border || f.total_width > kMaxTotalWidth ||
        f.max_hamming < 0 || f.max_hamming > 3) {
      det->err = std::string("tag family ") + (f.name ? f.name : "?") + ": outside the supported limits (nbits <= 64, width_at_border <= 8, "
                 "total_width <= 12, max_hamming <= 3)";
      return B200TAG_E_INVALID;
    }
    const int lo = (f.width_at_border - f.total_width) / 2, hi = lo + f.total_width;
    for (uint32_t b = 0; b < f.nbits; b++) {
      const int x = static_cast<int32_t>(f.bit_x[b]), y = static_cast<int32_t>(f.bit_y[b]);
      if (x < lo || x >= hi || y < lo || y >= hi) {
        det->err = std::string("tag family ") + (f.name ? f.name : "?") + ": a bit lies outside the tag";
        return B200TAG_E_INVALID;
      }
    }
    normal |= !f.reversed_border;
    reversed |= f.reversed_border != 0;
    min_wb = std::min(min_wb, f.width_at_border);
    total_codes += f.ncodes;
  }
  det->family_ncodes.clear();
  for (int i = 0; i < n; i++) det->family_ncodes.push_back(fams[i].ncodes);
  if (normal && reversed) {  // apriltag_detect.cu:108: exactly one border polarity across the families
    det->err = "tag families with normal and with reversed borders cannot be mixed (apriltag_detect.cu:108)";
    return B200TAG_E_INVALID;
  }
  std::vector<uint8_t> host(sizeof(DevFamily) * kMaxFamilies + total_codes * sizeof(uint64_t));
  DevFamily *df = reinterpret_cast<DevFamily *>(host.data());
  uint64_t *codes = reinterpret_cast<uint64_t *>(host.data() + sizeof(DevFamily) * kMaxFamilies);
  uint32_t off = 0;
  for (int i = 0; i < n; i++) {
    const b200tag_family &f = fams[i];
    memset(&df[i], 0, sizeof(DevFamily));
    df[i].nbits = f.nbits; df[i].ncodes = f.ncodes;
    df[i].width_at_border = f.width_at_border; df[i].total_width = f.total_width;
    df[i].reversed_border = f.reversed_border != 0; df[i].max_hamming = f.max_hamming;
    df[i].codes_off = off;
    for (uint32_t b = 0; b < f.nbits; b++) {
      df[i].bit_x[b] = static_cast<int8_t>(static_cast<int32_t>(f.bit_x[b]));
      df[i].bit_y[b] = static_cast<int8_t>(static_cast<int32_t>(f.bit_y[b]));
    }
    memcpy(codes + off, f.codes, f.ncodes * sizeof(uint64_t));
    off += f.ncodes;
  }
  if (cudaMalloc(&det->d_families, host.size()) != cudaSuccess ||
      cudaMemcpy(det->d_families, host.data(), host.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
    cudaGetLastError();
    det->err = "uploading the tag families failed";
    return B200TAG_E_CUDA;
  }
  det->fp.families = static_cast<const DevFamily *>(det->d_families);
  det->fp.family_codes = reinterpret_cast<const uint64_t *>(static_cast<const uint8_t *>(det->d_families) + sizeof(DevFamily) * kMaxFamilies);
  det->fp.nfamilies = n;
  det->min_width_at_border = min_wb;
  det->normal_border = normal;
  det->reversed_border = reversed;
  return 0;
}
}  // namespace

const b200tag_family *b200tag_builtin_family(const char *name) {
  if (!name) return nullptr;
  const Builtin *t = builtin_families();
  for (int i = 0; i < 3; i++)
    if (strcmp(name, t[i].fam.name) == 0) return &t[i].fam;
  return nullptr;
}

int b200tag_create(const b200tag_config *cfg, b200tag_detector **out) {
  return b200tag_create_families(cfg, b200tag_builtin_family("tag36h11"), 1, out);
}

int b200tag_debug_reconcile(b200tag_detection *dets, int count) {
  if (!dets || count < 0) return B200TAG_E_INVALID;
  std::vector<b200tag_detection> v(dets, dets + count);
  reconcile(v);
  std::copy(v.begin(), v.end(), dets);
  return static_cast<int>(v.size());
}

int b200tag_create_families(const b200tag_config *cfg, const b200tag_family *families, int nfamilies, b200tag_detector **out) {
  if (!cfg || !out) return B200TAG_E_INVALID;
  *out = nullptr;
  std::string why;
  if (int rc = validate(*cfg, &why)) {
    g_create_error = why;
    return rc;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    g_create_error = "no CUDA device visible";
    return B200TAG_E_NO_DEVICE;
  }
  b200tag_detector *det = new b200tag_detector();
  det->cfg = *cfg;
  auto fail = [&](int rc) {
    g_create_error = det->err;
    b200tag_destroy(det);
    return rc;
  };
  if (cfg->device >= ndev) {
    det->err = "device ordinal out of range";
    return fail(B200TAG_E_NO_DEVICE);
  }
  if (cfg->device >= 0) det->device = cfg->device;
  else if (cudaGetDevice(&det->device) != cudaSuccess) {
    det->err = "cudaGetDevice failed";
    return fail(B200TAG_E_NO_DEVICE);
  }
  DeviceGuard on_device(det->device);  // the caller's current device is left as it was
  {
    FrameParams keep;  // install_families fills det->fp's family fields; build_params starts from a clean struct
    if (int rc = install_families(det, families, nfamilies)) return fail(rc);
    keep = det->fp;
    build_params(det);
    det->fp.families = keep.families; det->fp.family_codes = keep.family_codes; det->fp.nfamilies = keep.nfamilies;
  }
  FrameParams &p = det->fp;
  const size_t N = static_cast<size_t>(p.W) * p.H, n = static_cast<size_t>(p.w) * p.h;
  const size_t tiles = static_cast<size_t>(p.tiles_x) * p.tiles_y;
  const int B = cfg->max_batch;
  const int bpp = cfg->format == B200TAG_FMT_GRAY8 ? 1 : (cfg->format == B200TAG_FMT_YUYV ? 2 : 3);
  det->in_bytes = N * bpp;
  p.point_cap = cfg->max_points ? cfg->max_points : static_cast<uint32_t>(2 * n);
  uint32_t hc = 4096;
  while (hc < n / 8 && hc < (1u << 19)) hc <<= 1;  // 20-bit blob indices in Counters::alloc
  p.hash_cap = hc;
  p.blob_cap = cfg->max_blobs ? cfg->max_blobs : static_cast<uint32_t>(std::min<size_t>(65536, std::max<size_t>(4096, n / 32)));
  p.quad_cap = std::min<uint32_t>(p.blob_cap, 8192);
  p.det_cap = cfg->max_detections ? cfg->max_detections : 256;
  p.cluster_cap = cfg->keep_stages ? hc : 0;

  ArenaPlan plan;
  const size_t o_in = plan.take(align_up(det->in_bytes, 256) * B);
  const size_t in_stride = align_up(det->in_bytes, 256);
  const size_t o_gray = cfg->format == B200TAG_FMT_GRAY8 ? 0 : plan.take(N * B);
  const size_t o_quad = plan.take(n * B);
  const size_t o_quad_tmp = p.blur_ksz ? plan.take(n * B) : 0;
  const size_t o_mmr = plan.take(tiles * 2 * B);
  const size_t o_mm = plan.take(tiles * 2 * B);
  const size_t o_th = plan.take(n * B);
  const size_t o_lab = plan.take(n * 4 * B);
  const size_t o_sz = plan.take(n * 4 * B);
  const size_t ccl_tiles = ccl_tiles_per_frame(p.w, p.h);
  const size_t o_troots = plan.take(ccl_tiles * ccl_root_cap() * 4 * B);
  const size_t o_tnroots = plan.take(ccl_tiles * 4 * B);
  const size_t o_pts = plan.take(static_cast<size_t>(p.point_cap) * 8 * B);
  const size_t HB = static_cast<size_t>(hc) * B;
  const size_t o_hkey = plan.take(HB * 8);
  const size_t o_hcnt = plan.take(HB * 4);
  const size_t o_soff = plan.take(HB * 4);
  const size_t o_sclu = cfg->keep_stages ? plan.take(HB * 4) : 0;
  const size_t o_occ = plan.take(HB * 4);
  const size_t o_blobs = plan.take(static_cast<size_t>(p.blob_cap) * sizeof(b200tag_blob) * B);
  const size_t o_segp = plan.take(static_cast<size_t>(p.point_cap) * 4 * B);
  const size_t o_small = plan.take(static_cast<size_t>(p.blob_cap) * sizeof(WorkItem) * B);
  const size_t o_large = plan.take(static_cast<size_t>(p.blob_cap) * sizeof(WorkItem) * B);
  const size_t o_clusters = p.cluster_cap ? plan.take(static_cast<size_t>(p.cluster_cap) * sizeof(b200tag_blob) * B) : 0;
  const size_t o_seg = plan.take(static_cast<size_t>(p.point_cap) * 8 * B);
  const size_t o_lfp = plan.take(static_cast<size_t>(p.point_cap) * sizeof(b200tag_lfp) * B);
  const size_t o_errs = plan.take(static_cast<size_t>(p.point_cap) * 4 * B);
  const size_t o_filt = plan.take(static_cast<size_t>(p.point_cap) * 8 * B);
  const size_t o_pkws = plan.take((static_cast<size_t>(p.point_cap) / 2 + 1) * 8 * B);
  const size_t o_ptab = plan.take(static_cast<size_t>(p.blob_cap) * sizeof(PeakTable) * B);
  const size_t o_fq = plan.take(static_cast<size_t>(p.blob_cap) * sizeof(b200tag_fit_quad) * B);
  const size_t o_quads = plan.take(static_cast<size_t>(p.quad_cap) * sizeof(b200tag_quad) * B);
  const size_t o_ctr = plan.take(sizeof(Counters) * B);
  det->arena_bytes = plan.off;
  cudaError_t e = cudaMalloc(&det->arena, det->arena_bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    char buf[256];
    snprintf(buf, sizeof(buf), "cudaMalloc of %zu bytes failed: %s", det->arena_bytes, cudaGetErrorString(e));
    det->err = buf;
    det->arena = nullptr;
    return fail(e == cudaErrorMemoryAllocation ? B200TAG_E_NOMEM : B200TAG_E_NO_DEVICE);
  }
  uint8_t *base = static_cast<uint8_t *>(det->arena);
  det->d_in = base + o_in;
  p.in = det->d_in; p.in_stride = in_stride;
  det->in_bytes = N * bpp;
  if (cfg->format == B200TAG_FMT_GRAY8) { p.gray = det->d_in; p.gray_stride = in_stride; }
  else { p.gray = base + o_gray; p.gray_stride = N; }
  p.quad = base + o_quad;
  p.quad_tmp = p.blur_ksz ? base + o_quad_tmp : nullptr;
  p.minmax_raw = base + o_mmr;
  p.minmax = base + o_mm;
  p.thresh = base + o_th;
  p.labels = reinterpret_cast<uint32_t *>(base + o_lab);
  p.sizes = reinterpret_cast<uint32_t *>(base + o_sz);
  p.tile_roots = reinterpret_cast<uint32_t *>(base + o_troots);
  p.tile_nroots = reinterpret_cast<uint32_t *>(base + o_tnroots);
  p.points = reinterpret_cast<uint64_t *>(base + o_pts);
  p.h_key = reinterpret_cast<unsigned long long *>(base + o_hkey);
  p.h_count = reinterpret_cast<uint32_t *>(base + o_hcnt);
  p.slot_off = reinterpret_cast<uint32_t *>(base + o_soff);
  p.slot_cluster = cfg->keep_stages ? reinterpret_cast<uint32_t *>(base + o_sclu) : nullptr;
  p.seg_pts = reinterpret_cast<uint32_t *>(base + o_segp);
  p.occupied = reinterpret_cast<uint32_t *>(base + o_occ);
  p.blobs = reinterpret_cast<b200tag_blob *>(base + o_blobs);
  p.small_list = reinterpret_cast<WorkItem *>(base + o_small);
  p.large_list = reinterpret_cast<WorkItem *>(base + o_large);
  p.clusters = p.cluster_cap ? reinterpret_cast<b200tag_blob *>(base + o_clusters) : nullptr;
  p.seg_keys = reinterpret_cast<uint64_t *>(base + o_seg);
  p.lfp = reinterpret_cast<b200tag_lfp *>(base + o_lfp);
  p.errs = reinterpret_cast<float *>(base + o_errs);
  p.filt = reinterpret_cast<double *>(base + o_filt);
  p.peak_ws = reinterpret_cast<uint64_t *>(base + o_pkws);
  p.peak_tables = reinterpret_cast<PeakTable *>(base + o_ptab);
  p.fit_quads = reinterpret_cast<b200tag_fit_quad *>(base + o_fq);
  p.quads = reinterpret_cast<b200tag_quad *>(base + o_quads);
  p.counters = reinterpret_cast<Counters *>(base + o_ctr);

  auto ck = [&](cudaError_t ce, const char *what) {
    if (ce != cudaSuccess) {
      det->err = std::string(what) + ": " + cudaGetErrorString(ce);
      return false;
    }
    return true;
  };
  if (!ck(cudaStreamCreateWithFlags(&det->stream, cudaStreamNonBlocking), "cudaStreamCreate")) return fail(B200TAG_E_CUDA);
  for (int i = 0; i < 3; i++) {
    if (!ck(cudaStreamCreateWithFlags(&det->side.s[i], cudaStreamNonBlocking), "cudaStreamCreate(side)")) return fail(B200TAG_E_CUDA);
    if (!ck(cudaEventCreateWithFlags(&det->side.join[i], cudaEventDisableTiming), "cudaEventCreate")) return fail(B200TAG_E_CUDA);
  }
  if (!ck(cudaEventCreateWithFlags(&det->side.fork, cudaEventDisableTiming), "cudaEventCreate")) return fail(B200TAG_E_CUDA);
  if (!ck(cudaHostAlloc(reinterpret_cast<void **>(&det->h_counters), sizeof(Counters) * B, cudaHostAllocDefault), "cudaHostAlloc"))
    return fail(B200TAG_E_CUDA);
  if (!ck(cudaHostAlloc(reinterpret_cast<void **>(&det->h_dets), sizeof(b200tag_detection) * p.det_cap * B, cudaHostAllocMapped),
          "cudaHostAlloc(mapped)"))
    return fail(B200TAG_E_CUDA);
  if (!ck(cudaHostGetDevicePointer(reinterpret_cast<void **>(&det->d_dets_alias), det->h_dets, 0), "cudaHostGetDevicePointer"))
    return fail(B200TAG_E_CUDA);
  p.dets = det->d_dets_alias;  // the decode kernel writes detections straight into pinned host memory
  if (const char *e = getenv("B200TAG_NO_GRAPH")) det->use_graphs = !(e[0] == '1');
  launch_blobs_init(det->stream);  // one-time attributes / tables, outside any later graph capture
  launch_hash_clear(p, B, det->stream);
  if (!ck(cudaStreamSynchronize(det->stream), "initial hash clear")) return fail(B200TAG_E_CUDA);
  det->dets.resize(B);
  det->poses.resize(B);
  det->positions.resize(B);
  det->field_poses.resize(B);
  det->covs.resize(B);
  det->field_covs.resize(B);
  det->floor_poses.resize(B);
  det->floor_covs.resize(9 * B);
  det->quads.resize(B);
  det->quads_valid.assign(B, false);
  memset(det->h_counters, 0, sizeof(Counters) * B);
  *out = det;
  return 0;
}

void b200tag_destroy(b200tag_detector *det) {
  if (!det) return;
  DeviceGuard on_device(det->device);
  if (det->stream) {
    cudaStreamSynchronize(det->stream);
    drop_graphs(det);
    cudaStreamDestroy(det->stream);
  }
  for (int i = 0; i < 3; i++) {
    if (det->side.s[i]) cudaStreamDestroy(det->side.s[i]);
    if (det->side.join[i]) cudaEventDestroy(det->side.join[i]);
  }
  if (det->side.fork) cudaEventDestroy(det->side.fork);
  if (det->jpeg.h_block) cudaFreeHost(det->jpeg.h_block);
  if (det->jpeg.d_block) cudaFree(det->jpeg.d_block);
  if (det->jpeg.d_ws) cudaFree(det->jpeg.d_ws);
  if (det->jpeg.d_coef) cudaFree(det->jpeg.d_coef);
  if (det->jpeg.d_rst) cudaFree(det->jpeg.d_rst);
  if (det->jpeg.d_dcs) cudaFree(det->jpeg.d_dcs);
#ifdef B200TAG_HAVE_NVJPEG
  if (det->mjpg.state) det->mjpg.state_destroy(det->mjpg.state);
  if (det->mjpg.handle) det->mjpg.destroy(det->mjpg.handle);
  if (det->mjpg.lib) dlclose(det->mjpg.lib);
#endif
  if (det->arena) cudaFree(det->arena);
  if (det->d_families) cudaFree(det->d_families);
  if (det->h_counters) cudaFreeHost(det->h_counters);
  if (det->h_dets) cudaFreeHost(det->h_dets);
  if (det->h_poses) cudaFreeHost(det->h_poses);
  if (det->d_field_layout) cudaFree(det->d_field_layout);
  if (det->d_field_keys) cudaFree(det->d_field_keys);
  if (det->d_field_scratch) cudaFree(det->d_field_scratch);
  if (det->h_field) cudaFreeHost(det->h_field);
  if (det->h_cov) cudaFreeHost(det->h_cov);
  if (det->h_field_cov) cudaFreeHost(det->h_field_cov);
  if (det->h_floor) cudaFreeHost(det->h_floor);
  if (det->h_floor_cov) cudaFreeHost(det->h_floor_cov);
  if (det->h_gyro) cudaFreeHost(det->h_gyro);
  delete det;
}

int b200tag_enqueue_device(b200tag_detector *det, const void *device_images, size_t stride, int count) {
  if (!det || !device_images || count < 1 || count > det->cfg.max_batch) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  if (det->pending) {
    if (int rc = finish_impl(det)) if (rc != B200TAG_E_OVERFLOW) return rc;
  }
  return enqueue_impl(det, device_images, stride, count, nullptr);
}

int b200tag_enqueue_host(b200tag_detector *det, const uint8_t *const *host_images, int count) {
  if (!det || !host_images || count < 1 || count > det->cfg.max_batch) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  if (det->pending) {
    if (int rc = finish_impl(det)) if (rc != B200TAG_E_OVERFLOW) return rc;
  }
  for (int f = 0; f < count; f++) {
    if (!host_images[f]) return B200TAG_E_INVALID;
    // GpuMemory::MemcpyAsyncFrom, apriltag_gpu.cu:729 (works for pageable and pinned buffers)
    CK(cudaMemcpyAsync(det->d_in + static_cast<size_t>(f) * det->fp.in_stride, host_images[f], det->in_bytes,
                       cudaMemcpyHostToDevice, det->stream));
  }
  return enqueue_impl(det, det->d_in, det->fp.in_stride, count, nullptr);
}

int b200tag_enqueue_host_block(b200tag_detector *det, const uint8_t *host_frames, size_t frame_stride_bytes, int count) {
  if (!det || !host_frames || count < 1 || count > det->cfg.max_batch) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  const size_t stride = frame_stride_bytes ? frame_stride_bytes : det->in_bytes;
  if (stride < det->in_bytes) return B200TAG_E_INVALID;
  if (det->pending) {
    if (int rc = finish_impl(det)) if (rc != B200TAG_E_OVERFLOW) return rc;
  }
  // the frames of one allocation (a camera ring buffer) cross PCIe in a single copy
  if (stride == det->in_bytes && det->fp.in_stride == det->in_bytes) {
    CK(cudaMemcpyAsync(det->d_in, host_frames, det->in_bytes * static_cast<size_t>(count), cudaMemcpyHostToDevice, det->stream));
  } else {
    CK(cudaMemcpy2DAsync(det->d_in, det->fp.in_stride, host_frames, stride, det->in_bytes, static_cast<size_t>(count),
                         cudaMemcpyHostToDevice, det->stream));
  }
  return enqueue_impl(det, det->d_in, det->fp.in_stride, count, nullptr);
}

// Camera wire format (SURVEY section 8 row f2): the cameras deliver MJPG (system_config.json "format": "MJPG"), which
// the reference's camera node has OpenCV decode to bgr8 on the CPU (camera_publisher.cpp:198,336) before the detector
// node converts bgr8 -> YUYV -> gray.  Here the JPEG bitstreams cross PCIe as they are (about a tenth of the YUYV
// bytes), nvJPEG decodes their luminance plane straight into the detector's input staging buffer on the detector's
// stream, and the gray pipeline runs behind it.
#ifdef B200TAG_HAVE_NVJPEG
static int mjpg_open(b200tag_detector *det) {
  MjpgDecoder &m = det->mjpg;
  if (m.handle) return 0;
  if (!m.lib) {
    for (const char *name : {"libnvjpeg.so.12", "libnvjpeg.so", "/usr/local/cuda/lib64/libnvjpeg.so.12"}) {
      m.lib = dlopen(name, RTLD_NOW | RTLD_LOCAL);
      if (m.lib) break;
    }
    if (!m.lib) {
      det->err = std::string("nvJPEG not found: ") + dlerror();
      return B200TAG_E_INVALID;
    }
    bool ok = true;
    auto bind = [&](auto &fn, const char *sym) {
      fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(m.lib, sym));
      ok = ok && fn != nullptr;
    };
    bind(m.create, "nvjpegCreateEx");
    bind(m.destroy, "nvjpegDestroy");
    bind(m.state_create, "nvjpegJpegStateCreate");
    bind(m.state_destroy, "nvjpegJpegStateDestroy");
    bind(m.image_info, "nvjpegGetImageInfo");
    bind(m.batched_init, "nvjpegDecodeBatchedInitialize");
    bind(m.batched, "nvjpegDecodeBatched");
    if (!ok) {
      det->err = "nvJPEG library lacks the batched-decode entry points";
      dlclose(m.lib);
      m.lib = nullptr;
      return B200TAG_E_INVALID;
    }
  }
  // B200TAG_NVJPEG_BACKEND=hardware|gpu|hybrid|default picks one backend; otherwise the first that can be created, in
  // the order GPU Huffman decode, default.  (The fixed-function engine is opt-in: it wants pinned input buffers.)
  std::vector<int> order = {NVJPEG_BACKEND_GPU_HYBRID, NVJPEG_BACKEND_DEFAULT};
  if (const char *e = getenv("B200TAG_NVJPEG_BACKEND")) {
    const std::string v(e);
    if (v == "hardware") order = {NVJPEG_BACKEND_HARDWARE};
    else if (v == "gpu") order = {NVJPEG_BACKEND_GPU_HYBRID};
    else if (v == "hybrid") order = {NVJPEG_BACKEND_HYBRID};
    else if (v == "default") order = {NVJPEG_BACKEND_DEFAULT};
  }
  for (int b : order) {
    if (m.create(static_cast<nvjpegBackend_t>(b), nullptr, nullptr, NVJPEG_FLAGS_DEFAULT, &m.handle) == NVJPEG_STATUS_SUCCESS) {
      m.backend = b;
      break;
    }
    m.handle = nullptr;
  }
  if (!m.handle) {
    det->err = "nvjpegCreateEx failed for every requested backend";
    return B200TAG_E_CUDA;
  }
  if (m.state_create(m.handle, &m.state) != NVJPEG_STATUS_SUCCESS) {
    m.destroy(m.handle);
    m.handle = nullptr;
    det->err = "nvjpegJpegStateCreate failed";
    return B200TAG_E_CUDA;
  }
  m.batch = 0;
  return 0;
}
#endif

// The detector's own decoder.  Returns 0 when the batch was enqueued, 1 when some frame is a valid JPEG of a kind the
// kernel does not handle (progressive, 12-bit, ...: the caller falls back to nvJPEG), or a negative error.
static int mjpg_native(b200tag_detector *det, const uint8_t *const *jpegs, const size_t *sizes, int count) {
  NativeJpeg &J = det->jpeg;
  J.parsed.resize(count);
  det->host_status.assign(static_cast<size_t>(count), 0u);
  std::vector<int> set_of(count, 0);
  std::vector<int> set_owner;  // frame whose tables define each distinct set
  size_t bytes = 0;
  for (int f = 0; f < count; f++) {
    if (!jpegs[f] || sizes[f] == 0) return B200TAG_E_INVALID;
    std::string why;
    const int rc = jpeg_parse(jpegs[f], sizes[f], &J.parsed[f], &why);
    if (rc == kJpegUnsupported) return 1;
    if (rc != kJpegOk) {
      det->err = "frame " + std::to_string(f) + ": not a JPEG bitstream this decoder can parse (" + why + ")";
      return B200TAG_E_INVALID;
    }
    {  // a complete frame ends with EOI (FF D9), possibly followed by padding; a cut-off one is decoded as far as it
       // goes (the rest of the plane stays flat gray) and flagged, so that the caller can drop it
      size_t e = sizes[f];
      while (e > 2 && e + 16 > sizes[f] && jpegs[f][e - 1] == 0) e--;
      if (e < 2 || jpegs[f][e - 2] != 0xff || jpegs[f][e - 1] != 0xd9) det->host_status[f] |= B200TAG_ST_JPEG_TRUNCATED;
    }
    const JpegFrame &fr = J.parsed[f].frame;
    if (fr.width != det->cfg.width || fr.height != det->cfg.height) {
      det->err = "frame " + std::to_string(f) + ": JPEG is " + std::to_string(fr.width) + "x" + std::to_string(fr.height) +
                 ", detector was created for " + std::to_string(det->cfg.width) + "x" + std::to_string(det->cfg.height);
      return B200TAG_E_INVALID;
    }
    int set = -1;
    for (size_t k = 0; k < set_owner.size(); k++)
      if (J.parsed[set_owner[k]].dht == J.parsed[f].dht) set = static_cast<int>(k);
    if (set < 0) {
      if (set_owner.size() >= 255) return 1;
      set = static_cast<int>(set_owner.size());
      set_owner.push_back(f);
    }
    set_of[f] = set;
    bytes += (sizes[f] - J.parsed[f].scan_begin + 15) & ~static_cast<size_t>(15);
  }
  const size_t frames_bytes = (sizeof(JpegFrame) * count + 15) & ~static_cast<size_t>(15);
  const size_t tables_bytes = (sizeof(JpegTables) * set_owner.size() + 15) & ~static_cast<size_t>(15);
  const size_t total = frames_bytes + tables_bytes + bytes + 64;
  if (total > 0x7fffffffull) return 1;
  const size_t B = static_cast<size_t>(det->cfg.max_batch);
  auto ws_layout = [&](size_t cap, size_t *chunks, size_t *subs) {
    *chunks = cap / kJpegChunk + B + 16;
    *subs = cap / (kJpegSubBits / 8) + B + 16;
  };
  if (!J.init) {  // fixed-size buffers: allocated together, committed only when all three exist
    const size_t stride = static_cast<size_t>((det->cfg.width + 31) / 32 * 32) * static_cast<size_t>((det->cfg.height + 31) / 32 * 32);
    int16_t *coef = nullptr, *dcs = nullptr;
    uint32_t *rst = nullptr;
    const cudaError_t e1 = cudaMalloc(reinterpret_cast<void **>(&coef), stride * B * sizeof(int16_t));
    const cudaError_t e2 = e1 == cudaSuccess ? cudaMalloc(reinterpret_cast<void **>(&rst), stride / 64 * B * sizeof(uint32_t)) : e1;
    const cudaError_t e3 = e2 == cudaSuccess ? cudaMalloc(reinterpret_cast<void **>(&dcs), stride / 64 * B * sizeof(int16_t)) : e2;
    if (e3 != cudaSuccess) {
      cudaFree(coef); cudaFree(rst); cudaFree(dcs);
      cudaGetLastError();
      det->err = std::string("allocating the JPEG coefficient buffers failed: ") + cudaGetErrorString(e3);
      return B200TAG_E_NOMEM;
    }
    J.coef_stride = stride; J.d_coef = coef; J.d_rst = rst; J.d_dcs = dcs;
    J.init = true;
    CK(cudaMemsetAsync(J.d_coef, 0, J.coef_stride * B * sizeof(int16_t), det->stream));
    CK(cudaMemsetAsync(J.d_dcs, 0, J.coef_stride / 64 * B * sizeof(int16_t), det->stream));
  }
  if (total > J.cap) {  // per-batch buffers grow together: the old set is released only once the new one exists
    CK(cudaStreamSynchronize(det->stream));
    const size_t want = (total + total / 2 + 4095) & ~static_cast<size_t>(4095);
    size_t chunks, subs;
    ws_layout(want, &chunks, &subs);
    uint8_t *h_block = nullptr, *d_block = nullptr, *d_ws = nullptr;
    const cudaError_t e1 = cudaHostAlloc(reinterpret_cast<void **>(&h_block), want, cudaHostAllocDefault);
    const cudaError_t e2 = e1 == cudaSuccess ? cudaMalloc(reinterpret_cast<void **>(&d_block), want) : e1;
    const cudaError_t e3 = e2 == cudaSuccess ? cudaMalloc(reinterpret_cast<void **>(&d_ws), want + subs * 16 + (2 * chunks + subs) * 4 +
                                                                                              B * (kJpegSyncRounds + 3) * 4 + 256) : e2;
    if (e3 != cudaSuccess) {
      if (h_block) cudaFreeHost(h_block);
      cudaFree(d_block); cudaFree(d_ws);
      cudaGetLastError();
      det->err = std::string("allocating the JPEG batch buffers failed: ") + cudaGetErrorString(e3);
      return B200TAG_E_NOMEM;
    }
    if (J.h_block) cudaFreeHost(J.h_block);
    if (J.d_block) cudaFree(J.d_block);
    if (J.d_ws) cudaFree(J.d_ws);
    J.h_block = h_block; J.d_block = d_block; J.d_ws = d_ws;
    J.cap = want;
  }
  JpegFrame *hf = reinterpret_cast<JpegFrame *>(J.h_block);
  JpegTables *ht = reinterpret_cast<JpegTables *>(J.h_block + frames_bytes);
  size_t off = frames_bytes + tables_bytes;
  for (size_t k = 0; k < set_owner.size(); k++) {
    if (!jpeg_build_tables(J.parsed[set_owner[k]].dht, &ht[k])) {
      det->err = "frame " + std::to_string(set_owner[k]) + ": invalid Huffman table";
      return B200TAG_E_INVALID;
    }
  }
  JpegBatch jb;
  memset(&jb, 0, sizeof(jb));
  uint32_t chunk_off = 0, sub_off = 0;
  bool any_parallel = false;
  for (int f = 0; f < count; f++) {
    const size_t n = sizes[f] - J.parsed[f].scan_begin;
    memcpy(J.h_block + off, jpegs[f] + J.parsed[f].scan_begin, n);
    hf[f] = J.parsed[f].frame;
    hf[f].data_off = static_cast<uint32_t>(off);
    hf[f].data_len = static_cast<uint32_t>(n);
    hf[f].tables = static_cast<uint8_t>(set_of[f]);
    hf[f].chunk_off = chunk_off;
    hf[f].sub_off = sub_off;
    const uint32_t nch = static_cast<uint32_t>((n + kJpegChunk - 1) / kJpegChunk);
    const uint32_t nsub = static_cast<uint32_t>((n * 8 + kJpegSubBits - 1) / kJpegSubBits) + 1;
    chunk_off += nch;
    sub_off += nsub;
    jb.max_chunks = std::max(jb.max_chunks, nch);
    jb.max_subs = std::max(jb.max_subs, nsub);
    jb.max_luma_blocks = std::max<uint32_t>(jb.max_luma_blocks, static_cast<uint32_t>(hf[f].mcus_x) * hf[f].mcus_y * hf[f].hmax * hf[f].vmax);
    any_parallel = true;
    if (hf[f].restart_interval) {
      const uint32_t nmcu = static_cast<uint32_t>(hf[f].mcus_x) * hf[f].mcus_y;
      jb.max_intervals = std::max(jb.max_intervals, (nmcu + hf[f].restart_interval - 1) / hf[f].restart_interval);
    }
    if (static_cast<size_t>(hf[f].mcus_x) * hf[f].mcus_y * hf[f].hmax * hf[f].vmax * 64 > J.coef_stride) return 1;
    off += (n + 15) & ~static_cast<size_t>(15);
  }
  size_t chunks, subs;
  ws_layout(J.cap, &chunks, &subs);
  uint8_t *w = J.d_ws;
  jb.raw = J.d_block;
  jb.clean = w; w += J.cap;
  jb.sync = reinterpret_cast<unsigned long long *>(w); w += subs * 8;
  jb.sync_in = reinterpret_cast<unsigned long long *>(w); w += subs * 8;
  jb.chunk_cnt = reinterpret_cast<uint32_t *>(w); w += chunks * 4;
  jb.chunk_rst = reinterpret_cast<uint32_t *>(w); w += chunks * 4;
  jb.nblk = reinterpret_cast<uint32_t *>(w); w += subs * 4;
  jb.changed = reinterpret_cast<uint32_t *>(w); w += B * kJpegSyncRounds * 4;
  jb.proven = reinterpret_cast<uint32_t *>(w); w += B * 4;
  jb.clean_len = reinterpret_cast<uint32_t *>(w); w += B * 4;
  jb.nrst = reinterpret_cast<uint32_t *>(w);
  jb.rst_pos = J.d_rst;
  jb.rst_stride = static_cast<uint32_t>(J.coef_stride / 64);
  jb.frames = reinterpret_cast<const JpegFrame *>(J.d_block);
  jb.tables = reinterpret_cast<const JpegTables *>(J.d_block + frames_bytes);
  jb.coef = J.d_coef;
  jb.coef_stride = J.coef_stride;
  jb.dcs = J.d_dcs;
  jb.out = det->d_in;
  jb.out_stride = det->fp.in_stride;
  jb.count = count;
  CK(cudaMemcpyAsync(J.d_block, J.h_block, off, cudaMemcpyHostToDevice, det->stream));
  // B200TAG_MJPG_DECODER=sequential keeps every frame on the warp-per-frame kernel (tests / comparison)
  const char *which = getenv("B200TAG_MJPG_DECODER");
  if (which && std::string(which) == "sequential") any_parallel = false;
  launch_jpeg_decode(jb, any_parallel, det->stream);
  J.d_proven = jb.proven;
  J.last_parallel = any_parallel;
  CK(cudaGetLastError());
  return 0;
}

int b200tag_enqueue_mjpg(b200tag_detector *det, const uint8_t *const *jpegs, const size_t *sizes, int count) {
  if (!det || !jpegs || !sizes || count < 1 || count > det->cfg.max_batch) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  if (det->cfg.format != B200TAG_FMT_GRAY8) {
    det->err = "b200tag_enqueue_mjpg needs a detector created for B200TAG_FMT_GRAY8 (the JPEG luminance plane is the image)";
    return B200TAG_E_INVALID;
  }
  if (det->pending) {
    if (int rc = finish_impl(det)) if (rc != B200TAG_E_OVERFLOW) return rc;
  }
  // B200TAG_MJPG_DECODER=nvjpeg sends everything through nvJPEG (the comparison arm of tools/bench_mjpg.py)
  const char *which = getenv("B200TAG_MJPG_DECODER");
  if (!(which && std::string(which) == "nvjpeg")) {
    const int rc = mjpg_native(det, jpegs, sizes, count);
    if (rc < 0) return rc;
    if (rc == 0) {
      det->jpeg.last_native = true;
      return enqueue_impl(det, det->d_in, det->fp.in_stride, count, nullptr, true);
    }
  }
  det->jpeg.last_native = false;
#ifdef B200TAG_HAVE_NVJPEG
  if (int rc = mjpg_open(det)) return rc;
  MjpgDecoder &m = det->mjpg;
  std::vector<nvjpegImage_t> dst(count);
  for (int f = 0; f < count; f++) {
    if (!jpegs[f] || sizes[f] == 0) return B200TAG_E_INVALID;
    int ncomp = 0, w[NVJPEG_MAX_COMPONENT] = {0}, h[NVJPEG_MAX_COMPONENT] = {0};
    nvjpegChromaSubsampling_t ss;
    if (m.image_info(m.handle, jpegs[f], sizes[f], &ncomp, &ss, w, h) != NVJPEG_STATUS_SUCCESS) {
      det->err = "frame " + std::to_string(f) + ": not a JPEG bitstream nvJPEG can parse";
      return B200TAG_E_INVALID;
    }
    if (w[0] != det->cfg.width || h[0] != det->cfg.height) {
      det->err = "frame " + std::to_string(f) + ": JPEG is " + std::to_string(w[0]) + "x" + std::to_string(h[0]) +
                 ", detector was created for " + std::to_string(det->cfg.width) + "x" + std::to_string(det->cfg.height);
      return B200TAG_E_INVALID;
    }
    memset(&dst[f], 0, sizeof(nvjpegImage_t));
    dst[f].channel[0] = det->d_in + static_cast<size_t>(f) * det->fp.in_stride;
    dst[f].pitch[0] = static_cast<size_t>(det->cfg.width);
  }
  if (m.batch != count) {
    if (m.batched_init(m.handle, m.state, count, 1, NVJPEG_OUTPUT_Y) != NVJPEG_STATUS_SUCCESS) {
      det->err = "nvjpegDecodeBatchedInitialize failed";
      return B200TAG_E_CUDA;
    }
    m.batch = count;
  }
  const nvjpegStatus_t st = m.batched(m.handle, m.state, jpegs, sizes, dst.data(), det->stream);
  if (st != NVJPEG_STATUS_SUCCESS) {
    det->err = "nvjpegDecodeBatched failed with status " + std::to_string(static_cast<int>(st));
    return st == NVJPEG_STATUS_BAD_JPEG || st == NVJPEG_STATUS_JPEG_NOT_SUPPORTED ? B200TAG_E_INVALID : B200TAG_E_CUDA;
  }
  return enqueue_impl(det, det->d_in, det->fp.in_stride, count, nullptr);
#else
  det->err = "this JPEG kind (progressive / 12-bit / arithmetic) needs nvJPEG, which this build was compiled without";
  return B200TAG_E_INVALID;
#endif
}

int b200tag_detect_mjpg(b200tag_detector *det, const uint8_t *const *jpegs, const size_t *sizes, int count) {
  if (int rc = b200tag_enqueue_mjpg(det, jpegs, sizes, count)) return rc;
  return finish_impl(det);
}

const char *b200tag_mjpg_backend(const b200tag_detector *det) {
  if (det && det->jpeg.last_native) return "native";
  if (!det || !det->mjpg.handle) return "";
#ifdef B200TAG_HAVE_NVJPEG
  switch (det->mjpg.backend) {
    case NVJPEG_BACKEND_HARDWARE: return "hardware";
    case NVJPEG_BACKEND_GPU_HYBRID: return "gpu";
    case NVJPEG_BACKEND_HYBRID: return "hybrid";
    default: return "default";
  }
#else
  return "";
#endif
}

int b200tag_jpeg_probe(const uint8_t *jpeg, size_t size, int32_t info[8], uint8_t *dht_out, size_t dht_cap, size_t *dht_len) {
  JpegParsed P;
  std::string why;
  const int rc = jpeg_parse(jpeg, size, &P, &why);
  if (rc != kJpegOk) return rc == kJpegUnsupported ? 1 : B200TAG_E_INVALID;
  if (info) {
    const JpegFrame &f = P.frame;
    const int32_t v[8] = {f.width, f.height, f.nblocks, f.hmax, f.vmax, f.restart_interval, static_cast<int32_t>(P.scan_begin),
                          f.mcus_x * f.mcus_y};
    memcpy(info, v, sizeof(v));
  }
  if (dht_len) *dht_len = P.dht.size();
  if (dht_out && dht_cap >= P.dht.size()) memcpy(dht_out, P.dht.data(), P.dht.size());
  return 0;
}

int b200tag_mjpg_parallel_frames(b200tag_detector *det, int count) {
  if (!det || count < 1 || count > det->cfg.max_batch) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  if (!det->jpeg.last_native || !det->jpeg.last_parallel) return 0;
  std::vector<uint32_t> h(count);
  CK(cudaStreamSynchronize(det->stream));
  CK(cudaMemcpy(h.data(), det->jpeg.d_proven, sizeof(uint32_t) * count, cudaMemcpyDeviceToHost));
  int n = 0;
  for (uint32_t v : h) n += v ? 1 : 0;
  return n;
}

int b200tag_debug_jpeg_model(const uint8_t *jpeg, size_t size, uint8_t *out, size_t out_cap, int *rounds) {
  return jpeg_model_decode(jpeg, size, out, out_cap, rounds);
}

int b200tag_finish(b200tag_detector *det) {
  if (!det) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  return finish_impl(det);
}

void *b200tag_stream(b200tag_detector *det) { return det ? static_cast<void *>(det->stream) : nullptr; }

int b200tag_detect_device(b200tag_detector *det, const void *device_images, size_t stride, int count) {
  if (int rc = b200tag_enqueue_device(det, device_images, stride, count)) return rc;
  return b200tag_finish(det);
}

int b200tag_detect_batch(b200tag_detector *det, const uint8_t *const *host_images, int count) {
  if (int rc = b200tag_enqueue_host(det, host_images, count)) return rc;
  return b200tag_finish(det);
}

int b200tag_detect(b200tag_detector *det, const uint8_t *host_image) {
  const uint8_t *imgs[1] = {host_image};
  return b200tag_detect_batch(det, imgs, 1);
}

const b200tag_detection *b200tag_detections(const b200tag_detector *det, int frame, int *count) {
  if (count) *count = 0;
  if (!det || frame < 0 || frame >= det->last_count || det->pending) return nullptr;
  if (count) *count = static_cast<int>(det->dets[frame].size());
  return det->dets[frame].data();
}

const b200tag_pose *b200tag_poses(const b200tag_detector *det, int frame, int *count) {
  if (count) *count = 0;
  if (!det || frame < 0 || frame >= det->last_count || det->pending || !(det->last_pose.tagsize > 0)) return nullptr;
  if (count) *count = static_cast<int>(det->poses[frame].size());
  return det->poses[frame].data();
}

const b200tag_field_pose *b200tag_field_pose_get(const b200tag_detector *det, int frame) {
  if (!det || frame < 0 || frame >= det->last_count || det->pending || !det->last_field) return nullptr;
  return &det->field_poses[frame];
}

const b200tag_floor_pose *b200tag_floor_pose_get(const b200tag_detector *det, int frame) {
  if (!det || frame < 0 || frame >= det->last_count || det->pending || !det->last_floor) return nullptr;
  return &det->floor_poses[frame];
}

const double *b200tag_floor_covariance_get(const b200tag_detector *det, int frame) {
  if (!det || frame < 0 || frame >= det->last_count || det->pending || !det->last_floor || !(det->last_pose.sigma > 0))
    return nullptr;
  return &det->floor_covs[9 * static_cast<size_t>(frame)];
}

const b200tag_covariance *b200tag_pose_covariances(const b200tag_detector *det, int frame, int *count) {
  if (count) *count = 0;
  if (!det || frame < 0 || frame >= det->last_count || det->pending || !(det->last_pose.tagsize > 0) ||
      !(det->last_pose.sigma > 0))
    return nullptr;
  if (count) *count = static_cast<int>(det->covs[frame].size());
  return det->covs[frame].data();
}

const b200tag_field_covariance *b200tag_field_covariance_get(const b200tag_detector *det, int frame) {
  if (!det || frame < 0 || frame >= det->last_count || det->pending || !det->last_field || !(det->last_pose.sigma > 0))
    return nullptr;
  return &det->field_covs[frame];
}

const b200tag_tag_position *b200tag_tag_positions(const b200tag_detector *det, int frame, int *count) {
  if (count) *count = 0;
  if (!det || frame < 0 || frame >= det->last_count || det->pending || !(det->last_pose.tagsize > 0)) return nullptr;
  if (count) *count = static_cast<int>(det->positions[frame].size());
  return det->positions[frame].data();
}

int b200tag_frame_info_get(const b200tag_detector *det, int frame, b200tag_frame_info *info) {
  if (!det || !info || frame < 0 || frame >= det->last_count || det->pending) return B200TAG_E_INVALID;
  const Counters &c = det->h_counters[frame];
  info->status = c.status | (static_cast<size_t>(frame) < det->host_status.size() ? det->host_status[frame] : 0u);
  info->num_points = std::min(c.num_points, det->fp.point_cap);
  info->num_clusters = alloc_clusters(c.alloc);
  info->num_blobs = c.num_selected_blobs;
  info->num_selected_points = c.num_selected_points;
  info->num_fit_quads = std::min(c.num_fit_quads, det->fp.blob_cap);
  info->num_quads = std::min(c.num_quads, det->fp.quad_cap);
  info->num_detections = std::min(c.num_detections, det->fp.det_cap);
  return 0;
}

const b200tag_quad *b200tag_quads(const b200tag_detector *cdet, int frame, int *count) {
  if (count) *count = 0;
  b200tag_detector *det = const_cast<b200tag_detector *>(cdet);
  if (!det || frame < 0 || frame >= det->last_count || det->pending) return nullptr;
  DeviceGuard on_device(det->device);
  if (!det->quads_valid[frame]) {
    const uint32_t nq = std::min(det->h_counters[frame].num_quads, det->fp.quad_cap);
    det->quads[frame].resize(nq);
    if (nq) {
      if (cudaMemcpy(det->quads[frame].data(), det->fp.quads + static_cast<size_t>(frame) * det->fp.quad_cap,
                     nq * sizeof(b200tag_quad), cudaMemcpyDeviceToHost) != cudaSuccess)
        return nullptr;
      std::sort(det->quads[frame].begin(), det->quads[frame].end(), [](const b200tag_quad &a, const b200tag_quad &b) {
        return a.rep0 != b.rep0 ? a.rep0 < b.rep0 : a.rep1 < b.rep1;
      });
    }
    det->quads_valid[frame] = true;
  }
  if (count) *count = static_cast<int>(det->quads[frame].size());
  return det->quads[frame].data();
}

int b200tag_copy_stage(b200tag_detector *det, int frame, int stage, void *dst, size_t cap, size_t *out_bytes) {
  if (!det || frame < 0 || frame >= det->last_count || det->pending) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  const FrameParams &p = det->fp;
  const Counters &c = det->h_counters[frame];
  const size_t N = static_cast<size_t>(p.W) * p.H, n = static_cast<size_t>(p.w) * p.h;
  const size_t tiles = static_cast<size_t>(p.tiles_x) * p.tiles_y;
  const size_t f = static_cast<size_t>(frame);
  const void *src = nullptr;
  size_t bytes = 0;
  const uint32_t np = std::min(c.num_points, p.point_cap);
  const uint32_t nsel = std::min(c.num_seg_points, p.point_cap);  // segments of all candidate blobs
  switch (stage) {
    case B200TAG_STAGE_GRAY:
      if (det->cfg.format == B200TAG_FMT_GRAY8) {
        // the gray image is the input itself: available while it sits in the detector's own staging buffer
        // (host frames, decoded JPEG luminance), not for caller-owned device frames
        if (det->last_images != det->d_in) return B200TAG_E_INVALID;
        src = det->d_in + f * det->last_stride; bytes = N; break;
      }
      src = p.gray + f * N; bytes = N; break;
    case B200TAG_STAGE_QUAD_IMAGE: src = p.quad + f * n; bytes = n; break;
    case B200TAG_STAGE_THRESHOLD: src = p.thresh + f * n; bytes = n; break;
    case B200TAG_STAGE_LABELS: {  // label words carry colour / size flags in their top bits (dev_types.h): strip them
      bytes = n * 4;
      if (out_bytes) *out_bytes = bytes;
      if (!dst) return 0;
      if (cap < bytes) return B200TAG_E_INVALID;
      CK(cudaMemcpy(dst, p.labels + f * n, bytes, cudaMemcpyDeviceToHost));
      uint32_t *o = static_cast<uint32_t *>(dst);
      for (size_t i = 0; i < n; i++) o[i] &= 0x0fffffffu;
      return 0;
    }
    case B200TAG_STAGE_SIZES: src = p.sizes + f * n; bytes = n * 4; break;
    case B200TAG_STAGE_MINMAX:
      if (!p.keep_stages) return B200TAG_E_INVALID;
      src = p.minmax + f * tiles * 2; bytes = tiles * 2; break;
    case B200TAG_STAGE_POINTS: {
      bytes = static_cast<size_t>(np) * sizeof(b200tag_point);
      if (out_bytes) *out_bytes = bytes;
      if (!dst) return 0;
      if (cap < bytes) return B200TAG_E_INVALID;
      std::vector<uint64_t> raw(np);
      if (np) CK(cudaMemcpy(raw.data(), p.points + f * p.point_cap, np * 8ull, cudaMemcpyDeviceToHost));
      b200tag_point *o = static_cast<b200tag_point *>(dst);
      for (uint32_t i = 0; i < np; i++) {
        const uint32_t sp = point_seg(raw[i]);
        o[i].slot = point_slot(raw[i]);
        o[i].x = static_cast<uint16_t>(sp_x(sp));
        o[i].y = static_cast<uint16_t>(sp_y(sp));
        o[i].dir = static_cast<uint8_t>(sp_dir(sp));
        o[i].black_to_white = static_cast<uint8_t>(sp_b2w(sp));
        o[i].pad[0] = o[i].pad[1] = 0;
      }
      return 0;
    }
    case B200TAG_STAGE_BLOBS: src = p.blobs + f * p.blob_cap; bytes = std::min(alloc_blobs(c.alloc), p.blob_cap) * sizeof(b200tag_blob); break;
    case B200TAG_STAGE_CLUSTERS:
      if (!p.clusters) return B200TAG_E_INVALID;
      src = p.clusters + f * p.cluster_cap; bytes = std::min(alloc_clusters(c.alloc), p.cluster_cap) * sizeof(b200tag_blob); break;
    case B200TAG_STAGE_SORTED_POINTS: src = p.seg_keys + f * p.point_cap; bytes = nsel * 8ull; break;
    case B200TAG_STAGE_LINE_FIT_POINTS: src = p.lfp + f * p.point_cap; bytes = nsel * sizeof(b200tag_lfp); break;
    case B200TAG_STAGE_ERRORS: src = p.errs + f * p.point_cap; bytes = nsel * 4ull; break;
    case B200TAG_STAGE_FILTERED_ERRORS: src = p.filt + f * p.point_cap; bytes = nsel * 8ull; break;
    case B200TAG_STAGE_FIT_QUADS: src = p.fit_quads + f * p.blob_cap; bytes = std::min(c.num_fit_quads, p.blob_cap) * sizeof(b200tag_fit_quad); break;
    case B200TAG_STAGE_QUADS: src = p.quads + f * p.quad_cap; bytes = std::min(c.num_quads, p.quad_cap) * sizeof(b200tag_quad); break;
    case B200TAG_STAGE_RAW_DETECTIONS: {
      bytes = std::min(c.num_detections, p.det_cap) * sizeof(b200tag_detection);
      if (out_bytes) *out_bytes = bytes;
      if (!dst) return 0;
      if (cap < bytes) return B200TAG_E_INVALID;
      memcpy(dst, det->h_dets + f * p.det_cap, bytes);
      return 0;
    }
    default: return B200TAG_E_INVALID;
  }
  if (out_bytes) *out_bytes = bytes;
  if (!dst) return 0;
  if (cap < bytes) return B200TAG_E_INVALID;
  if (bytes) CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
  return 0;
}

int b200tag_set_camera(b200tag_detector *det, double fx, double cx, double fy, double cy) {
  if (!det) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  drop_graphs(det);  // the parameters are baked into the captured launches
  det->cfg.fx = det->fp.fx = fx; det->cfg.cx = det->fp.cx = cx;
  det->cfg.fy = det->fp.fy = fy; det->cfg.cy = det->fp.cy = cy;
  return 0;
}

int b200tag_set_pose_estimation(b200tag_detector *det, double tagsize, double fx, double fy, double cx, double cy,
                                const double *rotation, const double *offset) {
  if (!det || !(tagsize >= 0) || fx == 0 || fy == 0) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  if (tagsize > 0 && !det->h_poses) {
    const size_t bytes = sizeof(b200tag_pose) * det->fp.det_cap * static_cast<size_t>(det->cfg.max_batch);
    b200tag_pose *h = nullptr, *d = nullptr;
    CK(cudaHostAlloc(reinterpret_cast<void **>(&h), bytes, cudaHostAllocMapped));
    if (cudaHostGetDevicePointer(reinterpret_cast<void **>(&d), h, 0) != cudaSuccess) {
      cudaGetLastError();
      cudaFreeHost(h);
      det->err = "cudaHostGetDevicePointer(poses) failed";
      return B200TAG_E_CUDA;
    }
    det->h_poses = h;
    det->d_poses_alias = d;
  }
  drop_graphs(det);  // the parameters are baked into the captured launches
  b200tag_detector::PoseSettings &ps = det->pose;
  ps.tagsize = tagsize; ps.fx = fx; ps.fy = fy; ps.cx = cx; ps.cy = cy;
  static const double kEye[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, kZero[3] = {0, 0, 0};
  memcpy(ps.rotation, rotation ? rotation : kEye, sizeof(ps.rotation));
  memcpy(ps.offset, offset ? offset : kZero, sizeof(ps.offset));
  return 0;
}

int b200tag_set_field_layout(b200tag_detector *det, const b200tag_field_tag *layout, int count) {
  if (!det) return B200TAG_E_INVALID;
  std::vector<pose::FieldKey> keys(static_cast<size_t>(std::max(count, 0)));
  if (!field_layout_keys(layout, count, det->family_ncodes.data(), static_cast<int>(det->family_ncodes.size()), keys.data())) {
    det->err = "invalid field layout";
    return B200TAG_E_INVALID;
  }
  DeviceGuard on_device(det->device);
  if (count > 0 && !det->h_field) {
    const size_t B = static_cast<size_t>(det->cfg.max_batch);
    const uint32_t stride = std::min<uint32_t>(det->fp.det_cap, B200TAG_MAX_FIELD_TAGS);
    void *dl = nullptr, *dk = nullptr, *ds = nullptr;
    b200tag_field_pose *h = nullptr, *d = nullptr;
    const bool ok = cudaMalloc(&dl, sizeof(b200tag_field_tag) * B200TAG_MAX_FIELD_TAGS) == cudaSuccess &&
                    cudaMalloc(&dk, sizeof(pose::FieldKey) * B200TAG_MAX_FIELD_TAGS) == cudaSuccess &&
                    cudaMalloc(&ds, field_tag_bytes() * stride * B) == cudaSuccess &&
                    cudaHostAlloc(reinterpret_cast<void **>(&h), sizeof(b200tag_field_pose) * B, cudaHostAllocMapped) == cudaSuccess &&
                    cudaHostGetDevicePointer(reinterpret_cast<void **>(&d), h, 0) == cudaSuccess;
    if (!ok) {
      cudaGetLastError();
      cudaFree(dl);
      cudaFree(dk);
      cudaFree(ds);
      if (h) cudaFreeHost(h);
      det->err = "allocating the field pose buffers failed";
      return B200TAG_E_CUDA;
    }
    det->d_field_layout = static_cast<b200tag_field_tag *>(dl);
    det->d_field_keys = static_cast<pose::FieldKey *>(dk);
    det->d_field_scratch = ds;
    det->field_scratch_stride = stride;
    det->h_field = h;
    det->d_field_alias = d;
  }
  if (count > 0) {  // stream-ordered: a batch in flight reads the old layout to its end
    CK(cudaMemcpyAsync(det->d_field_layout, layout, sizeof(b200tag_field_tag) * count, cudaMemcpyHostToDevice, det->stream));
    CK(cudaMemcpyAsync(det->d_field_keys, keys.data(), sizeof(pose::FieldKey) * count, cudaMemcpyHostToDevice, det->stream));
  }
  drop_graphs(det);  // the layout size is baked into the captured launches
  det->field_n = count;
  return 0;
}

int b200tag_set_pose_method(b200tag_detector *det, int method) {
  if (!det || (method != B200TAG_POSE_ORTHOGONAL_ITERATION && method != B200TAG_POSE_IPPE)) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  drop_graphs(det);  // the kernel is baked into the captured launches
  det->pose.method = method;
  return 0;
}

int b200tag_set_pose_distortion(b200tag_detector *det, const double *dist) {
  bool active;
  pose::Distortion D;
  if (!det || !read_distortion(dist, &active, &D)) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  drop_graphs(det);  // the kernel variant and the coefficients are baked into the captured launches
  const double c[5] = {D.k1, D.k2, D.p1, D.p2, D.k3};
  memcpy(det->pose.dist, c, sizeof(c));
  return 0;
}

int b200tag_set_pose_covariance(b200tag_detector *det, double sigma) {
  if (!det || !(sigma == 0 || valid_sigma(sigma))) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  if (sigma > 0 && !det->h_cov) {
    const size_t B = static_cast<size_t>(det->cfg.max_batch);
    b200tag_covariance *h = nullptr, *d = nullptr;
    b200tag_field_covariance *hf = nullptr, *df = nullptr;
    const bool ok = cudaHostAlloc(reinterpret_cast<void **>(&h), sizeof(b200tag_covariance) * det->fp.det_cap * B, cudaHostAllocMapped) == cudaSuccess &&
                    cudaHostGetDevicePointer(reinterpret_cast<void **>(&d), h, 0) == cudaSuccess &&
                    cudaHostAlloc(reinterpret_cast<void **>(&hf), sizeof(b200tag_field_covariance) * B, cudaHostAllocMapped) == cudaSuccess &&
                    cudaHostGetDevicePointer(reinterpret_cast<void **>(&df), hf, 0) == cudaSuccess;
    if (!ok) {
      cudaGetLastError();
      if (h) cudaFreeHost(h);
      if (hf) cudaFreeHost(hf);
      det->err = "allocating the covariance buffers failed";
      return B200TAG_E_CUDA;
    }
    det->h_cov = h;
    det->d_cov_alias = d;
    det->h_field_cov = hf;
    det->d_field_cov_alias = df;
  }
  drop_graphs(det);  // the kernels and sigma are baked into the captured launches
  det->pose.sigma = sigma;
  return 0;
}

int b200tag_set_floor_pose(b200tag_detector *det, double heading_weight) {
  if (!det || !(heading_weight == 0 || heading_weight > 0)) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  if (heading_weight > 0 && !det->h_floor) {
    const size_t B = static_cast<size_t>(det->cfg.max_batch);
    b200tag_floor_pose *h = nullptr, *d = nullptr;
    double *hc = nullptr, *dc = nullptr, *hg = nullptr, *dg = nullptr;
    const bool ok = cudaHostAlloc(reinterpret_cast<void **>(&h), sizeof(b200tag_floor_pose) * B, cudaHostAllocMapped) == cudaSuccess &&
                    cudaHostGetDevicePointer(reinterpret_cast<void **>(&d), h, 0) == cudaSuccess &&
                    cudaHostAlloc(reinterpret_cast<void **>(&hc), sizeof(double) * 9 * B, cudaHostAllocMapped) == cudaSuccess &&
                    cudaHostGetDevicePointer(reinterpret_cast<void **>(&dc), hc, 0) == cudaSuccess &&
                    cudaHostAlloc(reinterpret_cast<void **>(&hg), sizeof(double) * 2 * B, cudaHostAllocMapped) == cudaSuccess &&
                    cudaHostGetDevicePointer(reinterpret_cast<void **>(&dg), hg, 0) == cudaSuccess;
    if (!ok) {
      cudaGetLastError();
      if (h) cudaFreeHost(h);
      if (hc) cudaFreeHost(hc);
      if (hg) cudaFreeHost(hg);
      det->err = "allocating the floor pose buffers failed";
      return B200TAG_E_CUDA;
    }
    det->h_floor = h;
    det->d_floor_alias = d;
    det->h_floor_cov = hc;
    det->d_floor_cov_alias = dc;
    det->h_gyro = hg;
    det->d_gyro_alias = dg;
  }
  drop_graphs(det);  // the kernel and the weight are baked into the captured launches
  det->floor_weight = heading_weight;
  return 0;
}

int b200tag_set_robot_headings(b200tag_detector *det, const double *heading, int count) {
  if (!det || count < 0 || count > det->cfg.max_batch || (count > 0 && !heading)) return B200TAG_E_INVALID;
  for (int f = 0; f < count; f++)
    if (std::isinf(heading[f])) return B200TAG_E_INVALID;
  det->next_gyro.resize(2 * static_cast<size_t>(count));
  for (int f = 0; f < count; f++) floor_gyro(heading[f], &det->next_gyro[2 * f], &det->next_gyro[2 * f + 1]);
  det->next_gyro_set = true;
  return 0;
}

int b200tag_set_distortion(b200tag_detector *det, double k1, double k2, double p1, double p2, double k3) {
  if (!det) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  drop_graphs(det);
  det->cfg.k1 = det->fp.k1 = k1; det->cfg.k2 = det->fp.k2 = k2; det->cfg.p1 = det->fp.p1 = p1;
  det->cfg.p2 = det->fp.p2 = p2; det->cfg.k3 = det->fp.k3 = k3;
  return 0;
}

int b200tag_undistort(double *u, double *v, double fx, double cx, double fy, double cy, double k1, double k2, double p1,
                      double p2, double k3) {
  // GpuDetector::UnDistort, apriltag_detect.cu:335-402
  if (!u || !v) return B200TAG_E_INVALID;
  int converged = 1;
  const double xPP = (*u - cx) / fx, yPP = (*v - cy) / fy;
  double xP = xPP, yP = yPP;
  const double x0 = xP, y0 = yP;
  double prev_x = 0, prev_y = 0;
  int iterations = 0;
  do {
    prev_x = xP;
    prev_y = yP;
    const double rSq = xP * xP + yP * yP;
    const double radial = 1 + (k1 * rSq) + (k2 * rSq * rSq) + (k3 * rSq * rSq * rSq);
    const double radial_inv = 1 / radial;
    const double tdx = 2 * p1 * xP * yP + p2 * (rSq + k3 * rSq * rSq * rSq);
    const double tdy = p1 * (rSq + 2 * yP * yP) + 2 * p2 * xP * yP;
    xP = (x0 - tdx) * radial_inv;
    yP = (y0 - tdy) * radial_inv;
    if (iterations > 100) { converged = 0; break; }
    iterations++;
  } while (std::fabs(xP - prev_x) > 1e-6 || std::fabs(yP - prev_y) > 1e-6);
  *u = xP * fx + cx;
  *v = yP * fy + cy;
  return converged;
}

void *b200tag_alloc_pinned(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}

void *b200tag_alloc_pinned_wc(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocWriteCombined) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}

void b200tag_free_pinned(void *p) {
  if (p) cudaFreeHost(p);
}

int b200tag_debug_math(int op, const float *a, const float *b, float *out, int n) {
  if (!a || !b || !out || n <= 0 || (op != 0 && op != 1)) return B200TAG_E_INVALID;
  float *d = nullptr;
  if (cudaMalloc(&d, sizeof(float) * 3 * static_cast<size_t>(n)) != cudaSuccess) {
    cudaGetLastError();
    return B200TAG_E_NO_DEVICE;
  }
  int rc = 0;
  if (cudaMemcpy(d, a, sizeof(float) * n, cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(d + n, b, sizeof(float) * n, cudaMemcpyHostToDevice) != cudaSuccess)
    rc = B200TAG_E_CUDA;
  if (!rc) {
    b200tag::k_debug_math<<<(n + 255) / 256, 256>>>(op, d, d + n, d + 2 * static_cast<size_t>(n), n);
    if (cudaMemcpy(out, d + 2 * static_cast<size_t>(n), sizeof(float) * n, cudaMemcpyDeviceToHost) != cudaSuccess) rc = B200TAG_E_CUDA;
  }
  cudaFree(d);
  return rc;
}

}  // extern "C"

namespace {

// The test hooks' common part: the pose kernel of `method` on caller records, through device copies of them.
int estimate_poses_device(int method, const b200tag_detection *dets, int count, double tagsize, double fx, double fy,
                          double cx, double cy, const double *dist, b200tag_pose *out) {
  bool active;
  pose::Distortion D;
  if (count < 0 || (count > 0 && (!dets || !out)) || !(tagsize > 0) || fx == 0 || fy == 0) return B200TAG_E_INVALID;
  if ((method != B200TAG_POSE_ORTHOGONAL_ITERATION && method != B200TAG_POSE_IPPE) || !read_distortion(dist, &active, &D))
    return B200TAG_E_INVALID;
  if (count == 0) return 0;
  const size_t db = sizeof(b200tag_detection) * static_cast<size_t>(count), pb = sizeof(b200tag_pose) * static_cast<size_t>(count);
  uint8_t *d = nullptr;
  if (cudaMalloc(&d, db + pb) != cudaSuccess) {
    cudaGetLastError();
    return B200TAG_E_NO_DEVICE;
  }
  int rc = 0;
  const PoseLaunch pl{reinterpret_cast<const b200tag_detection *>(d), reinterpret_cast<b200tag_pose *>(d + db), nullptr,
                      0, static_cast<uint32_t>(count), tagsize, fx, fy, cx, cy, method, {D.k1, D.k2, D.p1, D.p2, D.k3}};
  if (cudaMemcpy(d, dets, db, cudaMemcpyHostToDevice) != cudaSuccess) rc = B200TAG_E_CUDA;
  if (!rc) {
    Launcher ln{nullptr, nullptr};
    launch_pose(pl, 1, ln);
    if (cudaGetLastError() != cudaSuccess || cudaMemcpy(out, d + db, pb, cudaMemcpyDeviceToHost) != cudaSuccess) rc = B200TAG_E_CUDA;
  }
  cudaFree(d);
  return rc;
}

// The field hook's common part: k_field_pose on one caller list; with sigma > 0 the variant with the covariance.
int field_pose_device(const b200tag_detection *dets, int count, const b200tag_field_tag *layout, int nlayout,
                      double tagsize, double fx, double fy, double cx, double cy, const double *dist,
                      const double *rotation, const double *offset, double sigma, b200tag_field_pose *out,
                      b200tag_field_covariance *cov) {
  bool active;
  pose::Distortion D;
  if (count < 0 || (count > 0 && !dets) || !out || !(tagsize > 0) || fx == 0 || fy == 0) return B200TAG_E_INVALID;
  if (!read_distortion(dist, &active, &D)) return B200TAG_E_INVALID;
  std::vector<pose::FieldKey> keys(static_cast<size_t>(std::max(nlayout, 0)));
  if (!field_layout_keys(layout, nlayout, nullptr, 0, keys.data())) return B200TAG_E_INVALID;
  const size_t db = sizeof(b200tag_detection) * static_cast<size_t>(count), lb = sizeof(b200tag_field_tag) * nlayout,
               kb = sizeof(pose::FieldKey) * nlayout, sb = field_tag_bytes() * std::max(count, 1);
  const size_t o_l = align_up(db, 256), o_k = align_up(o_l + lb, 256), o_s = align_up(o_k + kb, 256), o_o = align_up(o_s + sb, 256);
  const size_t o_c = align_up(o_o + sizeof(b200tag_field_pose), 256);
  uint8_t *d = nullptr;
  if (cudaMalloc(&d, o_c + (cov ? sizeof(b200tag_field_covariance) : 0)) != cudaSuccess) {
    cudaGetLastError();
    return B200TAG_E_NO_DEVICE;
  }
  static const double kEye[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, kZero[3] = {0, 0, 0};
  FieldLaunch fl{reinterpret_cast<const b200tag_detection *>(d), nullptr, 0, static_cast<uint32_t>(count),
                 reinterpret_cast<const b200tag_field_tag *>(d + o_l), reinterpret_cast<const pose::FieldKey *>(d + o_k), nlayout,
                 reinterpret_cast<pose::FieldTagData *>(d + o_s), 0, tagsize, fx, fy, cx, cy, {}, {},
                 reinterpret_cast<b200tag_field_pose *>(d + o_o), {D.k1, D.k2, D.p1, D.p2, D.k3},
                 cov ? reinterpret_cast<b200tag_field_covariance *>(d + o_c) : nullptr, cov ? sigma : 0};
  memcpy(fl.rotation, rotation ? rotation : kEye, sizeof(fl.rotation));
  memcpy(fl.offset, offset ? offset : kZero, sizeof(fl.offset));
  int rc = 0;
  if ((db && cudaMemcpy(d, dets, db, cudaMemcpyHostToDevice) != cudaSuccess) ||
      (lb && cudaMemcpy(d + o_l, layout, lb, cudaMemcpyHostToDevice) != cudaSuccess) ||
      (kb && cudaMemcpy(d + o_k, keys.data(), kb, cudaMemcpyHostToDevice) != cudaSuccess))
    rc = B200TAG_E_CUDA;
  if (!rc) {
    Launcher ln{nullptr, nullptr};
    launch_field_pose(fl, 1, ln);
    if (cudaGetLastError() != cudaSuccess || cudaMemcpy(out, d + o_o, sizeof(*out), cudaMemcpyDeviceToHost) != cudaSuccess ||
        (cov && cudaMemcpy(cov, d + o_c, sizeof(*cov), cudaMemcpyDeviceToHost) != cudaSuccess))
      rc = B200TAG_E_CUDA;
  }
  cudaFree(d);
  return rc;
}

// The floor hook: k_field_pose (for its scratch) and k_floor_pose on one caller list.
int floor_pose_device(const b200tag_detection *dets, int count, const b200tag_field_tag *layout, int nlayout,
                      double tagsize, double fx, double fy, double cx, double cy, const double *dist,
                      const double *rotation, const double *offset, double heading, double heading_weight, double sigma,
                      b200tag_floor_pose *out, double *cov) {
  bool active;
  pose::Distortion D;
  pose::FloorModel m;
  if (!read_distortion(dist, &active, &D) || !floor_model(rotation, offset, heading, heading_weight, &m))
    return B200TAG_E_INVALID;
  if (!(sigma == 0 || valid_sigma(sigma)) || (sigma > 0 && !cov)) return B200TAG_E_INVALID;
  if (count < 0 || (count > 0 && !dets) || !out || !(tagsize > 0) || fx == 0 || fy == 0) return B200TAG_E_INVALID;
  std::vector<pose::FieldKey> keys(static_cast<size_t>(std::max(nlayout, 0)));
  if (!field_layout_keys(layout, nlayout, nullptr, 0, keys.data())) return B200TAG_E_INVALID;
  const size_t db = sizeof(b200tag_detection) * static_cast<size_t>(count), lb = sizeof(b200tag_field_tag) * nlayout,
               kb = sizeof(pose::FieldKey) * nlayout, sb = field_tag_bytes() * std::max(count, 1);
  const size_t o_l = align_up(db, 256), o_k = align_up(o_l + lb, 256), o_s = align_up(o_k + kb, 256), o_o = align_up(o_s + sb, 256);
  const size_t o_g = align_up(o_o + sizeof(b200tag_field_pose), 256), o_f = align_up(o_g + 2 * sizeof(double), 256);
  const size_t o_c = align_up(o_f + sizeof(b200tag_floor_pose), 256);
  uint8_t *d = nullptr;
  if (cudaMalloc(&d, o_c + 9 * sizeof(double)) != cudaSuccess) {
    cudaGetLastError();
    return B200TAG_E_NO_DEVICE;
  }
  const double gyro[2] = {m.cg, m.sg};
  FieldLaunch fl{reinterpret_cast<const b200tag_detection *>(d), nullptr, 0, static_cast<uint32_t>(count),
                 reinterpret_cast<const b200tag_field_tag *>(d + o_l), reinterpret_cast<const pose::FieldKey *>(d + o_k), nlayout,
                 reinterpret_cast<pose::FieldTagData *>(d + o_s), 0, tagsize, fx, fy, cx, cy, {}, {},
                 reinterpret_cast<b200tag_field_pose *>(d + o_o), {D.k1, D.k2, D.p1, D.p2, D.k3}, nullptr, 0};
  memcpy(fl.rotation, m.rot, sizeof(fl.rotation));
  memcpy(fl.offset, m.off, sizeof(fl.offset));
  FloorLaunch gl{fl.scratch, 0, fl.out, reinterpret_cast<const double *>(d + o_g), heading_weight, fx, fy, cx, cy, {}, {},
                 {D.k1, D.k2, D.p1, D.p2, D.k3}, reinterpret_cast<b200tag_floor_pose *>(d + o_f),
                 reinterpret_cast<double *>(d + o_c), sigma};
  memcpy(gl.rotation, m.rot, sizeof(gl.rotation));
  memcpy(gl.offset, m.off, sizeof(gl.offset));
  int rc = 0;
  if ((db && cudaMemcpy(d, dets, db, cudaMemcpyHostToDevice) != cudaSuccess) ||
      (lb && cudaMemcpy(d + o_l, layout, lb, cudaMemcpyHostToDevice) != cudaSuccess) ||
      (kb && cudaMemcpy(d + o_k, keys.data(), kb, cudaMemcpyHostToDevice) != cudaSuccess) ||
      cudaMemcpy(d + o_g, gyro, sizeof(gyro), cudaMemcpyHostToDevice) != cudaSuccess)
    rc = B200TAG_E_CUDA;
  if (!rc) {
    Launcher ln{nullptr, nullptr};
    launch_field_pose(fl, 1, ln);
    launch_floor_pose(gl, 1, ln);
    if (cudaGetLastError() != cudaSuccess || cudaMemcpy(out, d + o_f, sizeof(*out), cudaMemcpyDeviceToHost) != cudaSuccess ||
        (sigma > 0 && cudaMemcpy(cov, d + o_c, 9 * sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess))
      rc = B200TAG_E_CUDA;
    else
      out->heading = std::atan2(out->sin_heading, out->cos_heading);
  }
  cudaFree(d);
  return rc;
}

}  // namespace

extern "C" {

int b200tag_debug_floor_pose_device(const b200tag_detection *dets, int count, const b200tag_field_tag *layout,
                                    int nlayout, double tagsize, double fx, double fy, double cx, double cy,
                                    const double *dist, const double *rotation, const double *offset, double heading,
                                    double heading_weight, double sigma, b200tag_floor_pose *out, double cov[9]) {
  return floor_pose_device(dets, count, layout, nlayout, tagsize, fx, fy, cx, cy, dist, rotation, offset, heading,
                           heading_weight, sigma, out, cov);
}

int b200tag_debug_estimate_poses_device(const b200tag_detection *dets, int count, double tagsize, double fx, double fy,
                                        double cx, double cy, b200tag_pose *out) {
  return estimate_poses_device(B200TAG_POSE_ORTHOGONAL_ITERATION, dets, count, tagsize, fx, fy, cx, cy, nullptr, out);
}

int b200tag_debug_estimate_poses_ippe_device(const b200tag_detection *dets, int count, double tagsize, double fx,
                                             double fy, double cx, double cy, b200tag_pose *out) {
  return estimate_poses_device(B200TAG_POSE_IPPE, dets, count, tagsize, fx, fy, cx, cy, nullptr, out);
}

int b200tag_debug_estimate_poses_distorted_device(int method, const b200tag_detection *dets, int count, double tagsize,
                                                  double fx, double fy, double cx, double cy, const double *dist,
                                                  b200tag_pose *out) {
  return estimate_poses_device(method, dets, count, tagsize, fx, fy, cx, cy, dist, out);
}

int b200tag_debug_estimate_field_pose_device(const b200tag_detection *dets, int count, const b200tag_field_tag *layout,
                                             int nlayout, double tagsize, double fx, double fy, double cx, double cy,
                                             const double *rotation, const double *offset, b200tag_field_pose *out) {
  return b200tag_debug_estimate_field_pose_distorted_device(dets, count, layout, nlayout, tagsize, fx, fy, cx, cy, nullptr,
                                                            rotation, offset, out);
}

int b200tag_debug_estimate_field_pose_distorted_device(const b200tag_detection *dets, int count,
                                                       const b200tag_field_tag *layout, int nlayout, double tagsize,
                                                       double fx, double fy, double cx, double cy, const double *dist,
                                                       const double *rotation, const double *offset,
                                                       b200tag_field_pose *out) {
  return field_pose_device(dets, count, layout, nlayout, tagsize, fx, fy, cx, cy, dist, rotation, offset, 0, out, nullptr);
}

int b200tag_debug_field_pose_covariance_device(const b200tag_detection *dets, int count, const b200tag_field_tag *layout,
                                               int nlayout, double tagsize, double fx, double fy, double cx, double cy,
                                               const double *dist, const double *rotation, const double *offset,
                                               double sigma, b200tag_field_pose *out, b200tag_field_covariance *cov) {
  if (!valid_sigma(sigma) || !cov) return B200TAG_E_INVALID;
  return field_pose_device(dets, count, layout, nlayout, tagsize, fx, fy, cx, cy, dist, rotation, offset, sigma, out, cov);
}

int b200tag_debug_pose_covariances_device(const b200tag_detection *dets, const b200tag_pose *poses, int count,
                                          double tagsize, double fx, double fy, double cx, double cy, const double *dist,
                                          double sigma, b200tag_covariance *out) {
  bool active;
  pose::Distortion D;
  if (!valid_sigma(sigma) || !read_distortion(dist, &active, &D)) return B200TAG_E_INVALID;
  if (count < 0 || (count > 0 && (!dets || !poses || !out))) return B200TAG_E_INVALID;
  if (count > 0 && (!(tagsize > 0) || fx == 0 || fy == 0)) return B200TAG_E_INVALID;
  if (count == 0) return 0;
  const size_t db = sizeof(b200tag_detection) * static_cast<size_t>(count), pb = sizeof(b200tag_pose) * static_cast<size_t>(count),
               cb = sizeof(b200tag_covariance) * static_cast<size_t>(count);
  uint8_t *d = nullptr;
  if (cudaMalloc(&d, db + pb + cb) != cudaSuccess) {
    cudaGetLastError();
    return B200TAG_E_NO_DEVICE;
  }
  int rc = 0;
  const PoseLaunch pl{reinterpret_cast<const b200tag_detection *>(d), reinterpret_cast<b200tag_pose *>(d + db), nullptr,
                      0, static_cast<uint32_t>(count), tagsize, fx, fy, cx, cy, B200TAG_POSE_IPPE, {D.k1, D.k2, D.p1, D.p2, D.k3}};
  if (cudaMemcpy(d, dets, db, cudaMemcpyHostToDevice) != cudaSuccess || cudaMemcpy(d + db, poses, pb, cudaMemcpyHostToDevice) != cudaSuccess)
    rc = B200TAG_E_CUDA;
  if (!rc) {
    Launcher ln{nullptr, nullptr};
    launch_pose_cov(pl, reinterpret_cast<b200tag_covariance *>(d + db + pb), sigma, 1, ln);
    if (cudaGetLastError() != cudaSuccess || cudaMemcpy(out, d + db + pb, cb, cudaMemcpyDeviceToHost) != cudaSuccess) rc = B200TAG_E_CUDA;
  }
  cudaFree(d);
  return rc;
}

int b200tag_kernels_per_batch(const b200tag_detector *det) { return det ? det->kernels_per_batch : 0; }

int b200tag_profile_device(b200tag_detector *det, const void *device_images, size_t stride, int count, int iters,
                           const char **names, float *ms, int cap, int *n_out) {
  if (!det || !device_images || count < 1 || count > det->cfg.max_batch || iters < 1) return B200TAG_E_INVALID;
  DeviceGuard on_device(det->device);
  if (det->pending) finish_impl(det);
  std::vector<double> acc;
  for (int it = 0; it < iters; it++) {
    det->timer.rewind();
    if (int rc = enqueue_impl(det, device_images, stride, count, &det->timer)) return rc;
    CK(cudaStreamSynchronize(det->stream));
    const size_t ns = det->timer.cursor;
    if (acc.size() < ns) acc.resize(ns, 0.0);
    for (size_t i = 0; i < ns; i++) {
      float t = 0;
      CK(cudaEventElapsedTime(&t, det->timer.spans[i].a, det->timer.spans[i].b));
      acc[i] += t;
    }
  }
  finish_impl(det);
  const int ns = static_cast<int>(acc.size());
  if (n_out) *n_out = ns;
  for (int i = 0; i < ns && i < cap; i++) {
    if (names) names[i] = det->timer.spans[i].name;
    if (ms) ms[i] = static_cast<float>(acc[i] / iters);
  }
  return 0;
}

}  // extern "C"
