// The pose step on the device (b200tag_set_pose_estimation): libapriltag's estimate_tag_pose for every raw detection of
// the batch, appended to the detection graph behind k_decode.  One warp per detection.  The homography start and the
// orthogonal iteration run on every lane with the same values, reading the per-detection constants from shared memory;
// lane 0 sets up the frame of the second-minimum search there, and the lanes split that search's grid.  The arithmetic is
// pose_core.h's, the same the host functions in pose.cc run.  With b200tag_set_pose_method(B200TAG_POSE_IPPE) the step
// is k_pose_ippe instead: the closed-form IPPE pose, one thread per detection.  With b200tag_set_pose_distortion each
// kernel's variant with kDistorted = true runs: it undistorts the corners first (pose_core.h's undistort_point); the
// variant without compiles to the kernel without the step.  With b200tag_set_pose_covariance, k_pose_cov runs behind
// either pose kernel and writes every pose's covariance.  With b200tag_set_floor_pose, k_floor_pose runs behind
// k_field_pose and fits the robot's (x, y, heading) on the floor to the same corners.
//
// A pose depends only on its own record, so computing it before the host's reconcile gives the pose of every
// detection that survives it.
#include <cuda_runtime.h>

#include <cstddef>

#include "dev_types.h"
#include "kernels.h"
#include "pose_core.h"

namespace b200tag {

namespace {

using namespace pose;

constexpr int kPoseWarps = 4;  // warps per CTA
constexpr unsigned kFull = 0xffffffffu;

struct PoseShared {
  OiConsts oi;              // what every step of the orthogonal iteration reads
  SecondMinFrame S;         // the frame and error quartic of the second-minimum search
  b200tag_detection det;    // the record, read once from mapped host memory
  M3 R1;                    // the first minimum, while the search runs
  V3 t1;
  double err1;
  b200tag_pose out;
};

// Step 3's search, split over the lanes: round k evaluates dE/dt at grid points 1 + 32k + lane, a ballot of the
// sign changes starts a bisection on each lane that holds one, and the refined minima are taken in grid order so that
// the first of equal errors wins, as in the host's serial loop.  Returns the number of distinct minima found.  Not
// inlined: register allocation of the search apart from the orthogonal iteration's keeps both free of spills.
__device__ __noinline__ int search_second_minimum(const SecondMinFrame &S, int lane, double *best_beta) {
  double carry_t = grid_t(0);
  double carry_d = S.q.dnum(carry_t);
  double best_err = HUGE_VAL;
  int n_minima = 0;
  *best_beta = 0;
  for (int base = 1; base <= kGrid; base += 32) {
    const int g = base + lane;
    double tt = 0, d = 0;
    if (g <= kGrid) {
      tt = grid_t(g);
      d = S.q.dnum(tt);
    }
    double prev_t = __shfl_up_sync(kFull, tt, 1), prev_d = __shfl_up_sync(kFull, d, 1);
    if (lane == 0) {
      prev_t = carry_t;
      prev_d = carry_d;
    }
    bool found = false;
    double beta = 0, e = 0;
    if (g <= kGrid && prev_d < 0 && d >= 0) {  // derivative goes from negative to positive: a minimum in between
      const double tmin = bisect_minimum(S.q, prev_t, tt);
      found = distinct_minimum(S, tmin, &beta);
      if (found) e = S.q.eval(tmin);
    }
    for (unsigned m = __ballot_sync(kFull, found); m; m &= m - 1) {
      const int src = __ffs(m) - 1;
      const double eb = __shfl_sync(kFull, e, src), bb = __shfl_sync(kFull, beta, src);
      n_minima++;
      if (eb < best_err) {
        best_err = eb;
        *best_beta = bb;
      }
    }
    carry_t = __shfl_sync(kFull, tt, 31);
    carry_d = __shfl_sync(kFull, d, 31);
  }
  return n_minima;
}

__device__ Distortion lens(const double *dist) { return Distortion{dist[0], dist[1], dist[2], dist[3], dist[4]}; }

__device__ void copy_pose_out(const PoseShared &sh, int lane, b200tag_pose *dst) {
  static_assert(sizeof(b200tag_pose) % 8 == 0 && sizeof(b200tag_pose) / 8 <= 32, "pose copy");
  if (lane < static_cast<int>(sizeof(b200tag_pose) / 8))
    reinterpret_cast<double *>(dst)[lane] = reinterpret_cast<const double *>(&sh.out)[lane];
  __syncwarp();  // sh is reused by this warp's next record
}

// b200tag_estimate_pose for one record, by one warp; with kDistorted, of the record undistort_record makes of it (lanes
// 0-3 undistort a corner each, lane 0 rebuilds H), or pose_failure's record when that fails.
template <bool kDistorted>
__device__ void estimate_pose_warp(const b200tag_detection *rec, const PoseLaunch &L, PoseShared &sh, int lane, b200tag_pose *dst) {
  static_assert(sizeof(b200tag_detection) % 8 == 0 && sizeof(b200tag_detection) / 8 <= 32, "record copy");
  if (lane < static_cast<int>(sizeof(b200tag_detection) / 8))
    reinterpret_cast<double *>(&sh.det)[lane] = reinterpret_cast<const double *>(rec)[lane];
  __syncwarp();
  if (kDistorted) {
    int fine = 1;
    if (lane < 4) fine = undistort_point(sh.det.p[lane], L.fx, L.fy, L.cx, L.cy, lens(L.dist), sh.det.p[lane]);
    fine = __all_sync(kFull, fine);
    __syncwarp();
    if (lane == 0 && fine) fine = record_homography(&sh.det);
    if (!__shfl_sync(kFull, fine, 0)) {
      if (lane == 0) pose_failure(&sh.out);
      __syncwarp();
      copy_pose_out(sh, lane, dst);
      return;
    }
    __syncwarp();
  }
  int ok = 0;
  if (lane == 0) {
    V3 v[4], p[4];
    rays_and_corners(sh.det, L.tagsize, L.fx, L.fy, L.cx, L.cy, v, p);
    ok = oi_prepare(v, p, &sh.oi);
  }
  ok = __shfl_sync(kFull, ok, 0);
  __syncwarp();
  {
    M3 R1;
    V3 t1;
    pose_from_homography(sh.det.H, L.tagsize, L.fx, L.fy, L.cx, L.cy, &R1, &t1);
    const double err1 = ok ? orthogonal_iteration(sh.oi, 50, &R1, &t1) : HUGE_VAL;
    int has = 0;
    if (lane == 0) {
      sh.R1 = R1;
      sh.t1 = t1;
      sh.err1 = err1;
      has = second_minimum_frame(sh.oi.v, sh.oi.p, R1, t1, &sh.S);
    }
    ok |= __shfl_sync(kFull, has, 0) << 1;
    __syncwarp();
  }
  M3 R2{};
  V3 t2{{0, 0, 0}};
  double err2 = HUGE_VAL, beta;
  if ((ok & 2) && search_second_minimum(sh.S, lane, &beta) == 1) {
    R2 = second_minimum_rotation(sh.S, beta);
    if (ok & 1) err2 = orthogonal_iteration(sh.oi, 50, &R2, &t2);
  }
  if (lane == 0) choose_pose(sh.R1, sh.t1, sh.err1, R2, t2, err2, &sh.out);
  __syncwarp();
  copy_pose_out(sh, lane, dst);
}

// blockIdx.y = frame; the warps of a frame's CTAs walk that frame's detections, as many as its counter says.
template <bool kDistorted>
__global__ void __launch_bounds__(kPoseWarps * 32) k_pose(PoseLaunch L) {
  __shared__ PoseShared sh[kPoseWarps];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const size_t frame = blockIdx.y;
  const uint32_t n = L.counters ? min(L.counters[frame].num_detections, L.stride) : L.count;
  const b200tag_detection *recs = L.dets + frame * L.stride;
  b200tag_pose *out = L.out + frame * L.stride;
  for (uint32_t i = blockIdx.x * kPoseWarps + w; i < n; i += gridDim.x * kPoseWarps)
    estimate_pose_warp<kDistorted>(recs + i, L, sh[w], lane, out + i);
}

constexpr int kIppeThreads = 128;  // threads per CTA of k_pose_ippe
static_assert(offsetof(b200tag_detection, p) % 16 == 0 && sizeof(b200tag_detection) % 16 == 0, "corner loads");
static_assert(sizeof(b200tag_pose) % 16 == 0, "pose stores");

// The IPPE pose (B200TAG_POSE_IPPE) of every raw detection: one thread per record, blockIdx.y = frame, as many records
// as the frame's counter holds.  A thread reads only the record's four corners from the mapped detection buffer and
// writes the pose to the same index of the mapped pose buffer; the arithmetic is ippe_pose, which the host's
// b200tag_estimate_poses_ippe runs too.  With kDistorted the thread undistorts the four corners first, one after the
// other, as b200tag_estimate_poses_distorted does.
template <bool kDistorted>
__global__ void __launch_bounds__(kIppeThreads) k_pose_ippe(PoseLaunch L) {
  const size_t frame = blockIdx.y;
  const uint32_t n = L.counters ? min(L.counters[frame].num_detections, L.stride) : L.count;
  const b200tag_detection *recs = L.dets + frame * L.stride;
  b200tag_pose *out = L.out + frame * L.stride;
  for (uint32_t i = blockIdx.x * kIppeThreads + threadIdx.x; i < n; i += gridDim.x * kIppeThreads) {
    const double2 *src = reinterpret_cast<const double2 *>(recs[i].p);
    double px[4][2];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const double2 c = src[k];
      px[k][0] = c.x;
      px[k][1] = c.y;
    }
    b200tag_pose pose;
    if (!kDistorted || undistort_corners(px, L.fx, L.fy, L.cx, L.cy, lens(L.dist), px))
      ippe_pose(px, L.tagsize, L.fx, L.fy, L.cx, L.cy, &pose);
    else
      pose_failure(&pose);
    const double2 *from = reinterpret_cast<const double2 *>(&pose);
    double2 *dst = reinterpret_cast<double2 *>(out + i);
#pragma unroll
    for (int k = 0; k < static_cast<int>(sizeof(b200tag_pose) / 16); k++) dst[k] = from[k];
  }
}

// The covariance (b200tag_set_pose_covariance) of every raw detection's pose, behind k_pose or k_pose_ippe: one thread
// per record, laid out as k_pose_ippe.  A thread reads the record's corners and its pose from the mapped buffers and
// writes the 36 entries to the same index of the mapped covariance buffer; the arithmetic is tag_covariance, which the
// host's b200tag_estimate_pose_covariances runs too.  kDistorted: through the lens of b200tag_set_pose_distortion.
template <bool kDistorted>
__global__ void __launch_bounds__(kIppeThreads) k_pose_cov(PoseLaunch L, b200tag_covariance *cov, double sigma) {
  static_assert(sizeof(b200tag_covariance) % 16 == 0, "covariance stores");
  const size_t frame = blockIdx.y;
  const uint32_t n = L.counters ? min(L.counters[frame].num_detections, L.stride) : L.count;
  const b200tag_detection *recs = L.dets + frame * L.stride;
  const b200tag_pose *poses = L.out + frame * L.stride;
  b200tag_covariance *out = cov + frame * L.stride;
  const FieldCamera cam{L.fx, L.fy, L.cx, L.cy};
  const Distortion D = lens(L.dist);
  for (uint32_t i = blockIdx.x * kIppeThreads + threadIdx.x; i < n; i += gridDim.x * kIppeThreads) {
    const double2 *src = reinterpret_cast<const double2 *>(recs[i].p);
    double px[4][2];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const double2 c = src[k];
      px[k][0] = c.x;
      px[k][1] = c.y;
    }
    b200tag_pose pose;
    const double2 *ps = reinterpret_cast<const double2 *>(poses + i);
#pragma unroll
    for (int k = 0; k < static_cast<int>(sizeof(b200tag_pose) / 16); k++) reinterpret_cast<double2 *>(&pose)[k] = ps[k];
    b200tag_covariance c;
    tag_covariance(px, pose, L.tagsize, cam, kDistorted ? &D : nullptr, sigma, c.C);
    double2 *dst = reinterpret_cast<double2 *>(out + i);
#pragma unroll
    for (int k = 0; k < static_cast<int>(sizeof(b200tag_covariance) / 16); k++) dst[k] = reinterpret_cast<const double2 *>(&c)[k];
  }
}

// The sum of v over the warp by the xor tree of pose_core.h (field_slot_tree): every lane ends with the same bits.
__device__ double warp_sum(double v) {
#pragma unroll
  for (int m = kFieldSlots / 2; m >= 1; m >>= 1) v = v + __shfl_xor_sync(kFull, v, m);
  return v;
}

// The field covariance of result `res` over the frame's `used` tags (k_field_pose with kCov): correspondence k on lane
// k % 32, the sums by warp_sum, then field_covariance on every lane; the lanes write the result between them.  Not
// inlined, so the solve's register allocation is that of the kernel without it.
template <bool kDistorted>
__device__ __noinline__ void field_covariance_warp(const FieldTagData *tags, int used, const b200tag_field_pose &res,
                                                   const FieldLaunch &L, int lane, b200tag_field_covariance *dst) {
  constexpr int kSums = kDistorted ? kCovSums : 22;  // without distortion B is not summed
  M3 R;
  V3 t;
  field_cov_pose(res, &R, &t);
  const FieldCamera cam{L.fx, L.fy, L.cx, L.cy};
  const Distortion D = lens(L.dist);
  double acc[kCovSums];
#pragma unroll
  for (int j = 0; j < kCovSums; j++) acc[j] = 0;
  for (int k = lane; k < 4 * used; k += 32) field_cov_corner_terms(tags[k >> 2], k & 3, R, t, cam, kDistorted ? &D : nullptr, acc);
  double S[kCovSums];
#pragma unroll
  for (int j = 0; j < kCovSums; j++) S[j] = j < kSums ? warp_sum(acc[j]) : 0.0;
  b200tag_field_covariance out;
  field_covariance(S, kDistorted, res, L.offset, L.sigma, &out);
  static_assert(sizeof(b200tag_field_covariance) / 8 <= 96, "covariance copy");
  for (int w = lane; w < static_cast<int>(sizeof(b200tag_field_covariance) / 8); w += 32)
    reinterpret_cast<double *>(dst)[w] = reinterpret_cast<const double *>(&out)[w];
}

// The field pose (b200tag_set_field_layout) of every frame: one warp per frame, blockIdx.x = frame, reading the frame's
// raw records from the mapped detection buffer, as many as its counter holds.  The lanes look the records up in the
// layout and keep, per layout tag, the record reconcile prefers; in layout order they write each used tag's corners and
// seeds to the frame's scratch, and then run field_solve with correspondence k on lane k % 32 and the 6x6 solve on every
// lane.  The arithmetic is pose_core.h's, the same b200tag_estimate_field_pose runs on the host.  With kDistorted the
// lane that owns a used layout tag undistorts its chosen record's corners first and leaves the tag out when one fails.
// With kCov the warp adds the covariance of the result (field_covariance_warp); the variants without it compile to the
// kernel without the step.
template <bool kDistorted, bool kCov>
__global__ void __launch_bounds__(32) k_field_pose(FieldLaunch L) {
  __shared__ int cnt[B200TAG_MAX_FIELD_TAGS], sel[B200TAG_MAX_FIELD_TAGS];
  __shared__ int dup;
  const int lane = threadIdx.x;
  const size_t frame = blockIdx.x;
  const uint32_t n = L.counters ? min(L.counters[frame].num_detections, L.stride) : L.count;
  const b200tag_detection *recs = L.dets + frame * L.stride;
  FieldTagData *tags = L.scratch + frame * L.scratch_stride;
  for (int i = lane; i < L.nlayout; i += 32) cnt[i] = 0;
  if (lane == 0) dup = 0;
  __syncwarp();
  for (uint32_t i = lane; i < n; i += 32) {
    const int li = field_lookup(L.keys, L.nlayout, recs[i].family, recs[i].id);
    if (li >= 0) {
      if (atomicAdd(&cnt[li], 1) > 0) dup = 1;
      sel[li] = static_cast<int>(i);
    }
  }
  __syncwarp();
  if (dup) {  // a layout tag seen more than once: the preferred record, the lowest index of identical ones
    for (uint32_t i = lane; i < n; i += 32) {
      const int32_t fam = recs[i].family, id = recs[i].id;
      const int li = field_lookup(L.keys, L.nlayout, fam, id);
      if (li < 0 || cnt[li] < 2) continue;
      bool wins = true;
      for (uint32_t k = 0; k < n && wins; k++) {
        if (k == i || recs[k].family != fam || recs[k].id != id) continue;
        wins = !field_prefers(recs[k], recs[i]) && (k > i || field_prefers(recs[i], recs[k]));
      }
      if (wins) sel[li] = static_cast<int>(i);
    }
    __syncwarp();
  }
  // the used tags in layout order; a tag whose IPPE candidates cannot be formed is left out
  const FieldCamera cam{L.fx, L.fy, L.cx, L.cy};
  const unsigned below = (1u << lane) - 1;
  int used = 0;
  for (int base = 0; base < L.nlayout; base += 32) {
    const int li = base + lane;
    const bool has = li < L.nlayout && cnt[li] > 0;
    const unsigned hm = __ballot_sync(kFull, has);
    bool ok = false;
    if (has) {
      const double2 *src = reinterpret_cast<const double2 *>(recs[sel[li]].p);
      double px[4][2];
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const double2 c = src[k];
        px[k][0] = c.x;
        px[k][1] = c.y;
      }
      ok = (!kDistorted || undistort_corners(px, L.fx, L.fy, L.cx, L.cy, lens(L.dist), px)) &&
           field_tag_data(L.layout[li], px, L.tagsize, cam, &tags[used + __popc(hm & below)]);
    }
    const unsigned om = __ballot_sync(kFull, ok);
    __syncwarp();
    for (unsigned m = om; om != hm && m; m &= m - 1) {  // move the formed tags down over the others, in order
      const int l = __ffs(m) - 1;
      const double *from = reinterpret_cast<const double *>(&tags[used + __popc(hm & ((1u << l) - 1))]);
      double *to = reinterpret_cast<double *>(&tags[used + __popc(om & ((1u << l) - 1))]);
      static_assert(sizeof(FieldTagData) % 8 == 0, "tag copy");
      if (from != to)
        for (int w = lane; w < static_cast<int>(sizeof(FieldTagData) / 8); w += 32) to[w] = from[w];
      __syncwarp();
    }
    used += __popc(om);
  }
  b200tag_field_pose res;
  if (used == 0) {
    field_empty(&res);
  } else {
    const int ncorr = 4 * used;
    auto cost = [&](const M3 &R, const V3 &t) {
      double acc = 0;
      for (int k = lane; k < ncorr; k += 32) {
        const FieldTagData &g = tags[k >> 2];
        V3 Y, P;
        double ru, rv;
        acc += field_corner_cost(g.px[k & 3][0], g.px[k & 3][1], g.X[k & 3], R, t, cam, &Y, &P, &ru, &rv);
      }
      return warp_sum(acc);
    };
    auto sum = [&](const M3 &R, const V3 &t, double *S) {
      double acc[kFieldSums];
#pragma unroll
      for (int j = 0; j < kFieldSums; j++) acc[j] = 0;
      for (int k = lane; k < ncorr; k += 32) {
        const FieldTagData &g = tags[k >> 2];
        field_corner_terms(g.px[k & 3][0], g.px[k & 3][1], g.X[k & 3], R, t, cam, acc);
      }
#pragma unroll
      for (int j = 0; j < kFieldSums; j++) S[j] = warp_sum(acc[j]);
    };
    field_solve(tags, used, cost, sum, L.rotation, L.offset, &res);
  }
  if (kCov) field_covariance_warp<kDistorted>(tags, used, res, L, lane, L.cov + frame);
  if (lane == 0) L.out[frame] = res;
}

// The floor covariance of result `res` over the frame's `ncorr` correspondences (k_floor_pose with kCov): correspondence k
// on lane k % 32, the sums by warp_sum, then floor_covariance on every lane; lanes 0-8 write an entry each.  Not
// inlined, so the solve's register allocation is that of the kernel without it.
template <bool kDistorted>
__device__ __noinline__ void floor_covariance_warp(const FieldTagData *tags, int ncorr, const b200tag_floor_pose &res,
                                                   const FloorModel &m, const FloorLaunch &L, int lane, double *dst) {
  constexpr int kSums = kDistorted ? kFloorCovSums : 7;  // without distortion M is not summed
  const FieldCamera cam{L.fx, L.fy, L.cx, L.cy};
  const FloorState st{res.x, res.y, res.cos_heading, res.sin_heading};
  const Distortion D = lens(L.dist);
  double acc[kFloorCovSums];
#pragma unroll
  for (int j = 0; j < kFloorCovSums; j++) acc[j] = 0;
  for (int k = lane; k < ncorr; k += 32) floor_cov_corner_terms(tags[k >> 2], k & 3, st, m, cam, kDistorted ? &D : nullptr, acc);
  double S[kFloorCovSums];
#pragma unroll
  for (int j = 0; j < kFloorCovSums; j++) S[j] = j < kSums ? warp_sum(acc[j]) : 0.0;
  double C[9];
  floor_covariance(S, kDistorted, res, m, L.sigma, C);
  if (lane < 9) dst[lane] = C[lane];
}

// The floor pose (b200tag_set_floor_pose) of every frame, behind k_field_pose: one warp per frame, blockIdx.x = frame,
// reading the used tags k_field_pose wrote to the frame's scratch (their count is its record's num_tags) and the
// frame's gyro heading.  Correspondence k on lane k % 32, the sums by warp_sum, floor_solve's 3x3 (or 2x2) step on every
// lane; the arithmetic is pose_core.h's, the same b200tag_estimate_floor_pose runs on the host.  With kCov the warp
// adds the 3x3 covariance of the result (kDistorted: through the lens).  heading is filled on the host.
template <bool kDistorted, bool kCov>
__global__ void __launch_bounds__(32) k_floor_pose(FloorLaunch L) {
  const int lane = threadIdx.x;
  const size_t frame = blockIdx.x;
  const int used = L.field[frame].num_tags;
  const FieldTagData *tags = L.scratch + frame * L.scratch_stride;
  FloorModel m;
#pragma unroll
  for (int k = 0; k < 9; k++) m.rot[k] = L.rotation[k];
#pragma unroll
  for (int k = 0; k < 3; k++) m.off[k] = L.offset[k];
  m.cg = L.gyro[2 * frame];
  m.sg = L.gyro[2 * frame + 1];
  m.w = L.weight;
  m.mode = floor_mode(m.cg, m.w);
  const FieldCamera cam{L.fx, L.fy, L.cx, L.cy};
  const int ncorr = 4 * used;
  b200tag_floor_pose res;
  if (used == 0) {
    floor_empty(m.mode, &res);
  } else {
    auto cost = [&](const FloorState &st) {
      double acc = 0;
      for (int k = lane; k < ncorr; k += 32) {
        const FieldTagData &g = tags[k >> 2];
        V3 W, P;
        double ru, rv;
        acc += floor_corner_cost(g.px[k & 3][0], g.px[k & 3][1], g.X[k & 3], st, m, cam, &W, &P, &ru, &rv);
      }
      return warp_sum(acc);
    };
    auto sum = [&](const FloorState &st, double *S) {
      double acc[kFloorSums];
#pragma unroll
      for (int j = 0; j < kFloorSums; j++) acc[j] = 0;
      for (int k = lane; k < ncorr; k += 32) {
        const FieldTagData &g = tags[k >> 2];
        floor_corner_terms(g.px[k & 3][0], g.px[k & 3][1], g.X[k & 3], st, m, cam, acc);
      }
#pragma unroll
      for (int j = 0; j < kFloorSums; j++) S[j] = warp_sum(acc[j]);
    };
    auto lin = [&](double *S) {
      double acc[kFloorLinSums];
#pragma unroll
      for (int j = 0; j < kFloorLinSums; j++) acc[j] = 0;
      for (int k = lane; k < ncorr; k += 32) {
        const FieldTagData &g = tags[k >> 2];
        floor_lin_terms(g.px[k & 3][0], g.px[k & 3][1], g.X[k & 3], m, cam, acc);
      }
#pragma unroll
      for (int j = 0; j < kFloorLinSums; j++) S[j] = warp_sum(acc[j]);
    };
    floor_solve(tags, used, m, cost, sum, lin, &res);
  }
  if (kCov) floor_covariance_warp<kDistorted>(tags, ncorr, res, m, L, lane, L.cov + 9 * frame);
  static_assert(sizeof(b200tag_floor_pose) % 8 == 0 && sizeof(b200tag_floor_pose) / 8 <= 32, "floor copy");
  if (lane < static_cast<int>(sizeof(b200tag_floor_pose) / 8))
    reinterpret_cast<double *>(L.out + frame)[lane] = reinterpret_cast<const double *>(&res)[lane];
}

}  // namespace

size_t field_tag_bytes() { return sizeof(FieldTagData); }

void launch_floor_pose(const FloorLaunch &L, int frames, Launcher &ln) {
  const bool cov = L.sigma > 0;
  const auto kernel = has_distortion(L.dist) ? (cov ? k_floor_pose<true, true> : k_floor_pose<true, false>)
                                             : (cov ? k_floor_pose<false, true> : k_floor_pose<false, false>);
  ln.timed("floor_pose", [&] { kernel<<<static_cast<unsigned>(frames), 32, 0, ln.s>>>(L); });
}

void launch_field_pose(const FieldLaunch &L, int frames, Launcher &ln) {
  const bool cov = L.sigma > 0;
  const auto kernel = has_distortion(L.dist) ? (cov ? k_field_pose<true, true> : k_field_pose<true, false>)
                                             : (cov ? k_field_pose<false, true> : k_field_pose<false, false>);
  ln.timed("field_pose", [&] { kernel<<<static_cast<unsigned>(frames), 32, 0, ln.s>>>(L); });
}

// One thread per record, all of a frame's records in one pass up to 1024 of them; CTAs past a frame's count exit.
static unsigned per_record_ctas(const PoseLaunch &L) {
  return L.counters ? min((L.stride + kIppeThreads - 1) / kIppeThreads, 8u) : (L.count + kIppeThreads - 1) / kIppeThreads;
}

void launch_pose_cov(const PoseLaunch &L, b200tag_covariance *cov, double sigma, int frames, Launcher &ln) {
  const unsigned ctas = per_record_ctas(L);
  const auto kernel = has_distortion(L.dist) ? k_pose_cov<true> : k_pose_cov<false>;
  ln.timed("pose_cov", [&] {
    if (ctas > 0) kernel<<<dim3(ctas, static_cast<unsigned>(frames)), kIppeThreads, 0, ln.s>>>(L, cov, sigma);
  });
}

void launch_pose(const PoseLaunch &L, int frames, Launcher &ln) {
  if (L.method == B200TAG_POSE_IPPE) {
    const unsigned ctas = per_record_ctas(L);
    const auto kernel = has_distortion(L.dist) ? k_pose_ippe<true> : k_pose_ippe<false>;
    ln.timed("pose_ippe", [&] {
      if (ctas > 0) kernel<<<dim3(ctas, static_cast<unsigned>(frames)), kIppeThreads, 0, ln.s>>>(L);
    });
    return;
  }
  // a frame of a batch has a handful of tags: 8 warps each, the rest loop; up to four frames (the single-frame latency
  // path, a cluttered 4K scene has ~100 tags): 128 warps each, one pass.  A list without counters is one frame.
  unsigned ctas = static_cast<unsigned>(frames) <= 4 ? 32u : 2u;
  if (!L.counters) ctas = static_cast<unsigned>((L.count + kPoseWarps - 1) / kPoseWarps);
  const auto kernel = has_distortion(L.dist) ? k_pose<true> : k_pose<false>;
  ln.timed("pose", [&] {
    if (ctas > 0) kernel<<<dim3(ctas, static_cast<unsigned>(frames)), kPoseWarps * 32, 0, ln.s>>>(L);
  });
}

}  // namespace b200tag
