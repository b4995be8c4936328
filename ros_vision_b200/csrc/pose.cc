// Tag pose from a detection: the step the node runs right after the hot path
// (reference: src/apriltags_cuda/src/apriltags_cuda_detector.cu:425-462 calls libapriltag's
// estimate_tag_pose(&info_, &pose) per detection; SURVEY.md section 8 row f3).  The arithmetic is in pose_core.h,
// which the device kernel (kernels_pose.cu) shares; here it runs serially, one detection and one grid point at a time.
#include <algorithm>
#include <cmath>
#include <vector>

#include "../../include/b200tag.h"
#include "pose_core.h"

namespace b200tag {

void locate_from_poses(const b200tag_detection *dets, const b200tag_pose *poses, int count, const double *rotation,
                       const double *offset, b200tag_tag_position *out) {
  static const double kEye[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, kZero[3] = {0, 0, 0};
  const double *Rx = rotation ? rotation : kEye, *ox = offset ? offset : kZero;
  for (int i = 0; i < count; i++) {
    const b200tag_pose &pose = poses[i];
    b200tag_tag_position &o = out[i];
    o.index = i;
    o.id = dets[i].id;
    for (int k = 0; k < 3; k++) o.camera[k] = pose.t[k];
    for (int r = 0; r < 3; r++) o.robot[r] = Rx[3 * r] * pose.t[0] + Rx[3 * r + 1] * pose.t[1] + Rx[3 * r + 2] * pose.t[2] + ox[r];
    o.distance = std::sqrt(pose.t[0] * pose.t[0] + pose.t[1] * pose.t[1] + pose.t[2] * pose.t[2]);
    o.err = pose.err;
  }
  std::stable_sort(out, out + count, [](const b200tag_tag_position &a, const b200tag_tag_position &b) { return a.distance < b.distance; });
}

bool field_layout_keys(const b200tag_field_tag *layout, int nlayout, const uint32_t *ncodes, int nfamilies, pose::FieldKey *keys) {
  if (nlayout < 0 || nlayout > B200TAG_MAX_FIELD_TAGS || (nlayout > 0 && !layout)) return false;
  for (int i = 0; i < nlayout; i++) {
    const b200tag_field_tag &L = layout[i];
    if (ncodes && (L.family < 0 || L.family >= nfamilies || L.id < 0 || static_cast<uint32_t>(L.id) >= ncodes[L.family]))
      return false;
    for (double x : L.R) if (!std::isfinite(x)) return false;
    for (double x : L.t) if (!std::isfinite(x)) return false;
    for (int r = 0; r < 3; r++)
      for (int c = 0; c < 3; c++) {
        const double d = L.R[3 * r] * L.R[3 * c] + L.R[3 * r + 1] * L.R[3 * c + 1] + L.R[3 * r + 2] * L.R[3 * c + 2];
        if (!(std::fabs(d - (r == c ? 1.0 : 0.0)) <= 1e-6)) return false;
      }
    pose::M3 R;
    for (int k = 0; k < 9; k++) R.a[k] = L.R[k];
    if (!(pose::det3(R) > 0)) return false;
    keys[i] = pose::FieldKey{L.family, L.id, i, 0};
  }
  std::sort(keys, keys + nlayout, [](const pose::FieldKey &a, const pose::FieldKey &b) { return pose::key_less(a.family, a.id, b.family, b.id); });
  for (int i = 1; i < nlayout; i++)
    if (keys[i].family == keys[i - 1].family && keys[i].id == keys[i - 1].id) return false;
  return true;
}

bool read_distortion(const double *dist, bool *active, pose::Distortion *D) {
  *active = false;
  *D = pose::Distortion{0, 0, 0, 0, 0};
  if (!dist) return true;
  for (int k = 0; k < 5; k++) {
    if (!std::isfinite(dist[k])) return false;
    *active = *active || dist[k] != 0;
  }
  *D = pose::Distortion{dist[0], dist[1], dist[2], dist[3], dist[4]};
  return true;
}

bool valid_sigma(double sigma) { return std::isfinite(sigma) && sigma > 0; }

bool floor_model(const double *rotation, const double *offset, double heading, double heading_weight, pose::FloorModel *m) {
  if (std::isinf(heading) || !(heading_weight > 0)) return false;
  static const double kEye[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, kZero[3] = {0, 0, 0};
  memcpy(m->rot, rotation ? rotation : kEye, sizeof(m->rot));
  memcpy(m->off, offset ? offset : kZero, sizeof(m->off));
  floor_gyro(heading, &m->cg, &m->sg);
  m->w = heading_weight;
  m->mode = pose::floor_mode(m->cg, heading_weight);
  return true;
}

void floor_gyro(double heading, double *cg, double *sg) {
  *cg = std::isnan(heading) ? NAN : std::cos(heading);
  *sg = std::isnan(heading) ? NAN : std::sin(heading);
}

}  // namespace b200tag

using namespace b200tag::pose;

namespace {

// Step 3: the second minimum's rotation, when there is exactly one other minimum (libapriltag's rule).
bool second_minimum(const V3 *v, const V3 *p, const M3 &R, const V3 &t, M3 *R2) {
  SecondMinFrame S;
  if (!second_minimum_frame(v, p, R, t, &S)) return false;
  double best_beta = 0, best_err = HUGE_VAL;
  int n_minima = 0;
  double prev_t = grid_t(0), prev_d = S.q.dnum(prev_t);
  for (int g = 1; g <= kGrid; g++) {
    const double tt = grid_t(g), d = S.q.dnum(tt);
    if (prev_d < 0 && d >= 0) {  // derivative goes from negative to positive: a minimum in between
      const double tmin = bisect_minimum(S.q, prev_t, tt);
      double bmin;
      if (distinct_minimum(S, tmin, &bmin)) {
        n_minima++;
        const double e = S.q.eval(tmin);
        if (e < best_err) { best_err = e; best_beta = bmin; }
      }
    }
    prev_t = tt;
    prev_d = d;
  }
  if (n_minima != 1) return false;
  *R2 = second_minimum_rotation(S, best_beta);
  return true;
}

}  // namespace

extern "C" {

int b200tag_estimate_pose(const b200tag_detection *det, double tagsize, double fx, double fy, double cx, double cy,
                          b200tag_pose *out) {
  if (!det || !out || !(tagsize > 0) || fx == 0 || fy == 0) return B200TAG_E_INVALID;
  V3 v[4], p[4];
  rays_and_corners(*det, tagsize, fx, fy, cx, cy, v, p);
  OiConsts c;
  const bool ok = oi_prepare(v, p, &c);
  M3 R1;
  V3 t1;
  pose_from_homography(det->H, tagsize, fx, fy, cx, cy, &R1, &t1);
  const double err1 = ok ? orthogonal_iteration(c, 50, &R1, &t1) : HUGE_VAL;
  M3 R2{};
  double err2 = HUGE_VAL;
  V3 t2{{0, 0, 0}};
  if (second_minimum(v, p, R1, t1, &R2) && ok) err2 = orthogonal_iteration(c, 50, &R2, &t2);
  choose_pose(R1, t1, err1, R2, t2, err2, out);
  return 0;
}

int b200tag_estimate_poses(const b200tag_detection *dets, int count, double tagsize, double fx, double fy, double cx,
                           double cy, b200tag_pose *out) {
  if (count < 0 || (count > 0 && (!dets || !out))) return B200TAG_E_INVALID;
  for (int i = 0; i < count; i++)
    if (int rc = b200tag_estimate_pose(dets + i, tagsize, fx, fy, cx, cy, out + i)) return rc;
  return 0;
}

int b200tag_estimate_poses_ippe(const b200tag_detection *dets, int count, double tagsize, double fx, double fy, double cx,
                                double cy, b200tag_pose *out) {
  if (count < 0 || (count > 0 && (!dets || !out))) return B200TAG_E_INVALID;
  if (count > 0 && (!(tagsize > 0) || fx == 0 || fy == 0)) return B200TAG_E_INVALID;
  for (int i = 0; i < count; i++) ippe_pose(dets[i].p, tagsize, fx, fy, cx, cy, out + i);
  return 0;
}

int b200tag_locate_tags(const b200tag_detection *dets, int count, double tagsize, double fx, double fy, double cx,
                        double cy, const double *rotation, const double *offset, b200tag_tag_position *out) {
  if (count < 0 || (count > 0 && (!dets || !out))) return B200TAG_E_INVALID;
  std::vector<b200tag_pose> poses(static_cast<size_t>(count));
  if (int rc = b200tag_estimate_poses(dets, count, tagsize, fx, fy, cx, cy, poses.data())) return rc;
  b200tag::locate_from_poses(dets, poses.data(), count, rotation, offset, out);
  return 0;
}

}  // extern "C"

namespace {

// The field covariance of result `res` over the corners of the used tags, summed in the solve's slot order.
void field_covariance_of(const FieldTagData *tags, int ntags, const FieldCamera &cam, const Distortion *lens,
                         const double *offset, double sigma, const b200tag_field_pose &res, b200tag_field_covariance *cov) {
  M3 R;
  V3 t;
  field_cov_pose(res, &R, &t);
  double slot[kFieldSlots][kCovSums] = {}, S[kCovSums];
  for (int k = 0; k < 4 * ntags; k++) {
    field_cov_corner_terms(tags[k >> 2], k & 3, R, t, cam, lens, slot[k % kFieldSlots]);
  }
  field_slot_tree<kCovSums>(slot, S);
  field_covariance(S, lens != nullptr, res, offset, sigma, cov);
}

// The used tags of b200tag_estimate_field_pose(_distorted), in layout order: per layout tag the detection reconcile
// prefers, its corners undistorted through `lens` (null: none); a tag whose corners fail or whose IPPE candidates cannot
// be formed is left out.
void field_tags(const b200tag_detection *dets, int count, const b200tag_field_tag *layout, int nlayout,
                const FieldKey *keys, double tagsize, const FieldCamera &cam, const Distortion *lens,
                std::vector<FieldTagData> *tags) {
  std::vector<int> sel(static_cast<size_t>(nlayout), -1);
  for (int i = 0; i < count; i++) {
    const int L = field_lookup(keys, nlayout, dets[i].family, dets[i].id);
    if (L >= 0 && (sel[L] < 0 || field_prefers(dets[i], dets[sel[L]]))) sel[L] = i;
  }
  for (int L = 0; L < nlayout; L++) {
    if (sel[L] < 0) continue;
    // only the chosen record's corners are undistorted; one that fails leaves the tag out
    double px[4][2];
    if (!lens) memcpy(px, dets[sel[L]].p, sizeof(px));
    else if (!undistort_corners(dets[sel[L]].p, cam.fx, cam.fy, cam.cx, cam.cy, *lens, px)) continue;
    FieldTagData d;
    if (field_tag_data(layout[L], px, tagsize, cam, &d)) tags->push_back(d);
  }
}

// b200tag_estimate_field_pose(_distorted); `lens` null: no undistortion step.  With `cov`, also the covariance of the
// result at sigma (b200tag_estimate_field_pose_covariance).
int field_pose(const b200tag_detection *dets, int count, const b200tag_field_tag *layout, int nlayout, double tagsize,
               double fx, double fy, double cx, double cy, const Distortion *lens, const double *rotation,
               const double *offset, b200tag_field_pose *out, double sigma = 0, b200tag_field_covariance *cov = nullptr) {
  if (count < 0 || (count > 0 && !dets) || !out || !(tagsize > 0) || fx == 0 || fy == 0) return B200TAG_E_INVALID;
  std::vector<FieldKey> keys(static_cast<size_t>(std::max(nlayout, 0)));
  if (!b200tag::field_layout_keys(layout, nlayout, nullptr, 0, keys.data())) return B200TAG_E_INVALID;
  static const double kEye[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, kZero[3] = {0, 0, 0};
  const double *Rx = rotation ? rotation : kEye, *ox = offset ? offset : kZero;
  const FieldCamera cam{fx, fy, cx, cy};
  std::vector<FieldTagData> tags;
  field_tags(dets, count, layout, nlayout, keys.data(), tagsize, cam, lens, &tags);
  const int ntags = static_cast<int>(tags.size());
  if (ntags == 0) {
    field_empty(out);
    if (cov) field_covariance_of(tags.data(), 0, cam, lens, ox, sigma, *out, cov);
    return 0;
  }
  const int ncorr = 4 * ntags;
  auto cost = [&](const M3 &R, const V3 &t) {
    double slot[kFieldSlots][1] = {};
    for (int k = 0; k < ncorr; k++) {
      const FieldTagData &g = tags[k >> 2];
      V3 Y, P;
      double ru, rv;
      slot[k % kFieldSlots][0] += field_corner_cost(g.px[k & 3][0], g.px[k & 3][1], g.X[k & 3], R, t, cam, &Y, &P, &ru, &rv);
    }
    double total;
    field_slot_tree<1>(slot, &total);
    return total;
  };
  auto sum = [&](const M3 &R, const V3 &t, double *S) {
    double slot[kFieldSlots][kFieldSums] = {};
    for (int k = 0; k < ncorr; k++) {
      const FieldTagData &g = tags[k >> 2];
      field_corner_terms(g.px[k & 3][0], g.px[k & 3][1], g.X[k & 3], R, t, cam, slot[k % kFieldSlots]);
    }
    field_slot_tree<kFieldSums>(slot, S);
  };
  field_solve(tags.data(), ntags, cost, sum, Rx, ox, out);
  if (cov) field_covariance_of(tags.data(), ntags, cam, lens, ox, sigma, *out, cov);
  return 0;
}

// b200tag_estimate_floor_pose after its checks; `lens` null: no undistortion step; cov (9) only when sigma > 0.
void floor_pose(const std::vector<FieldTagData> &tags, const FieldCamera &cam, const Distortion *lens, const FloorModel &m,
                double sigma, b200tag_floor_pose *out, double *cov) {
  const int ntags = static_cast<int>(tags.size()), ncorr = 4 * ntags;
  if (ntags == 0) {
    floor_empty(m.mode, out);
  } else {
    auto cost = [&](const FloorState &st) {
      double slot[kFieldSlots][1] = {};
      for (int k = 0; k < ncorr; k++) {
        const FieldTagData &g = tags[k >> 2];
        V3 W, P;
        double ru, rv;
        slot[k % kFieldSlots][0] += floor_corner_cost(g.px[k & 3][0], g.px[k & 3][1], g.X[k & 3], st, m, cam, &W, &P, &ru, &rv);
      }
      double total;
      field_slot_tree<1>(slot, &total);
      return total;
    };
    auto sum = [&](const FloorState &st, double *S) {
      double slot[kFieldSlots][kFloorSums] = {};
      for (int k = 0; k < ncorr; k++) {
        const FieldTagData &g = tags[k >> 2];
        floor_corner_terms(g.px[k & 3][0], g.px[k & 3][1], g.X[k & 3], st, m, cam, slot[k % kFieldSlots]);
      }
      field_slot_tree<kFloorSums>(slot, S);
    };
    auto lin = [&](double *S) {
      double slot[kFieldSlots][kFloorLinSums] = {};
      for (int k = 0; k < ncorr; k++) {
        const FieldTagData &g = tags[k >> 2];
        floor_lin_terms(g.px[k & 3][0], g.px[k & 3][1], g.X[k & 3], m, cam, slot[k % kFieldSlots]);
      }
      field_slot_tree<kFloorLinSums>(slot, S);
    };
    floor_solve(tags.data(), ntags, m, cost, sum, lin, out);
  }
  out->heading = std::atan2(out->sin_heading, out->cos_heading);
  if (!(sigma > 0)) return;
  const FloorState st{out->x, out->y, out->cos_heading, out->sin_heading};
  double slot[kFieldSlots][kFloorCovSums] = {}, S[kFloorCovSums];
  for (int k = 0; k < ncorr; k++) floor_cov_corner_terms(tags[k >> 2], k & 3, st, m, cam, lens, slot[k % kFieldSlots]);
  field_slot_tree<kFloorCovSums>(slot, S);
  floor_covariance(S, lens != nullptr, *out, m, sigma, cov);
}

}  // namespace

extern "C" {

int b200tag_estimate_field_pose(const b200tag_detection *dets, int count, const b200tag_field_tag *layout, int nlayout,
                                double tagsize, double fx, double fy, double cx, double cy, const double *rotation,
                                const double *offset, b200tag_field_pose *out) {
  return field_pose(dets, count, layout, nlayout, tagsize, fx, fy, cx, cy, nullptr, rotation, offset, out);
}

int b200tag_undistort_points(const double (*in)[2], int n, double fx, double fy, double cx, double cy, const double *dist,
                             double (*out)[2]) {
  bool active;
  Distortion D;
  if (n < 0 || (n > 0 && (!in || !out)) || fx == 0 || fy == 0 || !b200tag::read_distortion(dist, &active, &D))
    return B200TAG_E_INVALID;
  for (int i = 0; i < n; i++) {
    if (!active) {
      out[i][0] = in[i][0];
      out[i][1] = in[i][1];
    } else if (!undistort_point(in[i], fx, fy, cx, cy, D, out[i])) {
      out[i][0] = out[i][1] = NAN;
    }
  }
  return 0;
}

int b200tag_estimate_poses_distorted(const b200tag_detection *dets, int count, int method, double tagsize, double fx,
                                     double fy, double cx, double cy, const double *dist, b200tag_pose *out) {
  bool active;
  Distortion D;
  if ((method != B200TAG_POSE_ORTHOGONAL_ITERATION && method != B200TAG_POSE_IPPE) || !b200tag::read_distortion(dist, &active, &D))
    return B200TAG_E_INVALID;
  const bool ippe = method == B200TAG_POSE_IPPE;
  if (!active)
    return ippe ? b200tag_estimate_poses_ippe(dets, count, tagsize, fx, fy, cx, cy, out)
                : b200tag_estimate_poses(dets, count, tagsize, fx, fy, cx, cy, out);
  if (count < 0 || (count > 0 && (!dets || !out))) return B200TAG_E_INVALID;
  if (count > 0 && (!(tagsize > 0) || fx == 0 || fy == 0)) return B200TAG_E_INVALID;
  for (int i = 0; i < count; i++) {
    b200tag_detection rec = dets[i];
    if (ippe) {
      if (undistort_corners(rec.p, fx, fy, cx, cy, D, rec.p)) ippe_pose(rec.p, tagsize, fx, fy, cx, cy, out + i);
      else pose_failure(out + i);
    } else {
      if (undistort_record(&rec, fx, fy, cx, cy, D)) b200tag_estimate_pose(&rec, tagsize, fx, fy, cx, cy, out + i);
      else pose_failure(out + i);
    }
  }
  return 0;
}

int b200tag_estimate_field_pose_distorted(const b200tag_detection *dets, int count, const b200tag_field_tag *layout,
                                          int nlayout, double tagsize, double fx, double fy, double cx, double cy,
                                          const double *dist, const double *rotation, const double *offset,
                                          b200tag_field_pose *out) {
  bool active;
  Distortion D;
  if (!b200tag::read_distortion(dist, &active, &D)) return B200TAG_E_INVALID;
  return field_pose(dets, count, layout, nlayout, tagsize, fx, fy, cx, cy, active ? &D : nullptr, rotation, offset, out);
}

int b200tag_estimate_pose_covariances(const b200tag_detection *dets, const b200tag_pose *poses, int count, double tagsize,
                                      double fx, double fy, double cx, double cy, const double *dist, double sigma,
                                      b200tag_covariance *out) {
  bool active;
  Distortion D;
  if (!b200tag::valid_sigma(sigma) || !b200tag::read_distortion(dist, &active, &D)) return B200TAG_E_INVALID;
  if (count < 0 || (count > 0 && (!dets || !poses || !out))) return B200TAG_E_INVALID;
  if (count > 0 && (!(tagsize > 0) || fx == 0 || fy == 0)) return B200TAG_E_INVALID;
  const FieldCamera cam{fx, fy, cx, cy};
  for (int i = 0; i < count; i++) tag_covariance(dets[i].p, poses[i], tagsize, cam, active ? &D : nullptr, sigma, out[i].C);
  return 0;
}

int b200tag_estimate_field_pose_covariance(const b200tag_detection *dets, int count, const b200tag_field_tag *layout,
                                           int nlayout, double tagsize, double fx, double fy, double cx, double cy,
                                           const double *dist, const double *rotation, const double *offset, double sigma,
                                           b200tag_field_pose *out, b200tag_field_covariance *cov) {
  bool active;
  Distortion D;
  if (!b200tag::valid_sigma(sigma) || !cov || !b200tag::read_distortion(dist, &active, &D)) return B200TAG_E_INVALID;
  return field_pose(dets, count, layout, nlayout, tagsize, fx, fy, cx, cy, active ? &D : nullptr, rotation, offset, out,
                    sigma, cov);
}

int b200tag_estimate_floor_pose(const b200tag_detection *dets, int count, const b200tag_field_tag *layout, int nlayout,
                                double tagsize, double fx, double fy, double cx, double cy, const double *dist,
                                const double *rotation, const double *offset, double heading, double heading_weight,
                                double sigma, b200tag_floor_pose *out, double cov[9]) {
  bool active;
  Distortion D;
  FloorModel m;
  if (!b200tag::read_distortion(dist, &active, &D) || !b200tag::floor_model(rotation, offset, heading, heading_weight, &m))
    return B200TAG_E_INVALID;
  if (!(sigma == 0 || b200tag::valid_sigma(sigma)) || (sigma > 0 && !cov)) return B200TAG_E_INVALID;
  if (count < 0 || (count > 0 && !dets) || !out || !(tagsize > 0) || fx == 0 || fy == 0) return B200TAG_E_INVALID;
  std::vector<FieldKey> keys(static_cast<size_t>(std::max(nlayout, 0)));
  if (!b200tag::field_layout_keys(layout, nlayout, nullptr, 0, keys.data())) return B200TAG_E_INVALID;
  const FieldCamera cam{fx, fy, cx, cy};
  std::vector<FieldTagData> tags;
  field_tags(dets, count, layout, nlayout, keys.data(), tagsize, cam, active ? &D : nullptr, &tags);
  floor_pose(tags, cam, active ? &D : nullptr, m, sigma, out, cov);
  return 0;
}

}  // extern "C"
