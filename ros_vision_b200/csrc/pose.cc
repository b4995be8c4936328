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

int b200tag_estimate_field_pose(const b200tag_detection *dets, int count, const b200tag_field_tag *layout, int nlayout,
                                double tagsize, double fx, double fy, double cx, double cy, const double *rotation,
                                const double *offset, b200tag_field_pose *out) {
  if (count < 0 || (count > 0 && !dets) || !out || !(tagsize > 0) || fx == 0 || fy == 0) return B200TAG_E_INVALID;
  std::vector<FieldKey> keys(static_cast<size_t>(std::max(nlayout, 0)));
  if (!b200tag::field_layout_keys(layout, nlayout, nullptr, 0, keys.data())) return B200TAG_E_INVALID;
  static const double kEye[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, kZero[3] = {0, 0, 0};
  const double *Rx = rotation ? rotation : kEye, *ox = offset ? offset : kZero;
  // the detection reconcile prefers, per layout tag
  std::vector<int> sel(static_cast<size_t>(nlayout), -1);
  for (int i = 0; i < count; i++) {
    const int L = field_lookup(keys.data(), nlayout, dets[i].family, dets[i].id);
    if (L >= 0 && (sel[L] < 0 || field_prefers(dets[i], dets[sel[L]]))) sel[L] = i;
  }
  const FieldCamera cam{fx, fy, cx, cy};
  std::vector<FieldTagData> tags;
  for (int L = 0; L < nlayout; L++) {
    FieldTagData d;
    if (sel[L] >= 0 && field_tag_data(layout[L], dets[sel[L]].p, tagsize, cam, &d)) tags.push_back(d);
  }
  const int ntags = static_cast<int>(tags.size());
  if (ntags == 0) {
    field_empty(out);
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
  return 0;
}

}  // extern "C"
