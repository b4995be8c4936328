// Arithmetic of the pose step (b200tag_estimate_pose), shared by the host functions in pose.cc and the device kernel in
// kernels_pose.cu.  libapriltag (github.com/cgpadwick/apriltag tag 3.3.0) is not vendored in the reference tree, so
// this is a restatement of the published algorithm its apriltag_pose.c implements -- PARITY UNPINNED against
// libapriltag itself; checked against ground-truth poses and an independent numpy restatement (tests/test_pose.py):
//   1. initial pose from the homography (homography_to_pose + polar decomposition),
//   2. orthogonal iteration (Lu, Hager, Mjolsness 2000) for 50 steps,
//   3. the second local minimum of the object-space error (Schweighofer & Pinz 2006): rotate into the frame
//      where the ambiguity is a rotation about the y axis, minimise the quartic-over-(1+t^2)^2 error in
//      t = tan(beta / 2), refine that candidate by orthogonal iteration too,
//   4. return the pose with the smaller object-space error.
//
// One source for both sides keeps them in step: the library is built with -ffp-contract=off for the host and
// -fmad=false for the device, and steps 1 and 2 use only + - * /, sqrt, fabs and fmax, so the first local minimum
// comes out bit-identical on host and device.  Only step 3 calls tan / atan / atan2 / sin / cos, where glibc and
// libdevice may differ by an ulp.
//
// The second method, IPPE (ippe_pose, at the end), is closed form and uses only + - * /, sqrt, fabs and fmax: its
// poses are bit-identical on host and device.  So is the field pose (field_solve, at the end): the same operations, and
// every sum over correspondences taken in one order on both sides.  So is the exact inverse of the lens distortion model
// (undistort_point, after IPPE) that corrects the detections' corners before either pose.
#ifndef B200TAG_POSE_CORE_H_
#define B200TAG_POSE_CORE_H_

#include <cmath>
#include <cstdint>
#include <cstring>

#include "../../include/b200tag.h"

#ifdef __CUDACC__
#define POSE_HD __host__ __device__ inline
#define POSE_HD_CALL __host__ __device__ inline __noinline__  // a call of its own: keeps the caller's registers free of spills
#define POSE_UNROLL _Pragma("unroll")
#else
#define POSE_HD inline
#define POSE_HD_CALL inline
#define POSE_UNROLL
#endif

namespace b200tag {
namespace pose {

struct M3 {
  double a[9];
  POSE_HD double &operator()(int r, int c) { return a[r * 3 + c]; }
  POSE_HD double operator()(int r, int c) const { return a[r * 3 + c]; }
};
struct V3 {
  double v[3];
};

POSE_HD M3 ident() { return M3{{1, 0, 0, 0, 1, 0, 0, 0, 1}}; }
POSE_HD M3 mul(const M3 &A, const M3 &B) {
  M3 C{};
  POSE_UNROLL for (int i = 0; i < 3; i++)
    POSE_UNROLL for (int j = 0; j < 3; j++) C(i, j) = A(i, 0) * B(0, j) + A(i, 1) * B(1, j) + A(i, 2) * B(2, j);
  return C;
}
POSE_HD M3 transpose(const M3 &A) {
  M3 T{};
  POSE_UNROLL for (int i = 0; i < 3; i++)
    POSE_UNROLL for (int j = 0; j < 3; j++) T(i, j) = A(j, i);
  return T;
}
POSE_HD V3 mul(const M3 &A, const V3 &x) {
  return V3{{A(0, 0) * x.v[0] + A(0, 1) * x.v[1] + A(0, 2) * x.v[2], A(1, 0) * x.v[0] + A(1, 1) * x.v[1] + A(1, 2) * x.v[2],
             A(2, 0) * x.v[0] + A(2, 1) * x.v[1] + A(2, 2) * x.v[2]}};
}
POSE_HD V3 add(const V3 &a, const V3 &b) { return V3{{a.v[0] + b.v[0], a.v[1] + b.v[1], a.v[2] + b.v[2]}}; }
POSE_HD V3 sub(const V3 &a, const V3 &b) { return V3{{a.v[0] - b.v[0], a.v[1] - b.v[1], a.v[2] - b.v[2]}}; }
POSE_HD V3 scale(const V3 &a, double s) { return V3{{a.v[0] * s, a.v[1] * s, a.v[2] * s}}; }
POSE_HD double dot(const V3 &a, const V3 &b) { return a.v[0] * b.v[0] + a.v[1] * b.v[1] + a.v[2] * b.v[2]; }
POSE_HD V3 cross(const V3 &a, const V3 &b) {
  return V3{{a.v[1] * b.v[2] - a.v[2] * b.v[1], a.v[2] * b.v[0] - a.v[0] * b.v[2], a.v[0] * b.v[1] - a.v[1] * b.v[0]}};
}
POSE_HD M3 sub(const M3 &A, const M3 &B) {
  M3 C{};
  POSE_UNROLL for (int i = 0; i < 9; i++) C.a[i] = A.a[i] - B.a[i];
  return C;
}
POSE_HD double det3(const M3 &A) {
  return A(0, 0) * (A(1, 1) * A(2, 2) - A(1, 2) * A(2, 1)) - A(0, 1) * (A(1, 0) * A(2, 2) - A(1, 2) * A(2, 0)) +
         A(0, 2) * (A(1, 0) * A(2, 1) - A(1, 1) * A(2, 0));
}
POSE_HD bool inverse(const M3 &A, M3 *out) {
  const double d = det3(A);
  if (!(fabs(d) > 1e-300)) return false;
  M3 I{};
  I(0, 0) = (A(1, 1) * A(2, 2) - A(1, 2) * A(2, 1)) / d;
  I(0, 1) = (A(0, 2) * A(2, 1) - A(0, 1) * A(2, 2)) / d;
  I(0, 2) = (A(0, 1) * A(1, 2) - A(0, 2) * A(1, 1)) / d;
  I(1, 0) = (A(1, 2) * A(2, 0) - A(1, 0) * A(2, 2)) / d;
  I(1, 1) = (A(0, 0) * A(2, 2) - A(0, 2) * A(2, 0)) / d;
  I(1, 2) = (A(0, 2) * A(1, 0) - A(0, 0) * A(1, 2)) / d;
  I(2, 0) = (A(1, 0) * A(2, 1) - A(1, 1) * A(2, 0)) / d;
  I(2, 1) = (A(0, 1) * A(2, 0) - A(0, 0) * A(2, 1)) / d;
  I(2, 2) = (A(0, 0) * A(1, 1) - A(0, 1) * A(1, 0)) / d;
  *out = I;
  return true;
}

// One-sided Jacobi SVD of a 3x3 matrix: A = U diag(s) V^T.  Only U V^T is used by the callers.
POSE_HD void svd3(const M3 &A, M3 *U, M3 *V) {
  M3 W = A;  // columns are rotated until mutually orthogonal: W = A V
  M3 Vm = ident();
  for (int sweep = 0; sweep < 60; sweep++) {
    double off = 0;
    POSE_UNROLL for (int p = 0; p < 2; p++) {
      POSE_UNROLL for (int q = p + 1; q < 3; q++) {
        double alpha = 0, beta = 0, gamma = 0;
        POSE_UNROLL for (int i = 0; i < 3; i++) {
          alpha += W(i, p) * W(i, p);
          beta += W(i, q) * W(i, q);
          gamma += W(i, p) * W(i, q);
        }
        off = fmax(off, fabs(gamma) / sqrt(alpha * beta + 1e-300));
        if (fabs(gamma) < 1e-300) continue;
        const double zeta = (beta - alpha) / (2 * gamma);
        const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1 + zeta * zeta));
        const double c = 1 / sqrt(1 + t * t), s = c * t;
        POSE_UNROLL for (int i = 0; i < 3; i++) {
          const double wp = W(i, p), wq = W(i, q);
          W(i, p) = c * wp - s * wq;
          W(i, q) = s * wp + c * wq;
          const double vp = Vm(i, p), vq = Vm(i, q);
          Vm(i, p) = c * vp - s * vq;
          Vm(i, q) = s * vp + c * vq;
        }
      }
    }
    if (off < 1e-15) break;
  }
  // U = W with normalised columns; a (near) zero column is replaced by the cross product of the other two
  M3 Um{};
  double n[3];
  POSE_UNROLL for (int j = 0; j < 3; j++) n[j] = sqrt(W(0, j) * W(0, j) + W(1, j) * W(1, j) + W(2, j) * W(2, j));
  const double nmax = fmax(n[0], fmax(n[1], n[2]));
  int small = -1;
  POSE_UNROLL for (int j = 0; j < 3; j++) {
    if (n[j] > 1e-12 * nmax && n[j] > 0) {
      POSE_UNROLL for (int i = 0; i < 3; i++) Um(i, j) = W(i, j) / n[j];
    } else {
      small = j;
    }
  }
  // the replaced column, spelled out per case so that no matrix is indexed with a run-time value
  POSE_UNROLL for (int j = 0; j < 3; j++) {
    if (small == j) {
      const int a = (j + 1) % 3, b = (j + 2) % 3;
      const V3 ca{{Um(0, a), Um(1, a), Um(2, a)}}, cb{{Um(0, b), Um(1, b), Um(2, b)}};
      const V3 cc = cross(ca, cb);
      POSE_UNROLL for (int i = 0; i < 3; i++) Um(i, j) = cc.v[i];
    }
  }
  *U = Um;
  *V = Vm;
}

POSE_HD M3 outer_over_norm(const V3 &v) {  // v v^T / (v^T v)
  M3 F{};
  const double d = dot(v, v);
  POSE_UNROLL for (int i = 0; i < 3; i++)
    POSE_UNROLL for (int j = 0; j < 3; j++) F(i, j) = v.v[i] * v.v[j] / d;
  return F;
}

POSE_HD bool same_bits(double a, double b) {
#ifdef __CUDA_ARCH__
  return __double_as_longlong(a) == __double_as_longlong(b);
#else
  int64_t x, y;
  memcpy(&x, &a, sizeof(x));
  memcpy(&y, &b, sizeof(y));
  return x == y;
#endif
}

// What the orthogonal iteration reads on every step for one detection: its four image rays v, the tag corners p,
// p minus their mean, F = v v^T / v^T v and (I - mean F)^-1.  The device kernel keeps it in shared memory.
struct OiConsts {
  V3 v[4], p[4], p_res[4];
  M3 F[4];
  M3 M1inv;
};

// Fills `c` from v and p (4 points each); false when I - mean(F) cannot be inverted.
POSE_HD bool oi_prepare(const V3 *v, const V3 *p, OiConsts *c) {
  const int n = 4;
  V3 p_mean{{0, 0, 0}};
  POSE_UNROLL for (int i = 0; i < n; i++) p_mean = add(p_mean, scale(p[i], 1.0 / n));
  M3 avgF{};
  POSE_UNROLL for (int i = 0; i < n; i++) {
    c->v[i] = v[i];
    c->p[i] = p[i];
    c->p_res[i] = sub(p[i], p_mean);
    c->F[i] = outer_over_norm(v[i]);
    POSE_UNROLL for (int k = 0; k < 9; k++) avgF.a[k] += c->F[i].a[k] / n;
  }
  return inverse(sub(ident(), avgF), &c->M1inv);
}

// Lu-Hager-Mjolsness orthogonal iteration from *R; returns the object-space error of the final (R, t).  A step that
// gives back the rotation it started from, bit for bit, gives back the same t and error too, and so does every later
// step: the iteration stops there with the result of all `steps` steps.
POSE_HD double orthogonal_iteration(const OiConsts &c, int steps, M3 *R, V3 *t) {
  const int n = 4;
  double err = HUGE_VAL;
  for (int it = 0; it < steps; it++) {
    V3 M2{{0, 0, 0}};
    POSE_UNROLL for (int j = 0; j < n; j++) M2 = add(M2, scale(mul(sub(c.F[j], ident()), mul(*R, c.p[j])), 1.0 / n));
    *t = mul(c.M1inv, M2);
    V3 q[4], q_mean{{0, 0, 0}};
    POSE_UNROLL for (int j = 0; j < n; j++) {
      q[j] = mul(c.F[j], add(mul(*R, c.p[j]), *t));
      q_mean = add(q_mean, scale(q[j], 1.0 / n));
    }
    M3 M3m{};
    POSE_UNROLL for (int j = 0; j < n; j++) {
      const V3 d = sub(q[j], q_mean);
      POSE_UNROLL for (int r = 0; r < 3; r++)
        POSE_UNROLL for (int k = 0; k < 3; k++) M3m(r, k) += d.v[r] * c.p_res[j].v[k];
    }
    M3 U, V;
    svd3(M3m, &U, &V);
    M3 Rn = mul(U, transpose(V));
    if (det3(Rn) < 0) {
      Rn(0, 2) = -Rn(0, 2);
      Rn(1, 2) = -Rn(1, 2);
      Rn(2, 2) = -Rn(2, 2);
    }
    bool same = true;
    POSE_UNROLL for (int k = 0; k < 9; k++) same = same && same_bits(Rn.a[k], R->a[k]);
    *R = Rn;
    err = 0;
    POSE_UNROLL for (int j = 0; j < n; j++) {
      const V3 e = mul(sub(ident(), c.F[j]), add(mul(*R, c.p[j]), *t));
      err += dot(e, e);
    }
    if (same) break;
  }
  return err;
}

// homography_to_pose (libapriltag common/homography.c) + the estimate_pose_for_tag_homography wrapper.
POSE_HD void pose_from_homography(const double *H, double tagsize, double fx, double fy, double cx, double cy, M3 *R, V3 *t) {
  const double nfx = -fx;  // the wrapper passes -fx and flips the y and z axes afterwards
  double R20 = H[6], R21 = H[7], TZ = H[8];
  double R00 = (H[0] - cx * R20) / nfx, R01 = (H[1] - cx * R21) / nfx, TX = (H[2] - cx * TZ) / nfx;
  double R10 = (H[3] - cy * R20) / fy, R11 = (H[4] - cy * R21) / fy, TY = (H[5] - cy * TZ) / fy;
  const double l1 = sqrt(R00 * R00 + R10 * R10 + R20 * R20), l2 = sqrt(R01 * R01 + R11 * R11 + R21 * R21);
  double s = 1.0 / sqrt(l1 * l2);
  if (TZ > 0) s = -s;  // tag in front of a camera looking down -z
  R20 *= s; R21 *= s; TZ *= s; R00 *= s; R01 *= s; TX *= s; R10 *= s; R11 *= s; TY *= s;
  const double R02 = R10 * R21 - R20 * R11, R12 = R20 * R01 - R00 * R21, R22 = R00 * R11 - R10 * R01;
  M3 Rm{{R00, R01, R02, R10, R11, R12, R20, R21, R22}};
  M3 U, V;
  svd3(Rm, &U, &V);
  Rm = mul(U, transpose(V));  // polar decomposition: closest rotation
  const double sc = tagsize / 2.0;
  // fix = diag(1, -1, -1): camera looking down +z with y down
  *R = M3{{Rm(0, 0), Rm(0, 1), Rm(0, 2), -Rm(1, 0), -Rm(1, 1), -Rm(1, 2), -Rm(2, 0), -Rm(2, 1), -Rm(2, 2)}};
  *t = V3{{TX * sc, -TY * sc, -TZ * sc}};
}

// Rays through the four image corners `px` and the tag's corners in its own frame (step 1's inputs).
POSE_HD void rays_and_corners(const double (*px)[2], double tagsize, double fx, double fy, double cx, double cy, V3 *v, V3 *p) {
  const double sc = tagsize / 2.0;
  p[0] = V3{{-sc, sc, 0}}; p[1] = V3{{sc, sc, 0}}; p[2] = V3{{sc, -sc, 0}}; p[3] = V3{{-sc, -sc, 0}};
  POSE_UNROLL for (int i = 0; i < 4; i++) v[i] = V3{{(px[i][0] - cx) / fx, (px[i][1] - cy) / fy, 1}};
}
POSE_HD void rays_and_corners(const b200tag_detection &det, double tagsize, double fx, double fy, double cx, double cy, V3 *v, V3 *p) {
  rays_and_corners(det.p, tagsize, fx, fy, cx, cy, v, p);
}

// Object-space error as a function of the rotation beta about the y axis of the transformed frame, in
// t = tan(beta / 2): E(t) = (a0 + a1 t + a2 t^2 + a3 t^3 + a4 t^4) / (1 + t^2)^2.
struct Quartic {
  double a[5];
  POSE_HD double eval(double t) const {
    const double num = a[0] + t * (a[1] + t * (a[2] + t * (a[3] + t * a[4])));
    const double d = 1 + t * t;
    return num / (d * d);
  }
  // numerator of dE/dt times (1 + t^2)^3
  POSE_HD double dnum(double t) const {
    return a[1] + t * ((2 * a[2] - 4 * a[0]) + t * ((3 * a[3] - 3 * a[1]) + t * ((4 * a[4] - 2 * a[2]) - t * a[3])));
  }
};

// The rotated frame of the Schweighofer-Pinz search and the error quartic in it.
struct SecondMinFrame {
  M3 Rt, Rgamma, RzT;
  double beta0;  // beta of the pose the search started from
  Quartic q;
};

// Step 3 up to the search: false when the pose has no distinct second minimum to look for.
POSE_HD bool second_minimum_frame(const V3 *v, const V3 *p, const M3 &R, const V3 &t, SecondMinFrame *S) {
  const int n = 4;
  const double tn = sqrt(dot(t, t));
  if (!(tn > 0)) return false;
  const V3 rt3 = scale(t, 1.0 / tn);
  const V3 ex{{1, 0, 0}};
  V3 rt1 = sub(ex, scale(rt3, dot(ex, rt3)));
  const double n1 = sqrt(dot(rt1, rt1));
  if (!(n1 > 1e-12)) return false;
  rt1 = scale(rt1, 1.0 / n1);
  const V3 rt2 = cross(rt3, rt1);
  const M3 Rt{{rt1.v[0], rt1.v[1], rt1.v[2], rt2.v[0], rt2.v[1], rt2.v[2], rt3.v[0], rt3.v[1], rt3.v[2]}};
  const M3 R1p = mul(Rt, R);
  double r31 = R1p(2, 0), r32 = R1p(2, 1);
  double hyp = sqrt(r31 * r31 + r32 * r32);
  if (hyp < 1e-100) { r31 = 1; r32 = 0; hyp = 1; }
  const M3 Rz{{r31 / hyp, -r32 / hyp, 0, r32 / hyp, r31 / hyp, 0, 0, 0, 1}};
  const M3 Rtrans = mul(R1p, Rz);
  const double sin_gamma = -Rtrans(0, 1), cos_gamma = Rtrans(1, 1);
  const M3 Rgamma{{cos_gamma, -sin_gamma, 0, sin_gamma, cos_gamma, 0, 0, 0, 1}};
  const double sin_beta = -Rtrans(2, 0), cos_beta = Rtrans(2, 2);
  S->beta0 = atan2(sin_beta, cos_beta);

  V3 vt[4], pt[4];
  M3 Ft[4], avgF{};
  const M3 RzT = transpose(Rz);
  POSE_UNROLL for (int i = 0; i < n; i++) {
    vt[i] = mul(Rt, v[i]);
    pt[i] = mul(RzT, p[i]);
    Ft[i] = outer_over_norm(vt[i]);
    POSE_UNROLL for (int k = 0; k < 9; k++) avgF.a[k] += Ft[i].a[k] / n;
  }
  M3 G;
  if (!inverse(sub(ident(), avgF), &G)) return false;
  POSE_UNROLL for (int k = 0; k < 9; k++) G.a[k] /= n;
  // R_beta = (I + t M1 + t^2 M2) / (1 + t^2)
  const M3 Mk[3] = {ident(), M3{{0, 0, 2, 0, 0, 0, -2, 0, 0}}, M3{{-1, 0, 0, 0, 1, 0, 0, 0, -1}}};
  V3 b[3];
  POSE_UNROLL for (int k = 0; k < 3; k++) {
    V3 acc{{0, 0, 0}};
    POSE_UNROLL for (int i = 0; i < n; i++) acc = add(acc, mul(sub(Ft[i], ident()), mul(Rgamma, mul(Mk[k], pt[i]))));
    b[k] = mul(G, acc);
  }
  Quartic q{{0, 0, 0, 0, 0}};
  POSE_UNROLL for (int i = 0; i < n; i++) {
    V3 c[3];
    POSE_UNROLL for (int k = 0; k < 3; k++) c[k] = mul(sub(ident(), Ft[i]), add(mul(Rgamma, mul(Mk[k], pt[i])), b[k]));
    q.a[0] += dot(c[0], c[0]);
    q.a[1] += 2 * dot(c[0], c[1]);
    q.a[2] += dot(c[1], c[1]) + 2 * dot(c[0], c[2]);
    q.a[3] += 2 * dot(c[1], c[2]);
    q.a[4] += dot(c[2], c[2]);
  }
  S->Rt = Rt;
  S->Rgamma = Rgamma;
  S->RzT = RzT;
  S->q = q;
  return true;
}

// The search for stationary points of E over beta in (-pi, pi): the sign of dE/dt at grid points g = 0..kGrid, a
// minimum wherever it goes from negative to non-negative, refined by bisection.
constexpr int kGrid = 1440;
constexpr double kPi = 3.14159265358979323846;

POSE_HD double grid_t(int g) {  // t = tan(beta / 2) at grid point g; the ends stay 1e-9 inside (-pi, pi)
  if (g == 0) return tan((-kPi + 1e-9) / 2);
  const double beta = -kPi + (2 * kPi) * g / kGrid - (g == kGrid ? 1e-9 : 0);
  return tan(beta / 2);
}

POSE_HD double bisect_minimum(const Quartic &q, double lo, double hi) {
  for (int it = 0; it < 80; it++) {
    const double mid = 0.5 * (lo + hi);
    if (q.dnum(mid) < 0) lo = mid; else hi = mid;
  }
  return 0.5 * (lo + hi);
}

// A refined minimum counts when it is a different one than the search started from: then *beta is its angle.
POSE_HD bool distinct_minimum(const SecondMinFrame &S, double tmin, double *beta) {
  *beta = 2 * atan(tmin);
  return fabs(*beta - S.beta0) > 0.1;
}

// The rotation of the second minimum, back in the camera frame.
POSE_HD M3 second_minimum_rotation(const SecondMinFrame &S, double beta) {
  const double cb = cos(beta), sb = sin(beta);
  const M3 Rbeta{{cb, 0, sb, 0, 1, 0, -sb, 0, cb}};
  return mul(mul(mul(transpose(S.Rt), S.Rgamma), Rbeta), S.RzT);
}

// The better of the two minima into `out` (b200tag_estimate_pose's choice).
POSE_HD void choose_pose(const M3 &R1, const V3 &t1, double err1, const M3 &R2, const V3 &t2, double err2, b200tag_pose *out) {
  const bool first = err1 <= err2;
  POSE_UNROLL for (int k = 0; k < 9; k++) out->R[k] = first ? R1.a[k] : R2.a[k];
  POSE_UNROLL for (int k = 0; k < 3; k++) out->t[k] = first ? t1.v[k] : t2.v[k];
  out->err = first ? err1 : err2;
  out->err_other = first ? err2 : err1;
}

// ---- IPPE (b200tag_estimate_poses_ippe, B200TAG_POSE_IPPE) ----
// Infinitesimal Plane-based Pose Estimation (Collins & Bartoli 2014) of a square tag, the two candidates OpenCV's
// solvePnPGeneric(..., SOLVEPNP_IPPE_SQUARE) returns: the homography from the tag plane to normalised image points, its
// Jacobian at the tag centre, two rotations from the Jacobian in closed form and a least-squares translation for each.
// Only + - * /, sqrt, fabs and fmax: no iteration and no libm transcendental, so host and device agree bit for bit.

// Homography H (row-major, H22 = 1) from the tag plane to the normalised image points u[0..3] of the tag corners
// (-s, s), (s, s), (s, -s), (-s, -s): Heckbert's square-to-quad mapping of the unit square, (X, Y) on the tag being
// ((X + s) / 2s, (s - Y) / 2s) on the square.  False when the quad has no such mapping.
POSE_HD bool square_homography(const V3 *u, double s, double *H) {
  const double x0 = u[0].v[0], y0 = u[0].v[1], x1 = u[1].v[0], y1 = u[1].v[1];
  const double x2 = u[2].v[0], y2 = u[2].v[1], x3 = u[3].v[0], y3 = u[3].v[1];
  const double sx = x0 - x1 + x2 - x3, sy = y0 - y1 + y2 - y3;
  const double dx1 = x1 - x2, dx2 = x3 - x2, dy1 = y1 - y2, dy2 = y3 - y2;
  const double den = dx1 * dy2 - dx2 * dy1;
  if (!(fabs(den) > 0)) return false;
  const double g = (sx * dy2 - dx2 * sy) / den, h = (dx1 * sy - sx * dy1) / den;
  const double a = x1 - x0 + g * x1, b = x3 - x0 + h * x3, d = y1 - y0 + g * y1, e = y3 - y0 + h * y3;
  const double w = 0.5 * (g + h) + 1;  // homogeneous weight of the tag centre
  if (!(fabs(w) > 0)) return false;
  const double k = 0.5 / (s * w);
  H[0] = a * k; H[1] = -b * k; H[2] = (0.5 * (a + b) + x0) / w;
  H[3] = d * k; H[4] = -e * k; H[5] = (0.5 * (d + e) + y0) / w;
  H[6] = g * k; H[7] = -h * k; H[8] = 1;
  return true;
}

// The two IPPE rotations from H.  (p, q) is the image of the tag centre, J the Jacobian of H there, Rv the rotation
// taking e_z to (p, q, 1) / |(p, q, 1)| (Rodrigues' formula about e_z x v, with (1 - cos) / sin^2 = 1 / (n (n + 1))
// so that p = q = 0 gives the identity), A = B^-1 J and gamma its larger singular value.  False when B cannot be
// inverted or gamma is not positive.
POSE_HD bool ippe_rotations(const double *H, M3 *R) {
  const double p = H[2], q = H[5];
  const double J00 = H[0] - H[6] * p, J01 = H[1] - H[7] * p, J10 = H[3] - H[6] * q, J11 = H[4] - H[7] * q;
  const double n = sqrt(p * p + q * q + 1), w = 1 / (n * (n + 1));
  const M3 Rv{{1 - p * p * w, -p * q * w, p / n, -p * q * w, 1 - q * q * w, q / n, -p / n, -q / n, 1 / n}};
  const double B00 = Rv(0, 0) - p * Rv(2, 0), B01 = Rv(0, 1) - p * Rv(2, 1);
  const double B10 = Rv(1, 0) - q * Rv(2, 0), B11 = Rv(1, 1) - q * Rv(2, 1);
  const double detB = B00 * B11 - B01 * B10;
  if (!(fabs(detB) > 0)) return false;
  const double A00 = (B11 * J00 - B01 * J10) / detB, A01 = (B11 * J01 - B01 * J11) / detB;
  const double A10 = (B00 * J10 - B10 * J00) / detB, A11 = (B00 * J11 - B10 * J01) / detB;
  const double a = A00 * A00 + A10 * A10, b = A00 * A01 + A10 * A11, c = A01 * A01 + A11 * A11;
  const double gamma = sqrt(0.5 * (a + c + sqrt((a - c) * (a - c) + 4 * b * b)));
  if (!(gamma > 0)) return false;
  const double r00 = A00 / gamma, r01 = A01 / gamma, r10 = A10 / gamma, r11 = A11 / gamma;
  const double b0 = sqrt(fmax(0.0, 1 - r00 * r00 - r10 * r10));
  double b1 = sqrt(fmax(0.0, 1 - r01 * r01 - r11 * r11));
  if (r00 * r01 + r10 * r11 > 0) b1 = -b1;
  POSE_UNROLL for (int k = 0; k < 2; k++) {
    const double sg = k == 0 ? 1.0 : -1.0;
    const V3 c1{{r00, r10, sg * b0}}, c2{{r01, r11, sg * b1}}, c3 = cross(c1, c2);
    R[k] = mul(Rv, M3{{c1.v[0], c2.v[0], c3.v[0], c1.v[1], c2.v[1], c3.v[1], c1.v[2], c2.v[2], c3.v[2]}});
  }
  return true;
}

// The t minimising the image-plane residuals of R's corners, linearised: for every corner, [1, 0, -u_x] t =
// u_x (R p)_z - (R p)_x and [0, 1, -u_y] t = u_y (R p)_z - (R p)_y, solved through the 3x3 normal equations (whose
// matrix does not depend on R).  False when the corners coincide.
POSE_HD bool ippe_translation(const V3 *u, const V3 *p, const M3 &R, V3 *t) {
  double N02 = 0, N12 = 0, N22 = 0, r0 = 0, r1 = 0, r2 = 0;  // N00 = N11 = 4, N01 = 0
  POSE_UNROLL for (int i = 0; i < 4; i++) {
    const V3 rp = mul(R, p[i]);
    const double ux = u[i].v[0], uy = u[i].v[1];
    const double bx = ux * rp.v[2] - rp.v[0], by = uy * rp.v[2] - rp.v[1];
    N02 -= ux;
    N12 -= uy;
    N22 += ux * ux + uy * uy;
    r0 += bx;
    r1 += by;
    r2 -= ux * bx + uy * by;
  }
  const double det = 16 * N22 - 4 * N12 * N12 - 4 * N02 * N02;
  if (!(fabs(det) > 0)) return false;
  // the adjugate of N (symmetric)
  const double S00 = 4 * N22 - N12 * N12, S01 = N02 * N12, S02 = -4 * N02, S11 = 4 * N22 - N02 * N02, S12 = -4 * N12, S22 = 16;
  *t = V3{{(S00 * r0 + S01 * r1 + S02 * r2) / det, (S01 * r0 + S11 * r1 + S12 * r2) / det, (S02 * r0 + S12 * r1 + S22 * r2) / det}};
  return true;
}

// Object-space error sum |(I - F_j)(R p_j + t)|^2 with F_j = v_j v_j^T / v_j^T v_j, as orthogonal_iteration scores.
POSE_HD double object_space_error(const V3 *v, const V3 *p, const M3 &R, const V3 &t) {
  double err = 0;
  POSE_UNROLL for (int j = 0; j < 4; j++) {
    const V3 e = mul(sub(ident(), outer_over_norm(v[j])), add(mul(R, p[j]), t));
    err += dot(e, e);
  }
  return err;
}

// Both IPPE candidates of the tag with rays v and corners p (rays_and_corners) and their object-space errors; false
// when a candidate cannot be formed (an error is not below HUGE_VAL, which also catches a NaN from overflowing
// intermediates).
POSE_HD bool ippe_candidates(const V3 *v, const V3 *p, double tagsize, M3 *R, V3 *t, double *err) {
  double H[9];
  err[0] = err[1] = HUGE_VAL;
  bool ok = square_homography(v, tagsize / 2.0, H) && ippe_rotations(H, R);
  POSE_UNROLL for (int k = 0; k < 2; k++) {
    ok = ok && ippe_translation(v, p, R[k], &t[k]);
    if (ok) err[k] = object_space_error(v, p, R[k], t[k]);
  }
  return err[0] < HUGE_VAL && err[1] < HUGE_VAL;
}

// The record of a tag without a pose: R = I, t = 0 and both errors HUGE_VAL.
POSE_HD void pose_failure(b200tag_pose *out) {
  const M3 I = ident();
  const V3 z{{0, 0, 0}};
  choose_pose(I, z, HUGE_VAL, I, z, HUGE_VAL, out);
}

// IPPE pose of a tag whose corners are at image points px[0..3]: the candidate with the smaller object-space error,
// the other's error in err_other.  A quad for which a candidate cannot be formed gives pose_failure's record.
POSE_HD void ippe_pose(const double (*px)[2], double tagsize, double fx, double fy, double cx, double cy, b200tag_pose *out) {
  V3 v[4], p[4];
  rays_and_corners(px, tagsize, fx, fy, cx, cy, v, p);
  M3 R[2];
  V3 t[2];
  double err[2];
  if (!ippe_candidates(v, p, tagsize, R, t, err)) {
    pose_failure(out);
    return;
  }
  choose_pose(R[0], t[0], err[0], R[1], t[1], err[1], out);
}

// ---- Lens distortion (b200tag_undistort_points, b200tag_set_pose_distortion) ----
// The 5-coefficient Brown-Conrady model of OpenCV's projectPoints and of the decoder's redistort(): a pinhole point at
// normalised (x, y) = ((u - cx) / fx, (v - cy) / fy) is seen at
//   x' = x (1 + k1 r^2 + k2 r^4 + k3 r^6) + 2 p1 x y + p2 (r^2 + 2 x^2)
//   y' = y (1 + k1 r^2 + k2 r^4 + k3 r^6) + p1 (r^2 + 2 y^2) + 2 p2 x y,   r^2 = x^2 + y^2.
// The pose step inverts it exactly (not with the reference's UnDistort, whose tangential term differs when p2 != 0) by
// Newton's method on the 2x2 system.  Only + - * / and fabs, so host and device agree bit for bit.

struct Distortion {
  double k1, k2, p1, p2, k3;
};

constexpr int kUndistortMaxIterations = 20;

// The model at normalised (x, y): the distorted point and the Jacobian (symmetric, j01 = j10).
POSE_HD void distort_normalised(const Distortion &D, double x, double y, double *xd, double *yd, double *j00, double *j01,
                                double *j11) {
  const double r2 = x * x + y * y;
  const double radial = 1 + r2 * (D.k1 + r2 * (D.k2 + r2 * D.k3));
  const double dr = 2 * (D.k1 + r2 * (2 * D.k2 + r2 * (3 * D.k3)));  // 2 d(radial)/d(r^2)
  *xd = x * radial + 2 * D.p1 * x * y + D.p2 * (r2 + 2 * x * x);
  *yd = y * radial + D.p1 * (r2 + 2 * y * y) + 2 * D.p2 * x * y;
  *j00 = radial + x * x * dr + 2 * D.p1 * y + 6 * D.p2 * x;
  *j01 = x * y * dr + 2 * D.p1 * x + 2 * D.p2 * y;
  *j11 = radial + y * y * dr + 6 * D.p1 * y + 2 * D.p2 * x;
}

// The ideal pixel out[] seen at distorted pixel in[] (in == out is allowed).  Newton's method from the distorted point,
// stopped after a step of at most 1e-14 in both normalised coordinates; false when that takes more than
// kUndistortMaxIterations steps, when the Jacobian's determinant is not positive at some step (past the fold of a strong
// barrel model, where the model is not invertible), or when the result re-distorts more than 1e-9 (normalised) away.
POSE_HD bool undistort_point(const double *in, double fx, double fy, double cx, double cy, const Distortion &D, double *out) {
  const double xd = (in[0] - cx) / fx, yd = (in[1] - cy) / fy;
  double x = xd, y = yd, fxd, fyd, j00, j01, j11;
  bool done = false;
  for (int it = 0; it < kUndistortMaxIterations && !done; it++) {
    distort_normalised(D, x, y, &fxd, &fyd, &j00, &j01, &j11);
    const double det = j00 * j11 - j01 * j01;
    if (!(det > 0)) return false;
    const double ex = xd - fxd, ey = yd - fyd;
    const double dx = (j11 * ex - j01 * ey) / det, dy = (j00 * ey - j01 * ex) / det;
    x = x + dx;
    y = y + dy;
    done = fabs(dx) <= 1e-14 && fabs(dy) <= 1e-14;
  }
  if (!done) return false;
  distort_normalised(D, x, y, &fxd, &fyd, &j00, &j01, &j11);
  if (!(fabs(fxd - xd) <= 1e-9 && fabs(fyd - yd) <= 1e-9)) return false;
  out[0] = fx * x + cx;
  out[1] = fy * y + cy;
  return true;
}

// undistort_point on four corners; false when any fails.
POSE_HD bool undistort_corners(const double (*in)[2], double fx, double fy, double cx, double cy, const Distortion &D,
                               double (*out)[2]) {
  bool ok = true;
  POSE_UNROLL for (int i = 0; i < 4; i++) ok = undistort_point(in[i], fx, fy, cx, cy, D, out[i]) && ok;
  return ok;
}

// Rebuilds det->H and det->c from det->p in the decoder's convention: H maps the tag's (-1, 1), (1, 1), (1, -1),
// (-1, -1) to p[0..3] (H22 = 1), c = H (0, 0).  False when the corners have no such homography.
POSE_HD bool record_homography(b200tag_detection *det) {
  V3 u[4];
  POSE_UNROLL for (int i = 0; i < 4; i++) u[i] = V3{{det->p[i][0], det->p[i][1], 1}};
  double H[9];
  if (!square_homography(u, 1.0, H)) return false;
  POSE_UNROLL for (int k = 0; k < 9; k++) det->H[k] = H[k];
  det->c[0] = H[2];
  det->c[1] = H[5];
  return true;
}

// A detection as a pinhole camera would have recorded it: corners undistorted, H and c rebuilt from them.  False when a
// corner cannot be undistorted or the corners have no homography.
POSE_HD bool undistort_record(b200tag_detection *det, double fx, double fy, double cx, double cy, const Distortion &D) {
  return undistort_corners(det->p, fx, fy, cx, cy, D, det->p) && record_homography(det);
}

// ---- Field pose (b200tag_estimate_field_pose, b200tag_set_field_layout) ----
// One camera-from-field pose (R, t: X_cam = R X_field + t) fitted to the corners of every layout tag in view.  The
// caller selects the detections (field_lookup, field_prefers) and fills one FieldTagData per used tag, in layout order;
// field_solve does the rest.  Every sum over correspondences is taken in one order: correspondence k (tag k / 4, corner
// k % 4) adds into slot k % kFieldSlots in increasing k, and the slots are combined by the xor tree of field_slot_tree.
// The device runs a slot per lane and the tree with __shfl_xor_sync, the host loops; IEEE addition is commutative, so
// every lane and the host hold the same bits.

constexpr int kFieldSlots = 32;
constexpr int kFieldSums = 28;      // cost, J^T r (6), the upper triangle of J^T J (21)
constexpr int kFieldMaxIterations = 20;

// Layout lookup: (family, id) -> layout index, sorted by (family, id).
struct FieldKey {
  int32_t family, id, index, pad;
};
POSE_HD bool key_less(int32_t f0, int32_t i0, int32_t f1, int32_t i1) { return f0 != f1 ? f0 < f1 : i0 < i1; }
POSE_HD int field_lookup(const FieldKey *keys, int n, int32_t family, int32_t id) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (key_less(keys[mid].family, keys[mid].id, family, id)) lo = mid + 1; else hi = mid;
  }
  return lo < n && keys[lo].family == family && keys[lo].id == id ? keys[lo].index : -1;
}

// True when reconcile() prefers detection a to b: lower hamming, then larger decision_margin, then the smaller corner
// coordinates in p order.  False for a tie, which needs identical corners -- and the solve reads nothing else.
POSE_HD bool field_prefers(const b200tag_detection &a, const b200tag_detection &b) {
  double qa[10], qb[10];
  qa[0] = a.hamming; qb[0] = b.hamming;
  qa[1] = -a.decision_margin; qb[1] = -b.decision_margin;
  POSE_UNROLL for (int i = 0; i < 4; i++) {
    qa[2 + 2 * i] = a.p[i][0]; qb[2 + 2 * i] = b.p[i][0];
    qa[3 + 2 * i] = a.p[i][1]; qb[3 + 2 * i] = b.p[i][1];
  }
  POSE_UNROLL for (int k = 0; k < 10; k++) {
    if (qa[k] < qb[k]) return true;
    if (qb[k] < qa[k]) return false;
  }
  return false;
}

// What the solve reads of one used tag: its image corners, the same corners in the field, and its two seeds (each IPPE
// candidate composed with the layout entry into a camera-from-field pose).
struct FieldTagData {
  double px[4][2];
  V3 X[4];
  M3 R[2];
  V3 t[2];
};

struct FieldCamera {
  double fx, fy, cx, cy;
};

// Fills *d for the layout tag L seen at image corners px; false when its IPPE candidates cannot be formed.
POSE_HD bool field_tag_data(const b200tag_field_tag &L, const double (*px)[2], double tagsize, const FieldCamera &cam,
                            FieldTagData *d) {
  V3 v[4], p[4];
  rays_and_corners(px, tagsize, cam.fx, cam.fy, cam.cx, cam.cy, v, p);
  M3 R[2];
  V3 t[2];
  double err[2];
  if (!ippe_candidates(v, p, tagsize, R, t, err)) return false;
  M3 Lr;
  POSE_UNROLL for (int k = 0; k < 9; k++) Lr.a[k] = L.R[k];
  const V3 Lt{{L.t[0], L.t[1], L.t[2]}};
  const M3 LrT = transpose(Lr);
  POSE_UNROLL for (int i = 0; i < 4; i++) {
    d->px[i][0] = px[i][0];
    d->px[i][1] = px[i][1];
    d->X[i] = add(mul(Lr, p[i]), Lt);
  }
  // X_cam = Rc (Lr^T (X_field - Lt)) + tc
  POSE_UNROLL for (int k = 0; k < 2; k++) {
    const M3 Rf = mul(R[k], LrT);
    d->R[k] = Rf;
    d->t[k] = sub(t[k], mul(Rf, Lt));
  }
  return true;
}

// Squared pixel error of one correspondence (image point u, v; field point X) at pose (R, t), HUGE_VAL when the point
// is not in front of the camera.  *Y = R X, *P = R X + t for field_corner_terms.
POSE_HD double field_corner_cost(double u, double v, const V3 &X, const M3 &R, const V3 &t, const FieldCamera &cam, V3 *Y,
                                 V3 *P, double *ru, double *rv) {
  *Y = mul(R, X);
  *P = add(*Y, t);
  if (!(P->v[2] > 0)) return HUGE_VAL;
  const double iz = 1 / P->v[2];
  *ru = cam.fx * (P->v[0] * iz) + cam.cx - u;
  *rv = cam.fy * (P->v[1] * iz) + cam.cy - v;
  return *ru * *ru + *rv * *rv;
}

// Adds one correspondence's cost, J^T r and J^T J into acc[kFieldSums].  J is the Jacobian of the residual for the update
// R <- cayley(c) R, t <- t + dt at c = 0, dt = 0: d(R X + t)/dc = -2 [R X]x.
POSE_HD void field_corner_terms(double u, double v, const V3 &X, const M3 &R, const V3 &t, const FieldCamera &cam, double *acc) {
  V3 Y, P;
  double ru = 0, rv = 0;
  const double e = field_corner_cost(u, v, X, R, t, cam, &Y, &P, &ru, &rv);
  acc[0] += e;
  if (!(e < HUGE_VAL)) return;
  const double iz = 1 / P.v[2];
  const V3 du{{cam.fx * iz, 0, -cam.fx * (P.v[0] * iz) * iz}}, dv{{0, cam.fy * iz, -cam.fy * (P.v[1] * iz) * iz}};
  const V3 cu = cross(Y, du), cv = cross(Y, dv);
  const double Ju[6] = {2 * cu.v[0], 2 * cu.v[1], 2 * cu.v[2], du.v[0], du.v[1], du.v[2]};
  const double Jv[6] = {2 * cv.v[0], 2 * cv.v[1], 2 * cv.v[2], dv.v[0], dv.v[1], dv.v[2]};
  POSE_UNROLL for (int i = 0; i < 6; i++) acc[1 + i] += Ju[i] * ru + Jv[i] * rv;
  int o = 7;
  POSE_UNROLL for (int i = 0; i < 6; i++)
    POSE_UNROLL for (int j = i; j < 6; j++) acc[o++] += Ju[i] * Ju[j] + Jv[i] * Jv[j];
}

// The host's form of the slot tree: slot[l] += slot[l + m] for m = 16, 8, 4, 2, 1; the total ends in slot[0].  A warp
// computes the same with lane l adding lane l ^ m.
template <int K>
inline void field_slot_tree(double (*slot)[K], double *out) {
  for (int m = kFieldSlots / 2; m >= 1; m >>= 1)
    for (int l = 0; l < m; l++)
      for (int j = 0; j < K; j++) slot[l][j] = slot[l][j] + slot[l + m][j];
  for (int j = 0; j < K; j++) out[j] = slot[0][j];
}

// The Cholesky factor A = Lm Lm^T of a symmetric 6x6 matrix (only its lower triangle is read); false when A is not
// positive definite.
POSE_HD bool cholesky6(const double (*A)[6], double (*Lm)[6]) {
  POSE_UNROLL for (int j = 0; j < 6; j++) {
    double s = A[j][j];
    POSE_UNROLL for (int k = 0; k < j; k++) s -= Lm[j][k] * Lm[j][k];
    if (!(s > 0)) return false;
    Lm[j][j] = sqrt(s);
    POSE_UNROLL for (int i = j + 1; i < 6; i++) {
      double r = A[i][j];
      POSE_UNROLL for (int k = 0; k < j; k++) r -= Lm[i][k] * Lm[j][k];
      Lm[i][j] = r / Lm[j][j];
    }
  }
  return true;
}

// Solves (J^T J + lambda diag(J^T J)) d = -J^T r from the sums S by Cholesky; false when the matrix is not positive
// definite.
POSE_HD_CALL bool field_step(const double *S, double lambda, double *d) {
  double A[6][6];
  int o = 7;
  POSE_UNROLL for (int i = 0; i < 6; i++)
    POSE_UNROLL for (int j = i; j < 6; j++) A[i][j] = A[j][i] = S[o++];
  POSE_UNROLL for (int i = 0; i < 6; i++) A[i][i] = A[i][i] + lambda * A[i][i];
  double Lm[6][6] = {};
  if (!cholesky6(A, Lm)) return false;
  double y[6];
  POSE_UNROLL for (int i = 0; i < 6; i++) {
    double r = -S[1 + i];
    POSE_UNROLL for (int k = 0; k < i; k++) r -= Lm[i][k] * y[k];
    y[i] = r / Lm[i][i];
  }
  POSE_UNROLL for (int i = 5; i >= 0; i--) {
    double r = y[i];
    POSE_UNROLL for (int k = i + 1; k < 6; k++) r -= Lm[k][i] * d[k];
    d[i] = r / Lm[i][i];
  }
  return true;
}

// R <- cayley(d[0..2]) R, t <- t + d[3..5]; cayley(c) = ((1 - c.c) I + 2 c c^T + 2 [c]x) / (1 + c.c) is a rotation and
// needs no trigonometry.
POSE_HD void field_update(const M3 &R, const V3 &t, const double *d, M3 *Rn, V3 *tn) {
  const double a = d[0], b = d[1], c = d[2];
  const double n2 = a * a + b * b + c * c, s = 1 / (1 + n2), w = 1 - n2;
  const M3 C{{(w + 2 * a * a) * s, 2 * (a * b - c) * s, 2 * (a * c + b) * s,
              2 * (a * b + c) * s, (w + 2 * b * b) * s, 2 * (b * c - a) * s,
              2 * (a * c - b) * s, 2 * (b * c + a) * s, (w + 2 * c * c) * s}};
  *Rn = mul(C, R);
  *tn = V3{{t.v[0] + d[3], t.v[1] + d[4], t.v[2] + d[5]}};
}

// Levenberg-Marquardt from (*R, *t).  sum(R, t, S) fills S[kFieldSums] with the reduced sums at (R, t).  A step is
// accepted when it lowers the cost (lambda / 10), else rejected (lambda * 10).  The iteration stops after a step of at
// most 1e-10 in every parameter (Cayley vector, metres), accepted or not; after an accepted step that lowers the cost
// by at most 1e-12 of itself; when lambda exceeds 1e8; or after kFieldMaxIterations.
// Returns the final cost; *iterations counts accepted and rejected steps.
template <class SumFn>
POSE_HD double field_refine(SumFn &sum, M3 *R, V3 *t, int *iterations) {
  double S[kFieldSums];
  sum(*R, *t, S);
  double cost = S[0];
  int it = 0;
  if (cost < HUGE_VAL) {
    double lambda = 1e-3;
    while (it < kFieldMaxIterations) {
      it++;
      double d[6];
      if (field_step(S, lambda, d)) {
        M3 Rn;
        V3 tn;
        field_update(*R, *t, d, &Rn, &tn);
        double Sn[kFieldSums];
        sum(Rn, tn, Sn);
        bool small = true;
        POSE_UNROLL for (int j = 0; j < 6; j++) small = small && fabs(d[j]) <= 1e-10;
        if (Sn[0] < cost) {
          small = small || cost - Sn[0] <= 1e-12 * cost;
          *R = Rn;
          *t = tn;
          cost = Sn[0];
          POSE_UNROLL for (int j = 0; j < kFieldSums; j++) S[j] = Sn[j];
          lambda = lambda * 0.1;
          if (small) break;
          continue;
        }
        if (small) break;  // a step this small that does not lower the cost: the minimum, to rounding
      }
      lambda = lambda * 10;
      if (lambda > 1e8) break;
    }
  }
  *iterations = it;
  return cost;
}

POSE_HD void field_empty(b200tag_field_pose *out) {
  out->num_tags = 0;
  out->iterations = 0;
  out->reserved[0] = out->reserved[1] = 0;
  POSE_UNROLL for (int k = 0; k < 9; k++) out->camera_R[k] = out->robot_R[k] = (k % 4 == 0) ? 1.0 : 0.0;
  POSE_UNROLL for (int k = 0; k < 3; k++) out->camera_t[k] = out->robot_t[k] = 0;
  out->rms = out->rms_other = HUGE_VAL;
}

// The record of camera-from-field pose (R, t): the camera and the robot in the field.
POSE_HD void field_result(const M3 &R, const V3 &t, double cost, double cost_other, int ntags, int iterations,
                          const double *rotation, const double *offset, b200tag_field_pose *out) {
  const M3 Rc = transpose(R);
  const V3 tc = scale(mul(Rc, t), -1.0);
  M3 Rx, Rr;
  POSE_UNROLL for (int k = 0; k < 9; k++) Rx.a[k] = rotation[k];
  Rr = mul(Rc, transpose(Rx));
  const V3 tr = sub(tc, mul(Rr, V3{{offset[0], offset[1], offset[2]}}));
  out->num_tags = ntags;
  out->iterations = iterations;
  out->reserved[0] = out->reserved[1] = 0;
  POSE_UNROLL for (int k = 0; k < 9; k++) {
    out->camera_R[k] = Rc.a[k];
    out->robot_R[k] = Rr.a[k];
  }
  POSE_UNROLL for (int k = 0; k < 3; k++) {
    out->camera_t[k] = tc.v[k];
    out->robot_t[k] = tr.v[k];
  }
  const double n = 4.0 * ntags;
  out->rms = sqrt(cost / n);
  out->rms_other = cost_other < HUGE_VAL ? sqrt(cost_other / n) : HUGE_VAL;
}

// The solve over `ntags` used tags (ntags >= 1).  cost(R, t) returns the reduced seed score, sum(R, t, S) the reduced
// sums of field_refine.  Seeds are scored in tag order, candidate 0 before 1, and the first best wins; with one tag
// both candidates are refined, the lower cost returned (candidate 0 on a tie) and the other reported in rms_other.
template <class CostFn, class SumFn>
POSE_HD void field_solve(const FieldTagData *tags, int ntags, CostFn &cost, SumFn &sum, const double *rotation,
                         const double *offset, b200tag_field_pose *out) {
  if (ntags == 1) {
    M3 R0 = tags[0].R[0], R1 = tags[0].R[1];
    V3 t0 = tags[0].t[0], t1 = tags[0].t[1];
    int it0 = 0, it1 = 0;
    const double c0 = field_refine(sum, &R0, &t0, &it0);
    const double c1 = field_refine(sum, &R1, &t1, &it1);
    if (c1 < c0) field_result(R1, t1, c1, c0, 1, it1, rotation, offset, out);
    else field_result(R0, t0, c0, c1, 1, it0, rotation, offset, out);
    return;
  }
  int best = 0;
  double best_cost = HUGE_VAL;
  for (int s = 0; s < 2 * ntags; s++) {
    const double c = cost(tags[s >> 1].R[s & 1], tags[s >> 1].t[s & 1]);
    if (c < best_cost) {
      best_cost = c;
      best = s;
    }
  }
  M3 R = tags[best >> 1].R[best & 1];
  V3 t = tags[best >> 1].t[best & 1];
  int it = 0;
  const double c = field_refine(sum, &R, &t, &it);
  field_result(R, t, c, HUGE_VAL, ntags, it, rotation, offset, out);
}

// ---- Covariance (b200tag_estimate_pose_covariances, b200tag_estimate_field_pose_covariance) ----
// The first-order covariance of the pixel least-squares pose over a set of corners, linearised at a given
// camera-from-X pose (R, t), for xi = (r, dt): R_true = exp([r]x) R, t_true = t + dt (b200tag.h has the definition):
//   C = sigma^2 M^-1 B M^-1,   M = sum_i J_i^T J_i,   B = sum_i J_i^T A_i A_i^T J_i,
// J_i the 2x6 Jacobian of corner i's ideal-image projection, A_i the Jacobian of the undistortion at corner i in pixels.
// Without distortion A_i = I, B = M and C = sigma^2 M^-1: B is not summed.  The field's sums go through its slot order;
// only + - * / and sqrt, so host and device agree bit for bit.

constexpr int kCovSums = 43;  // corners behind the camera, the upper triangles of M (21) and of B (21)

// A_i (2x2, row-major) at ideal pixel (u, v): diag(fx, fy) (dx_d/dx_u)^-1 diag(1/fx, 1/fy), with dx_d/dx_u the model's
// Jacobian at the normalised point; false when its determinant is not positive.
POSE_HD bool undistortion_jacobian(double u, double v, const FieldCamera &cam, const Distortion &D, double *A) {
  double xd, yd, j00, j01, j11;
  distort_normalised(D, (u - cam.cx) / cam.fx, (v - cam.cy) / cam.fy, &xd, &yd, &j00, &j01, &j11);
  const double det = j00 * j11 - j01 * j01;
  if (!(det > 0)) return false;
  A[0] = j11 / det;
  A[1] = -j01 * cam.fx / (cam.fy * det);
  A[2] = -j01 * cam.fy / (cam.fx * det);
  A[3] = j00 / det;
  return true;
}

// Adds the terms of the point X seen at pose (R, t) into acc[kCovSums]: 1 into acc[0] when it is not in front of the
// camera; else J^T J into acc[1..21] and, when A is given, J^T A A^T J into acc[22..42].  d(R X + t) = r x (R X) + dt.
POSE_HD void cov_corner_terms(const V3 &X, const M3 &R, const V3 &t, const FieldCamera &cam, const double *A, double *acc) {
  const V3 Y = mul(R, X), P = add(Y, t);
  if (!(P.v[2] > 0)) {
    acc[0] += 1;
    return;
  }
  const double iz = 1 / P.v[2];
  const V3 du{{cam.fx * iz, 0, -cam.fx * (P.v[0] * iz) * iz}}, dv{{0, cam.fy * iz, -cam.fy * (P.v[1] * iz) * iz}};
  const V3 cu = cross(Y, du), cv = cross(Y, dv);
  const double Ju[6] = {cu.v[0], cu.v[1], cu.v[2], du.v[0], du.v[1], du.v[2]};
  const double Jv[6] = {cv.v[0], cv.v[1], cv.v[2], dv.v[0], dv.v[1], dv.v[2]};
  int o = 1;
  POSE_UNROLL for (int i = 0; i < 6; i++)
    POSE_UNROLL for (int j = i; j < 6; j++) acc[o++] += Ju[i] * Ju[j] + Jv[i] * Jv[j];
  if (!A) return;
  double K0[6], K1[6];  // the rows of A^T J
  POSE_UNROLL for (int i = 0; i < 6; i++) {
    K0[i] = A[0] * Ju[i] + A[2] * Jv[i];
    K1[i] = A[1] * Ju[i] + A[3] * Jv[i];
  }
  POSE_UNROLL for (int i = 0; i < 6; i++)
    POSE_UNROLL for (int j = i; j < 6; j++) acc[o++] += K0[i] * K0[j] + K1[i] * K1[j];
}

// cov_corner_terms for corner c of used field tag g (whose px are already undistorted), with A_i through the lens D
// (null: none); a corner where A_i cannot be formed counts as one behind the camera.
POSE_HD void field_cov_corner_terms(const FieldTagData &g, int c, const M3 &R, const V3 &t, const FieldCamera &cam,
                                    const Distortion *D, double *acc) {
  double A[4] = {1, 0, 0, 1};
  if (D && !undistortion_jacobian(g.px[c][0], g.px[c][1], cam, *D, A)) {
    acc[0] += 1;
    return;
  }
  cov_corner_terms(g.X[c], R, t, cam, D ? A : nullptr, acc);
}

// C = M^-1 B M^-1 (distorted) or M^-1 from the sums S of cov_corner_terms, exactly symmetric; false when a corner is
// behind the camera or M is not positive definite.
POSE_HD bool cov_from_sums(const double *S, bool distorted, double *C) {
  if (!(S[0] == 0)) return false;
  double M[6][6], Lm[6][6] = {};
  int o = 1;
  POSE_UNROLL for (int i = 0; i < 6; i++)
    POSE_UNROLL for (int j = i; j < 6; j++) M[i][j] = M[j][i] = S[o++];
  if (!cholesky6(M, Lm)) return false;
  double Mi[6][6];  // column k solves Lm Lm^T x = e_k
  POSE_UNROLL for (int k = 0; k < 6; k++) {
    double y[6];
    POSE_UNROLL for (int i = 0; i < 6; i++) {
      double r = i == k ? 1.0 : 0.0;
      POSE_UNROLL for (int m = 0; m < i; m++) r -= Lm[i][m] * y[m];
      y[i] = r / Lm[i][i];
    }
    POSE_UNROLL for (int i = 5; i >= 0; i--) {
      double r = y[i];
      POSE_UNROLL for (int m = i + 1; m < 6; m++) r -= Lm[m][i] * Mi[m][k];
      Mi[i][k] = r / Lm[i][i];
    }
  }
  if (!distorted) {
    POSE_UNROLL for (int i = 0; i < 6; i++)
      POSE_UNROLL for (int j = i; j < 6; j++) C[6 * i + j] = C[6 * j + i] = Mi[i][j];
    return true;
  }
  double B[6][6], T[6][6];
  POSE_UNROLL for (int i = 0; i < 6; i++)
    POSE_UNROLL for (int j = i; j < 6; j++) B[i][j] = B[j][i] = S[o++];
  POSE_UNROLL for (int i = 0; i < 6; i++)
    POSE_UNROLL for (int j = 0; j < 6; j++) {
      double s = 0;
      POSE_UNROLL for (int k = 0; k < 6; k++) s += Mi[i][k] * B[k][j];
      T[i][j] = s;
    }
  POSE_UNROLL for (int i = 0; i < 6; i++)
    POSE_UNROLL for (int j = i; j < 6; j++) {
      double s = 0;
      POSE_UNROLL for (int k = 0; k < 6; k++) s += T[i][k] * Mi[k][j];
      C[6 * i + j] = C[6 * j + i] = s;
    }
  return true;
}

// out = G C G^T (6x6, row-major), exactly symmetric; out must not alias C.
POSE_HD void cov_transform(const double *G, const double *C, double *out) {
  double T[36];
  POSE_UNROLL for (int i = 0; i < 6; i++)
    POSE_UNROLL for (int j = 0; j < 6; j++) {
      double s = 0;
      POSE_UNROLL for (int k = 0; k < 6; k++) s += G[6 * i + k] * C[6 * k + j];
      T[6 * i + j] = s;
    }
  POSE_UNROLL for (int i = 0; i < 6; i++)
    POSE_UNROLL for (int j = i; j < 6; j++) {
      double s = 0;
      POSE_UNROLL for (int k = 0; k < 6; k++) s += T[6 * i + k] * G[6 * j + k];
      out[6 * i + j] = out[6 * j + i] = s;
    }
}

// The last step: C * sigma^2 when ok, else all HUGE_VAL.  Scaling last makes C(2 sigma) = 4 C(sigma) bit for bit.
POSE_HD void cov_scale(bool ok, double sigma, double *C) {
  const double s2 = sigma * sigma;
  POSE_UNROLL for (int k = 0; k < 36; k++) C[k] = ok ? C[k] * s2 : HUGE_VAL;
}

// The covariance of tag pose `pose` (camera frame) from the tag's raw image corners `raw`, through the lens D (null:
// none), into C[36]; all HUGE_VAL for a failed record, a corner that cannot be undistorted or is behind the camera, or
// an M that is not positive definite.
POSE_HD void tag_covariance(const double (*raw)[2], const b200tag_pose &pose, double tagsize, const FieldCamera &cam,
                            const Distortion *D, double sigma, double *C) {
  bool ok = pose.err < HUGE_VAL;
  M3 R;
  POSE_UNROLL for (int k = 0; k < 9; k++) R.a[k] = pose.R[k];
  const V3 t{{pose.t[0], pose.t[1], pose.t[2]}};
  const double s = tagsize / 2.0;
  const V3 X[4] = {V3{{-s, s, 0}}, V3{{s, s, 0}}, V3{{s, -s, 0}}, V3{{-s, -s, 0}}};
  double S[kCovSums] = {};
  POSE_UNROLL for (int i = 0; i < 4; i++) {
    double A[4] = {1, 0, 0, 1}, u[2];
    if (D) ok = ok && undistort_point(raw[i], cam.fx, cam.fy, cam.cx, cam.cy, *D, u) && undistortion_jacobian(u[0], u[1], cam, *D, A);
    cov_corner_terms(X[i], R, t, cam, D ? A : nullptr, S);
  }
  ok = ok && cov_from_sums(S, D != nullptr, C);
  cov_scale(ok, sigma, C);
}

// The camera-from-field pose at which field record `res` is linearised: R = camera_R^T, t = -R camera_t.
POSE_HD void field_cov_pose(const b200tag_field_pose &res, M3 *R, V3 *t) {
  M3 Rc;
  POSE_UNROLL for (int k = 0; k < 9; k++) Rc.a[k] = res.camera_R[k];
  *R = transpose(Rc);
  *t = scale(mul(*R, V3{{res.camera_t[0], res.camera_t[1], res.camera_t[2]}}), -1.0);
}

// The covariances of field record `res` from the reduced sums S (kCovSums; B only when distorted) at field_cov_pose(res).
// The solve's xi (a, b) perturbs the camera-from-field pose in the camera frame; the camera in the field (Rc, tc) moves
// by r = -Rc a, dt = -Rc b + [tc]x Rc a, and the robot (Rr, tr = tc - Rr offset) by r, dt + [Rr offset]x r.  All
// HUGE_VAL when no tag was used or cov_from_sums fails.
POSE_HD_CALL void field_covariance(const double *S, bool distorted, const b200tag_field_pose &res, const double *offset,
                                   double sigma, b200tag_field_covariance *out) {
  double Cs[36] = {};
  const bool ok = res.num_tags > 0 && cov_from_sums(S, distorted, Cs);
  const double *Rc = res.camera_R, *tc = res.camera_t;
  double G[36] = {};
  POSE_UNROLL for (int i = 0; i < 3; i++)
    POSE_UNROLL for (int j = 0; j < 3; j++) {
      G[6 * i + j] = -Rc[3 * i + j];
      G[6 * (i + 3) + j + 3] = -Rc[3 * i + j];
      // row i of [tc]x times column j of Rc
      const int a = (i + 1) % 3, b = (i + 2) % 3;
      G[6 * (i + 3) + j] = tc[a] * Rc[3 * b + j] - tc[b] * Rc[3 * a + j];
    }
  cov_transform(G, Cs, out->camera);
  double q[3];
  POSE_UNROLL for (int i = 0; i < 3; i++)
    q[i] = res.robot_R[3 * i] * offset[0] + res.robot_R[3 * i + 1] * offset[1] + res.robot_R[3 * i + 2] * offset[2];
  double H[36] = {};
  POSE_UNROLL for (int i = 0; i < 6; i++) H[7 * i] = 1;
  POSE_UNROLL for (int i = 0; i < 3; i++) {
    const int a = (i + 1) % 3, b = (i + 2) % 3;
    H[6 * (i + 3) + a] = -q[b];  // [q]x: row i has -q[b] at column a and q[a] at column b
    H[6 * (i + 3) + b] = q[a];
  }
  cov_transform(H, out->camera, out->robot);
  cov_scale(ok, sigma, out->camera);
  cov_scale(ok, sigma, out->robot);
}

// ---- Floor pose (b200tag_estimate_floor_pose, b200tag_set_floor_pose) ----
// The robot on a flat floor: robot_R = Rz(theta), robot_t = (x, y, 0), so the camera-from-field pose maps a field point
// X to P = rotation^T (Rz^T (X - (x, y, 0)) - offset).  The heading is held as (c, s) = (cos theta, sin theta) and
// turned by the 2-D Cayley map.  The correspondences are the field pose's (FieldTagData, its slot order); the optional
// heading prior rho = w 2 (s cg - c sg) / (1 + c cg + s sg) is added once, after the reduction.  Unknowns (x, y, theta),
// or (x, y) in fixed mode, where (c, s) = (cg, sg).  Only + - * /, sqrt and fabs: host and device agree bit for bit.

constexpr int kFloorSums = 10;     // cost, J^T r (3), the upper triangle of J^T J (6): xx xy xt yy yt tt
constexpr int kFloorLinSums = 5;   // the heading seed's normal matrix (xx, xy, yy) and right-hand side (2)
constexpr int kFloorCovSums = 13;  // corners behind the camera, the upper triangles of H (6) and of M (6)

// The setting of one solve: extrinsics, mode (B200TAG_FLOOR_*), gyro heading (cg, sg; unused in free mode), weight w.
struct FloorModel {
  double rot[9], off[3];
  int mode;
  double cg, sg, w;
};

struct FloorState {
  double x, y, c, s;
};

// The mode of heading (cg, sg) (NaN: none) at weight w (+inf: fixed).
POSE_HD int floor_mode(double cg, double w) {
  return cg != cg ? B200TAG_FLOOR_FREE : (w < HUGE_VAL ? B200TAG_FLOOR_PRIOR : B200TAG_FLOOR_FIXED);
}

// Pixel residual of one correspondence (image point u, v; field point X) at state st, HUGE_VAL when the point is not
// in front of the camera.  *W = Rz^T (X - p), *P the camera-frame point.
POSE_HD double floor_corner_cost(double u, double v, const V3 &X, const FloorState &st, const FloorModel &m,
                                 const FieldCamera &cam, V3 *W, V3 *P, double *ru, double *rv) {
  const double dx = X.v[0] - st.x, dy = X.v[1] - st.y;
  *W = V3{{st.c * dx + st.s * dy, st.c * dy - st.s * dx, X.v[2]}};
  const V3 Q{{W->v[0] - m.off[0], W->v[1] - m.off[1], W->v[2] - m.off[2]}};
  POSE_UNROLL for (int i = 0; i < 3; i++) P->v[i] = m.rot[i] * Q.v[0] + m.rot[3 + i] * Q.v[1] + m.rot[6 + i] * Q.v[2];
  if (!(P->v[2] > 0)) return HUGE_VAL;
  const double iz = 1 / P->v[2];
  *ru = cam.fx * (P->v[0] * iz) + cam.cx - u;
  *rv = cam.fy * (P->v[1] * iz) + cam.cy - v;
  return *ru * *ru + *rv * *rv;
}

// The 1x3 rows Ju, Jv of d(ru, rv)/d(x, y, theta) at (W, P): dW/dx = (-c, s, 0), dW/dy = (-s, -c, 0),
// dW/dtheta = (W1, -W0, 0), dP = rotation^T dW.
POSE_HD void floor_jacobian(const V3 &W, const V3 &P, const FloorState &st, const FloorModel &m, const FieldCamera &cam,
                            double *Ju, double *Jv) {
  const double iz = 1 / P.v[2];
  const V3 du{{cam.fx * iz, 0, -cam.fx * (P.v[0] * iz) * iz}}, dv{{0, cam.fy * iz, -cam.fy * (P.v[1] * iz) * iz}};
  double a[2], b[2];  // the first two entries of rotation du, rotation dv
  POSE_UNROLL for (int j = 0; j < 2; j++) {
    a[j] = m.rot[3 * j] * du.v[0] + m.rot[3 * j + 1] * du.v[1] + m.rot[3 * j + 2] * du.v[2];
    b[j] = m.rot[3 * j] * dv.v[0] + m.rot[3 * j + 1] * dv.v[1] + m.rot[3 * j + 2] * dv.v[2];
  }
  Ju[0] = st.s * a[1] - st.c * a[0];
  Ju[1] = -(st.s * a[0] + st.c * a[1]);
  Ju[2] = a[0] * W.v[1] - a[1] * W.v[0];
  Jv[0] = st.s * b[1] - st.c * b[0];
  Jv[1] = -(st.s * b[0] + st.c * b[1]);
  Jv[2] = b[0] * W.v[1] - b[1] * W.v[0];
}

// Adds one correspondence's cost, J^T r and J^T J into acc[kFloorSums].
POSE_HD void floor_corner_terms(double u, double v, const V3 &X, const FloorState &st, const FloorModel &m,
                                const FieldCamera &cam, double *acc) {
  V3 W, P;
  double ru = 0, rv = 0;
  const double e = floor_corner_cost(u, v, X, st, m, cam, &W, &P, &ru, &rv);
  acc[0] += e;
  if (!(e < HUGE_VAL)) return;
  double Ju[3], Jv[3];
  floor_jacobian(W, P, st, m, cam, Ju, Jv);
  POSE_UNROLL for (int i = 0; i < 3; i++) acc[1 + i] += Ju[i] * ru + Jv[i] * rv;
  int o = 4;
  POSE_UNROLL for (int i = 0; i < 3; i++)
    POSE_UNROLL for (int j = i; j < 3; j++) acc[o++] += Ju[i] * Ju[j] + Jv[i] * Jv[j];
}

// The heading prior at st: false when 1 + cos(theta - theta_g) <= 0; else rho and g = d rho / d theta.
POSE_HD bool floor_prior(const FloorState &st, const FloorModel &m, double *rho, double *g) {
  const double D = 1 + st.c * m.cg + st.s * m.sg;
  if (!(D > 0)) return false;
  *rho = m.w * (2 * (st.s * m.cg - st.c * m.sg)) / D;
  *g = 2 * m.w / D;
  return true;
}

// The prior's terms added to reduced sums S (kFloorSums) in prior mode; S[0] = HUGE_VAL where it is not defined.
POSE_HD void floor_add_prior(const FloorState &st, const FloorModel &m, double *S) {
  if (m.mode != B200TAG_FLOOR_PRIOR) return;
  double rho, g;
  if (!floor_prior(st, m, &rho, &g)) {
    S[0] = HUGE_VAL;
    return;
  }
  S[0] = S[0] + rho * rho;
  S[3] = S[3] + g * rho;
  S[9] = S[9] + g * g;
}

// The seed score E from the reduced pixel cost e at st.
POSE_HD double floor_score(double e, const FloorState &st, const FloorModel &m) {
  if (m.mode != B200TAG_FLOOR_PRIOR) return e;
  double rho, g;
  return floor_prior(st, m, &rho, &g) ? e + rho * rho : HUGE_VAL;
}

// The Cholesky factor of a symmetric N x N matrix (lower triangle read), N = 2 or 3; false when not positive definite.
template <int N>
POSE_HD bool cholesky_small(const double (*A)[N], double (*Lm)[N]) {
  POSE_UNROLL for (int j = 0; j < N; j++) {
    double s = A[j][j];
    POSE_UNROLL for (int k = 0; k < j; k++) s -= Lm[j][k] * Lm[j][k];
    if (!(s > 0)) return false;
    Lm[j][j] = sqrt(s);
    POSE_UNROLL for (int i = j + 1; i < N; i++) {
      double r = A[i][j];
      POSE_UNROLL for (int k = 0; k < j; k++) r -= Lm[i][k] * Lm[j][k];
      Lm[i][j] = r / Lm[j][j];
    }
  }
  return true;
}

// Solves Lm Lm^T x = b.
template <int N>
POSE_HD void cholesky_solve(const double (*Lm)[N], const double *b, double *x) {
  double y[N];
  POSE_UNROLL for (int i = 0; i < N; i++) {
    double r = b[i];
    POSE_UNROLL for (int k = 0; k < i; k++) r -= Lm[i][k] * y[k];
    y[i] = r / Lm[i][i];
  }
  POSE_UNROLL for (int i = N - 1; i >= 0; i--) {
    double r = y[i];
    POSE_UNROLL for (int k = i + 1; k < N; k++) r -= Lm[k][i] * x[k];
    x[i] = r / Lm[i][i];
  }
}

// The full 3x3 matrix of an upper triangle (xx xy xt yy yt tt).
POSE_HD void floor_sym3(const double *u, double (*A)[3]) {
  A[0][0] = u[0]; A[0][1] = A[1][0] = u[1]; A[0][2] = A[2][0] = u[2];
  A[1][1] = u[3]; A[1][2] = A[2][1] = u[4]; A[2][2] = u[5];
}

// Solves (J^T J + lambda diag(J^T J)) d = -J^T r over the first N unknowns; false when not positive definite.
template <int N>
POSE_HD bool floor_step(const double *S, double lambda, double *d) {
  double F[3][3], A[N][N], Lm[N][N] = {}, b[N];
  floor_sym3(S + 4, F);
  POSE_UNROLL for (int i = 0; i < N; i++) {
    POSE_UNROLL for (int j = 0; j < N; j++) A[i][j] = F[i][j];
    A[i][i] = A[i][i] + lambda * A[i][i];
    b[i] = -S[1 + i];
  }
  if (!cholesky_small<N>(A, Lm)) return false;
  cholesky_solve<N>(Lm, b, d);
  return true;
}

// x, y += d[0], d[1]; with N = 3 the heading turns by phi, cos phi = (1 - d^2/4) / (1 + d^2/4),
// sin phi = d / (1 + d^2/4) for d = d[2].
template <int N>
POSE_HD FloorState floor_update(const FloorState &st, const double *d) {
  FloorState n{st.x + d[0], st.y + d[1], st.c, st.s};
  if (N == 3) {
    const double q = d[N - 1] * d[N - 1] / 4, den = 1 + q, cp = (1 - q) / den, sp = d[N - 1] / den;
    n.c = st.c * cp - st.s * sp;
    n.s = st.s * cp + st.c * sp;
  }
  return n;
}

// Levenberg-Marquardt from *st over the first N unknowns, with field_refine's stop rules.  sum(st, S) fills
// S[kFloorSums] with the reduced pixel sums at st; the prior is added here.  Returns the final E; *pixel is its pixel
// part and *iterations counts accepted and rejected steps.
template <int N, class SumFn>
POSE_HD double floor_refine(SumFn &sum, const FloorModel &m, FloorState *st, double *pixel, int *iterations) {
  double S[kFloorSums];
  sum(*st, S);
  *pixel = S[0];
  floor_add_prior(*st, m, S);
  double cost = S[0];
  int it = 0;
  if (cost < HUGE_VAL) {
    double lambda = 1e-3;
    while (it < kFieldMaxIterations) {
      it++;
      double d[N];
      if (floor_step<N>(S, lambda, d)) {
        const FloorState sn = floor_update<N>(*st, d);
        double Sn[kFloorSums];
        sum(sn, Sn);
        const double pn = Sn[0];
        floor_add_prior(sn, m, Sn);
        bool small = true;
        POSE_UNROLL for (int j = 0; j < N; j++) small = small && fabs(d[j]) <= 1e-10;
        if (Sn[0] < cost) {
          small = small || cost - Sn[0] <= 1e-12 * cost;
          *st = sn;
          cost = Sn[0];
          *pixel = pn;
          POSE_UNROLL for (int j = 0; j < kFloorSums; j++) S[j] = Sn[j];
          lambda = lambda * 0.1;
          if (small) break;
          continue;
        }
        if (small) break;
      }
      lambda = lambda * 10;
      if (lambda > 1e8) break;
    }
  }
  *iterations = it;
  return cost;
}

// The floor seed of camera-from-field pose (R, t): the robot pose projected onto the floor, (c, s) the normalised
// horizontal part of robot_R's first column (the gyro's in fixed mode); false when that part is zero.
POSE_HD bool floor_seed(const M3 &R, const V3 &t, const FloorModel &m, FloorState *st) {
  const M3 Rc = transpose(R);
  const V3 tc = scale(mul(Rc, t), -1.0);
  M3 Rx;
  POSE_UNROLL for (int k = 0; k < 9; k++) Rx.a[k] = m.rot[k];
  const M3 Rr = mul(Rc, transpose(Rx));
  const V3 tr = sub(tc, mul(Rr, V3{{m.off[0], m.off[1], m.off[2]}}));
  const double h = sqrt(Rr(0, 0) * Rr(0, 0) + Rr(1, 0) * Rr(1, 0));
  if (!(h > 0)) return false;
  *st = FloorState{tr.v[0], tr.v[1], Rr(0, 0) / h, Rr(1, 0) / h};
  if (m.mode == B200TAG_FLOOR_FIXED) {
    st->c = m.cg;
    st->s = m.sg;
  }
  return true;
}

// Adds one correspondence's terms of the heading seed into acc[kFloorLinSums]: m_k x (P0 + x bx + y by) = 0 with m_k
// the ideal normalised ray, P0 = rotation^T (Rz^T X - offset), bx = -rotation^T Rz^T e_x, by = -rotation^T Rz^T e_y
// at the gyro heading.
POSE_HD void floor_lin_terms(double u, double v, const V3 &X, const FloorModel &m, const FieldCamera &cam, double *acc) {
  const V3 ray{{(u - cam.cx) / cam.fx, (v - cam.cy) / cam.fy, 1}};
  const FloorState g{0, 0, m.cg, m.sg};
  V3 W, P0;
  double ru, rv;
  floor_corner_cost(u, v, X, g, m, cam, &W, &P0, &ru, &rv);
  const double qx[3] = {-m.cg, m.sg, 0}, qy[3] = {-m.sg, -m.cg, 0};
  V3 bx, by;
  POSE_UNROLL for (int i = 0; i < 3; i++) {
    bx.v[i] = m.rot[i] * qx[0] + m.rot[3 + i] * qx[1];
    by.v[i] = m.rot[i] * qy[0] + m.rot[3 + i] * qy[1];
  }
  const V3 ex = cross(ray, bx), ey = cross(ray, by), e0 = cross(ray, P0);
  acc[0] += dot(ex, ex);
  acc[1] += dot(ex, ey);
  acc[2] += dot(ey, ey);
  acc[3] += dot(ex, e0);
  acc[4] += dot(ey, e0);
}

// The heading seed from the reduced sums S (kFloorLinSums); false when the normal matrix is not positive definite.
POSE_HD bool floor_lin_seed(const double *S, const FloorModel &m, FloorState *st) {
  const double A[2][2] = {{S[0], S[1]}, {S[1], S[2]}};
  double Lm[2][2] = {}, q[2];
  if (!cholesky_small<2>(A, Lm)) return false;
  const double b[2] = {-S[3], -S[4]};
  cholesky_solve<2>(Lm, b, q);
  *st = FloorState{q[0], q[1], m.cg, m.sg};
  return true;
}

POSE_HD void floor_empty(int mode, b200tag_floor_pose *out) {
  out->num_tags = 0;
  out->iterations = 0;
  out->mode = mode;
  out->reserved = 0;
  out->x = out->y = 0;
  out->cos_heading = 1;
  out->sin_heading = 0;
  out->heading = 0;
  out->rms = out->rms_other = HUGE_VAL;
}

POSE_HD void floor_result(const FloorState &st, double pixel, double pixel_other, int ntags, int iterations, int mode,
                          b200tag_floor_pose *out) {
  out->num_tags = ntags;
  out->iterations = iterations;
  out->mode = mode;
  out->reserved = 0;
  out->x = st.x;
  out->y = st.y;
  out->cos_heading = st.c;
  out->sin_heading = st.s;
  out->heading = 0;  // atan2(sin, cos), filled on the host
  const double n = 4.0 * ntags;
  out->rms = pixel < HUGE_VAL ? sqrt(pixel / n) : HUGE_VAL;
  out->rms_other = pixel_other < HUGE_VAL ? sqrt(pixel_other / n) : HUGE_VAL;
}

// The solve over `ntags` used tags (ntags >= 1).  cost(st) returns the reduced pixel cost, sum(st, S) the reduced pixel
// sums of floor_refine, lin(S) the reduced sums of floor_lin_terms.  Seeds, scored by E in order with the first best
// winning: every used tag's IPPE candidates (0 first), then, with a heading, the linear (x, y) at the gyro heading.  In
// free mode with one tag each candidate's seed is refined and the lower cost returned (candidate 0 on a tie), the other
// in rms_other.  Without any seed the start is x = y = 0 at heading 0.
template <class CostFn, class SumFn, class LinFn>
POSE_HD void floor_solve(const FieldTagData *tags, int ntags, const FloorModel &m, CostFn &cost, SumFn &sum, LinFn &lin,
                         b200tag_floor_pose *out) {
  if (m.mode == B200TAG_FLOOR_FREE && ntags == 1) {
    FloorState st[2];
    double c[2], p[2];
    int it[2];
    POSE_UNROLL for (int k = 0; k < 2; k++) {
      st[k] = FloorState{0, 0, 1, 0};
      c[k] = p[k] = HUGE_VAL;
      it[k] = 0;
      if (floor_seed(tags[0].R[k], tags[0].t[k], m, &st[k])) c[k] = floor_refine<3>(sum, m, &st[k], &p[k], &it[k]);
    }
    const int b = c[1] < c[0] ? 1 : 0;
    floor_result(st[b], p[b], p[1 - b], 1, it[b], m.mode, out);
    return;
  }
  FloorState best{0, 0, 1, 0};
  if (m.mode == B200TAG_FLOOR_FIXED) {
    best.c = m.cg;
    best.s = m.sg;
  }
  double best_cost = HUGE_VAL;
  bool any = false;
  for (int s = 0; s < 2 * ntags; s++) {
    FloorState st;
    if (!floor_seed(tags[s >> 1].R[s & 1], tags[s >> 1].t[s & 1], m, &st)) continue;
    const double e = floor_score(cost(st), st, m);
    if (!any || e < best_cost) {
      best = st;
      best_cost = e;
      any = true;
    }
  }
  if (m.mode != B200TAG_FLOOR_FREE) {
    double S[kFloorLinSums];
    lin(S);
    FloorState st;
    if (floor_lin_seed(S, m, &st)) {
      const double e = floor_score(cost(st), st, m);
      if (!any || e < best_cost) best = st;
    }
  }
  double pixel;
  int it = 0;
  if (m.mode == B200TAG_FLOOR_FIXED) floor_refine<2>(sum, m, &best, &pixel, &it);
  else floor_refine<3>(sum, m, &best, &pixel, &it);
  floor_result(best, pixel, HUGE_VAL, ntags, it, m.mode, out);
}

// Adds the covariance terms of corner c of used tag g at state st into acc[kFloorCovSums]: 1 into acc[0] when it is
// behind the camera or A_i cannot be formed; else J^T J into acc[1..6] and, with the lens D, J^T A A^T J into
// acc[7..12].
POSE_HD void floor_cov_corner_terms(const FieldTagData &g, int c, const FloorState &st, const FloorModel &m,
                                    const FieldCamera &cam, const Distortion *D, double *acc) {
  double A[4] = {1, 0, 0, 1};
  if (D && !undistortion_jacobian(g.px[c][0], g.px[c][1], cam, *D, A)) {
    acc[0] += 1;
    return;
  }
  V3 W, P;
  double ru, rv;
  if (!(floor_corner_cost(g.px[c][0], g.px[c][1], g.X[c], st, m, cam, &W, &P, &ru, &rv) < HUGE_VAL)) {
    acc[0] += 1;
    return;
  }
  double Ju[3], Jv[3];
  floor_jacobian(W, P, st, m, cam, Ju, Jv);
  int o = 1;
  POSE_UNROLL for (int i = 0; i < 3; i++)
    POSE_UNROLL for (int j = i; j < 3; j++) acc[o++] += Ju[i] * Ju[j] + Jv[i] * Jv[j];
  if (!D) return;
  double K0[3], K1[3];  // the rows of A^T J
  POSE_UNROLL for (int i = 0; i < 3; i++) {
    K0[i] = A[0] * Ju[i] + A[2] * Jv[i];
    K1[i] = A[1] * Ju[i] + A[3] * Jv[i];
  }
  POSE_UNROLL for (int i = 0; i < 3; i++)
    POSE_UNROLL for (int j = i; j < 3; j++) acc[o++] += K0[i] * K0[j] + K1[i] * K1[j];
}

// C = Hi M Hi (distorted) or Hi over the first N unknowns, Hi = H^-1; the rest of the 3x3 C is 0.
template <int N>
POSE_HD bool floor_cov_solve(const double (*H)[3], const double (*M)[3], bool distorted, double *C) {
  double A[N][N], Lm[N][N] = {}, Hi[N][N];
  POSE_UNROLL for (int i = 0; i < N; i++)
    POSE_UNROLL for (int j = 0; j < N; j++) A[i][j] = H[i][j];
  if (!cholesky_small<N>(A, Lm)) return false;
  POSE_UNROLL for (int k = 0; k < N; k++) {
    double e[N], x[N];
    POSE_UNROLL for (int i = 0; i < N; i++) e[i] = i == k ? 1.0 : 0.0;
    cholesky_solve<N>(Lm, e, x);
    POSE_UNROLL for (int i = 0; i < N; i++) Hi[i][k] = x[i];
  }
  POSE_UNROLL for (int k = 0; k < 9; k++) C[k] = 0;
  if (!distorted) {
    POSE_UNROLL for (int i = 0; i < N; i++)
      POSE_UNROLL for (int j = i; j < N; j++) C[3 * i + j] = C[3 * j + i] = Hi[i][j];
    return true;
  }
  double T[N][N];
  POSE_UNROLL for (int i = 0; i < N; i++)
    POSE_UNROLL for (int j = 0; j < N; j++) {
      double s = 0;
      POSE_UNROLL for (int k = 0; k < N; k++) s += Hi[i][k] * M[k][j];
      T[i][j] = s;
    }
  POSE_UNROLL for (int i = 0; i < N; i++)
    POSE_UNROLL for (int j = i; j < N; j++) {
      double s = 0;
      POSE_UNROLL for (int k = 0; k < N; k++) s += T[i][k] * Hi[k][j];
      C[3 * i + j] = C[3 * j + i] = s;
    }
  return true;
}

// The 3x3 covariance of (x, y, theta) of floor record `res` from the reduced sums S (kFloorCovSums; M only when
// distorted): sigma^2 H^-1 M H^-1, H = J^T J + g g^T, M = sum J_i^T A_i A_i^T J_i + g g^T, g the prior's gradient
// (prior mode only).  Fixed mode: the (x, y) block, theta's row and column 0.  All HUGE_VAL when no tag was used, a
// corner failed, the prior is undefined or H is not positive definite.
POSE_HD_CALL void floor_covariance(const double *S, bool distorted, const b200tag_floor_pose &res, const FloorModel &m,
                                   double sigma, double *C) {
  bool ok = res.num_tags > 0 && S[0] == 0;
  double H[3][3], M[3][3];
  floor_sym3(S + 1, H);
  floor_sym3(distorted ? S + 7 : S + 1, M);
  if (m.mode == B200TAG_FLOOR_PRIOR) {
    double rho, g;
    const FloorState st{res.x, res.y, res.cos_heading, res.sin_heading};
    if (floor_prior(st, m, &rho, &g)) {
      H[2][2] = H[2][2] + g * g;
      M[2][2] = M[2][2] + g * g;
    } else {
      ok = false;
    }
  }
  if (ok) ok = m.mode == B200TAG_FLOOR_FIXED ? floor_cov_solve<2>(H, M, distorted, C) : floor_cov_solve<3>(H, M, distorted, C);
  const double s2 = sigma * sigma;
  POSE_UNROLL for (int k = 0; k < 9; k++) C[k] = ok ? C[k] * s2 : HUGE_VAL;
}

}  // namespace pose

// Host, pose.cc: the node's records from poses already estimated (robot frame, distance, closest first), the step
// b200tag_locate_tags and b200tag_tag_positions share.  poses[i] belongs to dets[i].
void locate_from_poses(const b200tag_detection *dets, const b200tag_pose *poses, int count, const double *rotation,
                       const double *offset, b200tag_tag_position *out);

// Host, pose.cc: the checks of b200tag_estimate_field_pose on a layout, plus, when `ncodes` is given, family < nfamilies
// and id < ncodes[family].  On success fills `keys` (nlayout entries, sorted) and returns true.
bool field_layout_keys(const b200tag_field_tag *layout, int nlayout, const uint32_t *ncodes, int nfamilies, pose::FieldKey *keys);

// Host, pose.cc: the check of a `dist` argument ({k1, k2, p1, p2, k3} or NULL): false when a coefficient is not finite.
// *active is true when a coefficient is non-zero; only then is there an undistortion step, and *D holds the model.
bool read_distortion(const double *dist, bool *active, pose::Distortion *D);

// Host, pose.cc: the check of a covariance's sigma: finite and > 0.
bool valid_sigma(double sigma);

// Host, pose.cc: the gyro heading's (cos, sin) with the host's libm, both NaN for a NaN heading.
void floor_gyro(double heading, double *cg, double *sg);

// Host, pose.cc: the checks of b200tag_estimate_floor_pose on heading (not infinite) and heading_weight (> 0, +inf
// allowed); on success fills *m (rotation / offset NULL: identity / zero).
bool floor_model(const double *rotation, const double *offset, double heading, double heading_weight, pose::FloorModel *m);

}  // namespace b200tag

#endif  // B200TAG_POSE_CORE_H_
