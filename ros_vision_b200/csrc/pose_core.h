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
// every sum over correspondences taken in one order on both sides.
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

// IPPE pose of a tag whose corners are at image points px[0..3]: the candidate with the smaller object-space error,
// the other's error in err_other.  A quad for which a candidate cannot be formed gives R = I, t = 0 and both errors
// HUGE_VAL.
POSE_HD void ippe_pose(const double (*px)[2], double tagsize, double fx, double fy, double cx, double cy, b200tag_pose *out) {
  V3 v[4], p[4];
  rays_and_corners(px, tagsize, fx, fy, cx, cy, v, p);
  M3 R[2];
  V3 t[2];
  double err[2];
  if (!ippe_candidates(v, p, tagsize, R, t, err)) {
    const M3 I = ident();
    const V3 z{{0, 0, 0}};
    choose_pose(I, z, HUGE_VAL, I, z, HUGE_VAL, out);
    return;
  }
  choose_pose(R[0], t[0], err[0], R[1], t[1], err[1], out);
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

// Solves (J^T J + lambda diag(J^T J)) d = -J^T r from the sums S by Cholesky; false when the matrix is not positive
// definite.
POSE_HD_CALL bool field_step(const double *S, double lambda, double *d) {
  double A[6][6];
  int o = 7;
  POSE_UNROLL for (int i = 0; i < 6; i++)
    POSE_UNROLL for (int j = i; j < 6; j++) A[i][j] = A[j][i] = S[o++];
  POSE_UNROLL for (int i = 0; i < 6; i++) A[i][i] = A[i][i] + lambda * A[i][i];
  double Lm[6][6] = {};
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

}  // namespace pose

// Host, pose.cc: the node's records from poses already estimated (robot frame, distance, closest first), the step
// b200tag_locate_tags and b200tag_tag_positions share.  poses[i] belongs to dets[i].
void locate_from_poses(const b200tag_detection *dets, const b200tag_pose *poses, int count, const double *rotation,
                       const double *offset, b200tag_tag_position *out);

// Host, pose.cc: the checks of b200tag_estimate_field_pose on a layout, plus, when `ncodes` is given, family < nfamilies
// and id < ncodes[family].  On success fills `keys` (nlayout entries, sorted) and returns true.
bool field_layout_keys(const b200tag_field_tag *layout, int nlayout, const uint32_t *ncodes, int nfamilies, pose::FieldKey *keys);

}  // namespace b200tag

#endif  // B200TAG_POSE_CORE_H_
