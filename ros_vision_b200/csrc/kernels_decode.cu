// Decode stage of the B200 AprilTag engine (sm_100a): one warp per candidate quad does
//   edge refinement with camera un/re-distortion     (reference: apriltag_detect.cu:307-564, CPU)
//   homography, gray model, 36 bilinear bit samples, sharpening, code lookup, detection
//                                                    (quad_decode_index in the libapriltag fork, CPU)
// The reference copies the full-resolution gray image back to the host (apriltag_gpu.cu:740) and
// runs all of this on a CPU worker pool; here the gray image never leaves HBM and only the
// ~176-byte detection records are returned.  Samples are computed lane-parallel, then folded
// in the reference's sequential order by one lane so sums match the CPU arithmetic.
// Compiled with -fmad=false (see kernels_blobs.cu).
#include <cuda_runtime.h>
#include <stdint.h>

#include "dev_types.h"
#include "kernels.h"

namespace b200tag {

// ReDistort, apriltag_detect.cu:307-331
__device__ void redistort(double *x, double *y, const FrameParams &c) {
  const double k1 = c.k1, k2 = c.k2, p1 = c.p1, p2 = c.p2, k3 = c.k3;
  const double xP = (*x - c.cx) / c.fx;
  const double yP = (*y - c.cy) / c.fy;
  const double rSq = xP * xP + yP * yP;
  const double linCoef = 1 + k1 * rSq + k2 * rSq * rSq + k3 * rSq * rSq * rSq;
  const double xPP = xP * linCoef + 2 * p1 * xP * yP + p2 * (rSq + 2 * xP * xP);
  const double yPP = yP * linCoef + p1 * (rSq + 2 * yP * yP) + 2 * p2 * xP * yP;
  *x = xPP * c.fx + c.cx;
  *y = yPP * c.fy + c.cy;
}

// GpuDetector::UnDistort, apriltag_detect.cu:335-402
__device__ bool undistort(double *u, double *v, const FrameParams &c) {
  bool converged = true;
  const double k1 = c.k1, k2 = c.k2, p1 = c.p1, p2 = c.p2, k3 = c.k3;
  const double xPP = (*u - c.cx) / c.fx;
  const double yPP = (*v - c.cy) / c.fy;
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
    if (iterations > 100) {
      converged = false;
      break;
    }
    iterations++;
  } while (fabs(xP - prev_x) > 1e-6 || fabs(yP - prev_y) > 1e-6);
  *u = xP * c.fx + c.cx;
  *v = yP * c.fy + c.cy;
  return converged;
}

__device__ __forceinline__ void h_project(const double *H, double x, double y, double *ox, double *oy) {
  const double xx = H[0] * x + H[1] * y + H[2];
  const double yy = H[3] * x + H[4] * y + H[5];
  const double zz = H[6] * x + H[7] * y + H[8];
  *ox = xx / zz;
  *oy = yy / zz;
}

// homography_compute2 (libapriltag common/homography.c): 8x9 Gaussian elimination with partial pivoting,
// run by one warp on a shared-memory matrix: lane = (row, quarter of the columns).  Every element sees
// exactly the operations of the sequential routine in the same order, so the result is bit-identical;
// only the independent row updates of one elimination step run side by side.  Returns 0 on success
// (uniform across the warp).
__device__ int homography_compute_warp(double *A /* shared, 72 */, const float p[4][2], double *Hout /* shared, 9 */, int lane) {
  if (lane < 4) {
    const int i = lane;
    const double c0 = (i == 0 || i == 3) ? -1 : 1, c1 = (i == 0 || i == 1) ? -1 : 1;
    const double c2 = p[i][0], c3 = p[i][1];
    double *r0 = &A[(2 * i) * 9], *r1 = &A[(2 * i + 1) * 9];
    r0[0] = c0; r0[1] = c1; r0[2] = 1; r0[3] = 0; r0[4] = 0; r0[5] = 0;
    r0[6] = -c0 * c2; r0[7] = -c1 * c2; r0[8] = c2;
    r1[0] = 0; r1[1] = 0; r1[2] = 0; r1[3] = c0; r1[4] = c1; r1[5] = 1;
    r1[6] = -c0 * c3; r1[7] = -c1 * c3; r1[8] = c3;
  }
  __syncwarp();
  const double epsilon = 1e-10;
  const int row = lane >> 2, sub = lane & 3;
  for (int col = 0; col < 8; col++) {
    // pivot: the first row >= col holding the largest magnitude (strict > in the sequential scan)
    const double val = (lane >= col && lane < 8) ? fabs(A[lane * 9 + col]) : -1.0;
    double mx = val;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));  // lanes 0..7 fold among themselves
    mx = __shfl_sync(0xffffffffu, mx, 0);
    if (!(mx > 0.0) || mx < epsilon) return -1;
    const int piv = __ffs(__ballot_sync(0xffffffffu, val == mx)) - 1;
    if (piv != col && lane >= col && lane < 9) {
      const double tmp = A[col * 9 + lane];
      A[col * 9 + lane] = A[piv * 9 + lane];
      A[piv * 9 + lane] = tmp;
    }
    __syncwarp();
    double f = 0;
    if (row > col) f = A[row * 9 + col] / A[col * 9 + col];
    __syncwarp();
    if (row > col) {
      if (sub == 0) A[row * 9 + col] = 0;
      for (int j = col + 1 + sub; j < 9; j += 4) A[row * 9 + j] -= f * A[col * 9 + j];
    }
    __syncwarp();
  }
  if (lane == 0) {
    for (int col = 7; col >= 0; col--) {
      double sum = 0;
      for (int i = col + 1; i < 8; i++) sum += A[col * 9 + i] * A[i * 9 + 8];
      A[col * 9 + 8] = (A[col * 9 + 8] - sum) / A[col * 9 + col];
    }
    for (int i = 0; i < 8; i++) Hout[i] = A[i * 9 + 8];
    Hout[8] = 1;
  }
  __syncwarp();
  return 0;
}

struct GrayModel {
  double A[3][3], B[3], C[3];
};
__device__ void gm_add(GrayModel *g, double x, double y, double gray) {
  g->A[0][0] += x * x; g->A[0][1] += x * y; g->A[0][2] += x;
  g->A[1][1] += y * y; g->A[1][2] += y; g->A[2][2] += 1;
  g->B[0] += x * gray; g->B[1] += y * gray; g->B[2] += gray;
}
__device__ void gm_solve(GrayModel *g) {  // mat33_sym_solve (libapriltag common/matd.c)
  const double *A = &g->A[0][0];
  double L[9], M[9];
  L[0] = sqrt(A[0]);
  L[3] = A[1] / L[0];
  L[6] = A[2] / L[0];
  L[4] = sqrt(A[4] - L[3] * L[3]);
  L[7] = (A[5] - L[3] * L[6]) / L[4];
  L[8] = sqrt(A[8] - L[6] * L[6] - L[7] * L[7]);
  M[0] = 1 / L[0];
  M[3] = -L[3] * M[0] / L[4];
  M[4] = 1 / L[4];
  M[6] = (-L[6] * M[0] - L[7] * M[3]) / L[8];
  M[7] = -L[7] * M[4] / L[8];
  M[8] = 1 / L[8];
  double t[3];
  t[0] = M[0] * g->B[0];
  t[1] = M[3] * g->B[0] + M[4] * g->B[1];
  t[2] = M[6] * g->B[0] + M[7] * g->B[1] + M[8] * g->B[2];
  g->C[0] = M[0] * t[0] + M[3] * t[1] + M[6] * t[2];
  g->C[1] = M[4] * t[1] + M[7] * t[2];
  g->C[2] = M[8] * t[2];
}
__device__ __forceinline__ double gm_interp(const GrayModel *g, double x, double y) { return g->C[0] * x + g->C[1] * y + g->C[2]; }

// value_for_pixel (libapriltag apriltag.c): bilinear sample at (px-0.5, py-0.5), -1 if out of bounds
__device__ double value_for_pixel(const uint8_t *im, int W, int H, double px, double py) {
  const int x1 = static_cast<int>(floor(px - 0.5));
  const int x2 = static_cast<int>(ceil(px - 0.5));
  const double x = px - 0.5 - x1;
  const int y1 = static_cast<int>(floor(py - 0.5));
  const int y2 = static_cast<int>(ceil(py - 0.5));
  const double y = py - 0.5 - y1;
  if (x1 < 0 || x2 >= W || y1 < 0 || y2 >= H) return -1;
  return im[static_cast<size_t>(y1) * W + x1] * (1 - x) * (1 - y) + im[static_cast<size_t>(y1) * W + x2] * x * (1 - y) +
         im[static_cast<size_t>(y2) * W + x1] * (1 - x) * y + im[static_cast<size_t>(y2) * W + x2] * x * y;
}

constexpr int kSampleChunk = 256;

struct DecodeShared {
  double sx[kSampleChunk], sy[kSampleChunk];
  uint8_t sv[kSampleChunk];
  double lines[4][4];
  float p[4][2];
  float e_nx[4], e_ny[4];  // per-edge normal and sample count (refine)
  int e_ns[4];
  double gm_x[64], gm_y[64];
  int gm_v[64];  // -1 = sample outside the image
  // (the tag's cell values and their sharpened copy live in sx / sy: the refinement samples are dead by then)
  double H[9];
  double A[72];  // homography system
  GrayModel white, black;
  uint32_t cur;
  int ok;
};
static_assert(kSampleChunk >= kMaxTotalWidth * kMaxTotalWidth, "cell values alias the sample buffers");

// quad_decode + the detection record for one family (libapriltag apriltag.c, RECALLED).  WB / TW / NB are the
// family's width_at_border / total_width / nbits as compile-time constants (tag36h11, the family the node configures:
// divisions and loop bounds fold), or 0 to take them from the family at run time.
template <int WB, int TW, int NB>
__device__ __forceinline__ void decode_family(const FrameParams &p, DecodeShared &S, const DevFamily &fam, int fi, const uint8_t *im,
                                              int W, int H, Counters *ctr, b200tag_detection *dets, int frame, int lane) {
  const int wb = WB ? WB : fam.width_at_border, tw = TW ? TW : fam.total_width, nbits = NB ? NB : static_cast<int>(fam.nbits);
  const uint64_t *codes = p.family_codes + fam.codes_off;
  double *values = S.sx, *sharp = S.sy;
  __syncwarp();

    // quad_decode: gray model from 8 border lines x width_at_border samples (width_at_border <= 8 is checked when the
    // detector is created; every libapriltag family has 5..8)
    const int per_line = wb;
    for (int j = lane; j < 64; j += 32) {
      const int pi = j >> 3, i = j & 7;
      float p0, p1, p2, p3;
      switch (pi) {
        case 0: p0 = -0.5f;     p1 = 0.5f;      p2 = 0; p3 = 1; break;
        case 1: p0 = 0.5f;      p1 = 0.5f;      p2 = 0; p3 = 1; break;
        case 2: p0 = wb + 0.5f; p1 = .5f;       p2 = 0; p3 = 1; break;
        case 3: p0 = wb - 0.5f; p1 = .5f;       p2 = 0; p3 = 1; break;
        case 4: p0 = 0.5f;      p1 = -0.5f;     p2 = 1; p3 = 0; break;
        case 5: p0 = 0.5f;      p1 = 0.5f;      p2 = 1; p3 = 0; break;
        case 6: p0 = 0.5f;      p1 = wb + 0.5f; p2 = 1; p3 = 0; break;
        default: p0 = 0.5f;     p1 = wb - 0.5f; p2 = 1; p3 = 0; break;
      }
      const double tagx01 = (p0 + i * p2) / (wb);
      const double tagy01 = (p1 + i * p3) / (wb);
      const double tagx = 2 * (tagx01 - 0.5);
      const double tagy = 2 * (tagy01 - 0.5);
      double px, py;
      h_project(S.H, tagx, tagy, &px, &py);
      const int ix = static_cast<int>(px), iy = static_cast<int>(py);
      int v = -1;
      if (i < per_line && !(ix < 0 || iy < 0 || ix >= W || iy >= H)) v = im[static_cast<size_t>(iy) * W + ix];
      S.gm_x[j] = tagx;
      S.gm_y[j] = tagy;
      S.gm_v[j] = v;
    }
    for (int j = lane; j < tw * tw; j += 32) values[j] = 0.0;
    __syncwarp();
    if (lane < 2) {  // lane 0 fits the white model, lane 1 the black one (each sums its samples in order)
      GrayModel m;
      for (int i = 0; i < 3; i++) {
        for (int j = 0; j < 3; j++) m.A[i][j] = 0;
        m.B[i] = m.C[i] = 0;
      }
      for (int jj = 0; jj < 32; jj++) {  // patterns alternate white, black: this lane's are 0, 2, 4, 6 or 1, 3, 5, 7
        const int j = (((jj >> 3) << 1) | lane) * 8 + (jj & 7);
        if (S.gm_v[j] < 0) continue;
        gm_add(&m, S.gm_x[j], S.gm_y[j], S.gm_v[j]);
      }
      gm_solve(&m);
      if (lane == 0) S.white = m; else S.black = m;
    }
    __syncwarp();
    if (lane == 0) {
      const int reversed_border = fam.reversed_border != 0;
      S.ok = !((gm_interp(&S.white, 0, 0) - gm_interp(&S.black, 0, 0) < 0) != reversed_border);
    }
    __syncwarp();
    if (!S.ok) return;

    const int min_coord = (wb - tw) / 2;
    for (int i = lane; i < nbits; i += 32) {
      const int bit_x = fam.bit_x[i], bit_y = fam.bit_y[i];
      const double tagx01 = (bit_x + 0.5) / (wb);
      const double tagy01 = (bit_y + 0.5) / (wb);
      const double tagx = 2 * (tagx01 - 0.5);
      const double tagy = 2 * (tagy01 - 0.5);
      double px, py;
      h_project(S.H, tagx, tagy, &px, &py);
      const double v = value_for_pixel(im, W, H, px, py);
      if (v == -1) continue;
      const double thresh = (gm_interp(&S.black, tagx, tagy) + gm_interp(&S.white, tagx, tagy)) / 2.0;
      values[tw * (bit_y - min_coord) + bit_x - min_coord] = v - thresh;
    }
    __syncwarp();
    for (int c = lane; c < tw * tw; c += 32) {  // sharpen()
      const int y = c / tw, x = c % tw;
      const double kernel[9] = {0, -1, 0, -1, 4, -1, 0, -1, 0};
      double acc = 0;
      for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
          if ((y + i - 1) < 0 || (y + i - 1) > tw - 1 || (x + j - 1) < 0 || (x + j - 1) > tw - 1) continue;
          acc += values[(y + i - 1) * tw + (x + j - 1)] * kernel[i * 3 + j];
        }
      sharp[c] = acc;
    }
    __syncwarp();
    for (int c = lane; c < tw * tw; c += 32) values[c] = values[c] + p.decode_sharpening * sharp[c];
    __syncwarp();

    // bits and decision margin, folded in bit order by every lane redundantly (nbits steps)
    float black_score = 0, white_score = 0;
    float black_score_count = 1, white_score_count = 1;
    uint64_t rcode = 0;
    for (int i = 0; i < nbits; i++) {
      const int bit_x = fam.bit_x[i], bit_y = fam.bit_y[i];
      rcode = (rcode << 1);
      const double v = values[(bit_y - min_coord) * tw + bit_x - min_coord];
      if (v > 0) {
        white_score += static_cast<float>(v);
        white_score_count++;
        rcode |= 1;
      } else {
        black_score -= static_cast<float>(v);
        black_score_count++;
      }
    }
    // quick_decode_codeword: lane-parallel popcount scan over the family's codes, first rotation that hits
    // (the hash table of libapriltag holds every code with <= max_hamming flipped bits; with the families' minimum
    // distances the hit is unique, so the smallest id within reach is the same answer)
    int id = -1, hamming = 255, rotation = 0;
    const int ncodes = static_cast<int>(fam.ncodes), maxh = fam.max_hamming;
    for (int ridx = 0; ridx < 4 && id < 0; ridx++) {
      int found = 0x7fffffff, fh = 255;
      for (int c = lane; c < ncodes; c += 32) {
        const int d = __popcll(rcode ^ __ldg(codes + c));
        if (d <= maxh && c < found) { found = c; fh = d; }
      }
      const int best = __reduce_min_sync(0xffffffffu, found);
      if (best != 0x7fffffff) {
        const uint32_t who = __ballot_sync(0xffffffffu, found == best);
        hamming = __shfl_sync(0xffffffffu, fh, __ffs(who) - 1);
        id = best;
        rotation = ridx;
      } else {  // rotate90 (libapriltag apriltag.c)
        int pp = nbits;
        uint64_t l = 0;
        if (nbits % 4 == 1) { pp = nbits - 1; l = 1; }
        rcode = ((rcode >> l) << (pp / 4 + l)) | (rcode >> (3 * pp / 4 + l) << l) | (rcode & l);
        rcode &= nbits >= 64 ? ~0ull : ((1ull << nbits) - 1);
      }
    }
    const float margin = fminf(white_score / white_score_count, black_score / black_score_count);
    if (lane == 0 && margin >= 0 && hamming < 255) {
      const uint32_t di = atomicAdd(&ctr->num_detections, 1u);
      if (di < p.det_cap) {
        b200tag_detection &d = dets[di];
        d.id = id;
        d.hamming = hamming;
        d.decision_margin = margin;
        d.frame = frame;
        d.family = fi;
        d.reserved = 0;
        // cos/sin(rotation * M_PI / 2.0) as the host libm returns them
        const double kc[4] = {1.0, 6.123233995736766e-17, -1.0, -1.8369701987210297e-16};
        const double ks[4] = {0.0, 1.0, 1.2246467991473532e-16, -1.0};
        const double cc = kc[rotation], ss = ks[rotation];
        for (int row = 0; row < 3; row++) {
          d.H[row * 3 + 0] = S.H[row * 3 + 0] * cc + S.H[row * 3 + 1] * ss;
          d.H[row * 3 + 1] = S.H[row * 3 + 0] * -ss + S.H[row * 3 + 1] * cc;
          d.H[row * 3 + 2] = S.H[row * 3 + 2];
        }
        h_project(d.H, 0, 0, &d.c[0], &d.c[1]);
        for (int i = 0; i < 4; i++) {
          const int tcx = (i == 1 || i == 2) ? 1 : -1;
          const int tcy = (i < 2) ? 1 : -1;
          h_project(d.H, tcx, tcy, &d.p[i][0], &d.p[i][1]);
        }
      } else {
        atomicOr(&ctr->status, B200TAG_ST_DETS_OVERFLOW);
      }
    }
}

// WARPS warps per candidate quad.  One warp (batches: quads outnumber the warps an SM can hold, so per-quad latency is
// hidden) or four (one or a few frames at a time: a frame has about a hundred quads for 148 SMs, so the time of this
// kernel is the time of ONE quad): the refinement samples -- the bulk of the work, independent of each other -- are
// spread over all threads; the ordered sums, the homography and the decode proper stay on the first warp, exactly as
// in the one-warp kernel, so the results are the same bit for bit.
template <int WARPS>
__global__ void __launch_bounds__(32 * WARPS) k_decode(FrameParams p) {
  __shared__ DecodeShared S;
  constexpr int NT = 32 * WARPS;
  auto csync = [] {
    if constexpr (WARPS == 1) __syncwarp();
    else __syncthreads();
  };
  const int frame = blockIdx.y;
  const int tid = threadIdx.x;
  const int lane = tid;  // (the first warp's lane index wherever "lane < k" picks workers below)
  const bool first_warp = tid < 32;
  Counters *ctr = p.counters + frame;
  const uint8_t *im = p.gray + frame * p.gray_stride;
  const b200tag_quad *quads = p.quads + static_cast<size_t>(frame) * p.quad_cap;
  b200tag_detection *dets = p.dets + static_cast<size_t>(frame) * p.det_cap;
  const uint32_t nquads = min(ctr->num_quads, p.quad_cap);
  const int W = p.W, H = p.H;
  uint32_t nxt = 0;
  if (tid == 0) nxt = atomicAdd(&ctr->next_quad, 1u);
  while (true) {
    csync();
    if (tid == 0) S.cur = nxt;
    csync();
    const uint32_t qi = S.cur;
    if (qi >= nquads) break;
    if (tid == 0) nxt = atomicAdd(&ctr->next_quad, 1u);  // the next item's round trip overlaps this quad
    const b200tag_quad quad = quads[qi];
    if (tid < 8) S.p[tid >> 1][tid & 1] = quad.corners[tid >> 1][tid & 1];
    csync();

    if (p.refine_edges) {  // RefineEdges, apriltag_detect.cu:405-564
      // The four edges only read the unrefined corners, so they are refined side by side: lanes 0..3 own one edge
      // each (normal, sample count, moment sums in the reference's sample order, line fit, corner), and the
      // samples of all four edges are spread over the whole warp.
      if (lane < 4) {
        const int a = lane, b = (lane + 1) & 3;
        float nx = S.p[b][1] - S.p[a][1];
        float ny = -S.p[b][0] + S.p[a][0];
        const float mag = sqrtf(nx * nx + ny * ny);
        nx /= mag;
        ny /= mag;
        if (quad.reversed_border) { nx = -nx; ny = -ny; }
        int nsamples = static_cast<int>(mag / 8);
        if (nsamples < 16) nsamples = 16;
        S.e_nx[lane] = nx;
        S.e_ny[lane] = ny;
        S.e_ns[lane] = nsamples;
      }
      csync();
      const int ns0 = S.e_ns[0], ns1 = S.e_ns[1], ns2 = S.e_ns[2], ns3 = S.e_ns[3];
      const int off1 = ns0, off2 = ns0 + ns1, off3 = ns0 + ns1 + ns2, total = off3 + ns3;
      double Mx = 0, My = 0, Mxx = 0, Mxy = 0, Myy = 0, N = 0;  // lanes 0..3: sums of their edge
      const int my_lo = lane == 0 ? 0 : (lane == 1 ? off1 : (lane == 2 ? off2 : off3));
      const int my_hi = lane == 0 ? off1 : (lane == 1 ? off2 : (lane == 2 ? off3 : total));
      for (int base = 0; base < total; base += kSampleChunk) {
        const int lim = min(kSampleChunk, total - base);
        for (int j = tid; j < lim; j += NT) {
          const int g = base + j;
          const int edge = (g >= off1) + (g >= off2) + (g >= off3);
          const int s = g - (edge == 0 ? 0 : (edge == 1 ? off1 : (edge == 2 ? off2 : off3)));
          const int nsamples = S.e_ns[edge];
          const int a = edge, b = (edge + 1) & 3;
          const float nx = S.e_nx[edge], ny = S.e_ny[edge];
          const float pax = S.p[a][0], pay = S.p[a][1], pbx = S.p[b][0], pby = S.p[b][1];
          const double alpha = (1.0 + s) / (nsamples + 1);
          const double x0 = alpha * pax + (1 - alpha) * pbx;
          const double y0 = alpha * pay + (1 - alpha) * pby;
          double Mn = 0, Mcount = 0;
          const double range = static_cast<double>(static_cast<float>(p.f)) + 1;
          // n runs over -range, -range + 0.25, ..., range (multiples of 0.25: exact in double).  The two
          // byte gathers of five consecutive n are issued together; the sums keep the order of n.
          const int nt = static_cast<int>(8 * range) + 1;
          for (int t0 = 0; t0 < nt; t0 += 5) {
            int g1v[5], g2v[5];
            double nv[5];
            bool okv[5];
#pragma unroll
            for (int k = 0; k < 5; k++) {
              const double n = -range + 0.25 * (t0 + k);
              const double grange = 1;
              const int x1 = static_cast<int>(x0 + (n + grange) * nx);
              const int y1 = static_cast<int>(y0 + (n + grange) * ny);
              const int x2 = static_cast<int>(x0 + (n - grange) * nx);
              const int y2 = static_cast<int>(y0 + (n - grange) * ny);
              const bool ok = (t0 + k < nt) && !(x1 < 0 || x1 >= W || y1 < 0 || y1 >= H) && !(x2 < 0 || x2 >= W || y2 < 0 || y2 >= H);
              nv[k] = n;
              okv[k] = ok;
              g1v[k] = ok ? im[static_cast<size_t>(y1) * W + x1] : 0;
              g2v[k] = ok ? im[static_cast<size_t>(y2) * W + x2] : 0;
            }
#pragma unroll
            for (int k = 0; k < 5; k++) {
              if (!okv[k] || g1v[k] < g2v[k]) continue;
              const double weight = static_cast<double>((g2v[k] - g1v[k]) * (g2v[k] - g1v[k]));
              Mn += weight * nv[k];
              Mcount += weight;
            }
          }
          uint8_t valid = 0;
          double bestx = 0, besty = 0;
          if (Mcount != 0) {
            const double n0 = Mn / Mcount;
            bestx = x0 + n0 * nx;
            besty = y0 + n0 * ny;
            undistort(&bestx, &besty, p);
            valid = 1;
          }
          S.sx[j] = bestx;
          S.sy[j] = besty;
          S.sv[j] = valid;
        }
        csync();
        if (lane < 4) {  // this chunk's samples of my edge, in sample order
          const int lo = max(base, my_lo) - base, hi = min(base + lim, my_hi) - base;
          for (int j = lo; j < hi; j++) {
            if (!S.sv[j]) continue;
            const double bx = S.sx[j], by = S.sy[j];
            Mx += bx; My += by; Mxx += bx * bx; Mxy += bx * by; Myy += by * by; N++;
          }
        }
        csync();
      }
      if (lane < 4) {
        const double Ex = Mx / N, Ey = My / N;
        const double Cxx = Mxx / N - Ex * Ex;
        const double Cxy = Mxy / N - Ex * Ey;
        const double Cyy = Myy / N - Ey * Ey;
        const double normal_theta = .5 * atan2f(static_cast<float>(-2 * Cxy), static_cast<float>(Cyy - Cxx));
        S.lines[lane][0] = Ex;
        S.lines[lane][1] = Ey;
        S.lines[lane][2] = cosf(static_cast<float>(normal_theta));
        S.lines[lane][3] = sinf(static_cast<float>(normal_theta));
      }
      __syncwarp();
      if (lane < 4) {
        const int i = lane;
        const double A00 = S.lines[i][3], A01 = -S.lines[(i + 1) & 3][3];
        const double A10 = -S.lines[i][2], A11 = S.lines[(i + 1) & 3][2];
        const double B0 = -S.lines[i][0] + S.lines[(i + 1) & 3][0];
        const double B1 = -S.lines[i][1] + S.lines[(i + 1) & 3][1];
        const double det = A00 * A11 - A10 * A01;
        if (fabs(det) > 0.001) {
          const double W00 = A11 / det, W01 = -A01 / det;
          const double L0 = W00 * B0 + W01 * B1;
          double px = S.lines[i][0] + L0 * A00;
          double py = S.lines[i][1] + L0 * A10;
          redistort(&px, &py, p);
          S.p[(i + 1) & 3][0] = static_cast<float>(px);
          S.p[(i + 1) & 3][1] = static_cast<float>(py);
        }
      }
      __syncwarp();
    }

    // the rest -- homography, gray model, bit samples, code scan, detection record -- is the first warp's
    if (first_warp) {
      // quad_update_homographies
      {
        int ok = homography_compute_warp(S.A, S.p, S.H, lane) == 0;
        if (ok) {
          const double *Hm = S.H;
          const double det = Hm[0] * (Hm[4] * Hm[8] - Hm[5] * Hm[7]) - Hm[1] * (Hm[3] * Hm[8] - Hm[5] * Hm[6]) +
                             Hm[2] * (Hm[3] * Hm[7] - Hm[4] * Hm[6]);
          if (!(fabs(det) > 1e-300)) ok = 0;
        }
        __syncwarp();
        if (lane == 0) S.ok = ok;
      }
      __syncwarp();
      if (S.ok) {
        // quad_decode_task: every family of the quad's border polarity gets its own decode of the same homography
        for (int fi = 0; fi < p.nfamilies; fi++) {
          const DevFamily &fam = p.families[fi];
          if ((fam.reversed_border != 0) != (quad.reversed_border != 0)) continue;
          if (fam.width_at_border == 8 && fam.total_width == 10 && fam.nbits == 36)
            decode_family<8, 10, 36>(p, S, fam, fi, im, W, H, ctr, dets, frame, lane);
          else
            decode_family<0, 0, 0>(p, S, fam, fi, im, W, H, ctr, dets, frame, lane);
        }
      }
    }
  }
}

void launch_decode(const FrameParams &p, int frames, Launcher &ln) {
  // batches: one warp per CTA, about 2400 CTAs in total (a frame has ~100 candidate quads); up to four frames: four
  // warps per quad, all 148 SMs
  const unsigned per_frame = static_cast<unsigned>(frames) >= 16 ? (2368u + frames - 1) / frames : 148u;
  ln.timed("decode", [&] {
    if (frames <= 4) k_decode<4><<<dim3(148u, frames), 128, 0, ln.s>>>(p);
    else k_decode<1><<<dim3(per_frame < 8u ? 8u : per_frame, frames), 32, 0, ln.s>>>(p);
  });
}

}  // namespace b200tag
