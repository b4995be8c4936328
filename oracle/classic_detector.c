/*
 * TEST INFRASTRUCTURE -- CPU restatement of the classic AprilTag 3 detector (libapriltag
 * apriltag_detector_detect), the reference's SECOND detection path: it is what
 * src/apriltags_cuda/test/gpu_detector_test.cu:104-157 runs next to GpuDetector (CpuDetectsAprilTag,
 * CpuNoAprilTagDetections, CpuAndGpuEqual: same id, centre and corners within 0.5 px) and what
 * opencv_cuda_demo.cu:117 falls back to.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may load it; the product never links it.
 *
 * PARITY UNPINNED at the source level: the detector lives in the un-vendored, 971-modified fork
 * github.com/cgpadwick/apriltag tag 3.3.0 (src/external/CMakeLists.txt:85-95); what follows restates the
 * published AprilTag 3 algorithm (apriltag.c, apriltag_quad_thresh.c) stage by stage -- SURVEY.md App. A.8 --
 * in double precision as upstream does.  It is pinned by the reference test's own known answers (one detection
 * on colorimage.jpg, none on colorimage_notags.jpg), by agreement with the GPU-semantics oracle within the
 * reference's own CPU-vs-GPU tolerance (0.5 px), and by cv2.aruco's AprilTag refinement as a third opinion.
 *
 * Differences from the GPU arithmetic (apriltag_oracle.c), all upstream's: union-find over image rows with the
 * x in [1, w-2] scan; gradient clusters with the connected_last de-duplication and a later removal of
 * consecutive duplicates; points ordered by a quadrant + slope key instead of atan2f; line-fit moments in
 * double with W = sqrt(gx^2 + gy^2) + 1 (not truncated) at coordinates p/2 + 0.5; refine_edges without camera
 * un/re-distortion.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "oracle_internal.h"

/* ---- unionfind.h ---------------------------------------------------------------------------------------- */
typedef struct {
  uint32_t *parent, *size;
} unionfind;

static uint32_t uf_rep(unionfind *uf, uint32_t id) {
  uint32_t root = id;
  while (uf->parent[root] != root) root = uf->parent[root];
  while (uf->parent[id] != root) { /* path compression */
    const uint32_t next = uf->parent[id];
    uf->parent[id] = root;
    id = next;
  }
  return root;
}
static uint32_t uf_size(unionfind *uf, uint32_t id) { return uf->size[uf_rep(uf, id)] + 1; }
static void uf_connect(unionfind *uf, uint32_t a, uint32_t b) {
  const uint32_t ar = uf_rep(uf, a), br = uf_rep(uf, b);
  if (ar == br) return;
  const uint32_t asz = uf->size[ar] + 1, bsz = uf->size[br] + 1;
  if (asz > bsz) {
    uf->parent[br] = ar;
    uf->size[ar] += bsz;
  } else {
    uf->parent[ar] = br;
    uf->size[br] += asz;
  }
}

/* connected_components / do_unionfind_first_line / do_unionfind_line2 (apriltag_quad_thresh.c) */
static void connected_components(unionfind *uf, const uint8_t *im, int w, int h) {
#define DO_UNIONFIND2(dx, dy) \
  if (im[(y + (dy)) * w + x + (dx)] == v) uf_connect(uf, (uint32_t)(y * w + x), (uint32_t)((y + (dy)) * w + x + (dx)));
  {
    const int y = 0;
    for (int x = 1; x < w - 1; x++) {
      const uint8_t v = im[y * w + x];
      if (v == 127) continue;
      DO_UNIONFIND2(-1, 0);
    }
  }
  for (int y = 1; y < h; y++) {
    uint8_t v_m1_m1, v_0_m1 = im[(y - 1) * w + 0], v_1_m1 = im[(y - 1) * w + 1], v_m1_0, v = im[y * w + 0];
    for (int x = 1; x < w - 1; x++) {
      v_m1_m1 = v_0_m1;
      v_0_m1 = v_1_m1;
      v_1_m1 = im[(y - 1) * w + x + 1];
      v_m1_0 = v;
      v = im[y * w + x];
      if (v == 127) continue;
      DO_UNIONFIND2(-1, 0);
      if (x == 1 || !((v_m1_0 == v_m1_m1) && (v_m1_m1 == v_0_m1))) {
        DO_UNIONFIND2(0, -1);
      }
      if (v == 255) {
        if (x == 1 || !(v_m1_0 == v_m1_m1 || v_0_m1 == v_m1_m1)) {
          DO_UNIONFIND2(-1, -1);
        }
        if (!(v_0_m1 == v_1_m1)) {
          DO_UNIONFIND2(1, -1);
        }
      }
    }
  }
#undef DO_UNIONFIND2
}

/* ---- gradient clusters ------------------------------------------------------------------------------------ */
struct pt {
  uint16_t x, y; /* half-pixel coordinates */
  int16_t gx, gy;
  float slope;
};
typedef struct {
  uint64_t id;
  struct pt *pts;
  int n, cap;
} cluster;
typedef struct {
  cluster *items;
  int n, cap;
  int *bucket;   /* head index per hash bucket, -1 = empty */
  int *next;     /* chain */
  int nbuckets;
} cluster_map;

static uint32_t u64hash_2(uint64_t x) { return (uint32_t)((2654435761ULL * x) >> 32); }

static cluster *cluster_get(cluster_map *m, uint64_t id) {
  const uint32_t b = u64hash_2(id) % (uint32_t)m->nbuckets;
  for (int e = m->bucket[b]; e >= 0; e = m->next[e])
    if (m->items[e].id == id) return &m->items[e];
  if (m->n == m->cap) {
    m->cap = m->cap ? 2 * m->cap : 1024;
    m->items = (cluster *)realloc(m->items, (size_t)m->cap * sizeof(cluster));
    m->next = (int *)realloc(m->next, (size_t)m->cap * sizeof(int));
  }
  cluster *c = &m->items[m->n];
  c->id = id;
  c->pts = NULL;
  c->n = c->cap = 0;
  m->next[m->n] = m->bucket[b];
  m->bucket[b] = m->n;
  m->n++;
  return c;
}
static void cluster_add(cluster *c, struct pt p) {
  if (c->n == c->cap) {
    c->cap = c->cap ? 2 * c->cap : 32;
    c->pts = (struct pt *)realloc(c->pts, (size_t)c->cap * sizeof(struct pt));
  }
  c->pts[c->n++] = p;
}

/* do_gradient_clusters (apriltag_quad_thresh.c): y in [1, h-2], x in [1, w-2] */
static void gradient_clusters(cluster_map *m, unionfind *uf, const uint8_t *im, int w, int h) {
  for (int y = 1; y < h - 1; y++) {
    int connected_last = 0;
    for (int x = 1; x < w - 1; x++) {
      const int v0 = im[y * w + x];
      if (v0 == 127) {
        connected_last = 0;
        continue;
      }
      const uint64_t rep0 = uf_rep(uf, (uint32_t)(y * w + x));
      if (uf_size(uf, (uint32_t)rep0) < 25) {
        connected_last = 0;
        continue;
      }
      int connected;
#define DO_CONN(dx, dy)                                                                                         \
  {                                                                                                             \
    const int v1 = im[(y + (dy)) * w + x + (dx)];                                                               \
    if (v0 + v1 == 255) {                                                                                       \
      const uint64_t rep1 = uf_rep(uf, (uint32_t)((y + (dy)) * w + x + (dx)));                                  \
      if (uf_size(uf, (uint32_t)rep1) > 24) {                                                                   \
        const uint64_t clusterid = rep0 < rep1 ? (rep1 << 32) + rep0 : (rep0 << 32) + rep1;                     \
        const struct pt p = {(uint16_t)(2 * x + (dx)), (uint16_t)(2 * y + (dy)), (int16_t)((dx) * (v1 - v0)),   \
                             (int16_t)((dy) * (v1 - v0)), 0.0f};                                                \
        cluster_add(cluster_get(m, clusterid), p);                                                              \
        connected = 1;                                                                                          \
      }                                                                                                         \
    }                                                                                                           \
  }
      DO_CONN(1, 0);
      DO_CONN(0, 1);
      if (!connected_last) {
        /* checking (1, 1) at the previous x and (-1, 1) here yields the same point twice */
        DO_CONN(-1, 1);
      }
      connected = 0;
      DO_CONN(1, 1);
      connected_last = connected;
#undef DO_CONN
    }
  }
}

/* ---- fit_quad ----------------------------------------------------------------------------------------------- */
/* ptsort: merge sort on the slope key; equal keys take the second run's element first, as upstream's MERGE does */
static void ptsort(struct pt *pts, int sz) {
  if (sz <= 1) return;
  if (sz == 2) {
    if (pts[0].slope - pts[1].slope > 0) {
      const struct pt t = pts[0];
      pts[0] = pts[1];
      pts[1] = t;
    }
    return;
  }
  struct pt *tmp = (struct pt *)malloc((size_t)sz * sizeof(struct pt));
  memcpy(tmp, pts, (size_t)sz * sizeof(struct pt));
  const int asz = sz / 2, bsz = sz - asz;
  struct pt *as = tmp, *bs = tmp + asz;
  ptsort(as, asz);
  ptsort(bs, bsz);
  int apos = 0, bpos = 0, out = 0;
  while (apos < asz && bpos < bsz) {
    if (as[apos].slope - bs[bpos].slope < 0) pts[out++] = as[apos++];
    else pts[out++] = bs[bpos++];
  }
  if (apos < asz) memcpy(&pts[out], &as[apos], (size_t)(asz - apos) * sizeof(struct pt));
  if (bpos < bsz) memcpy(&pts[out], &bs[bpos], (size_t)(bsz - bpos) * sizeof(struct pt));
  free(tmp);
}

struct line_fit_pt {
  double Mx, My, Mxx, Mxy, Myy, W;
};

/* compute_lfps: gradient-weighted prefix moments in double, coordinates p/2 + 0.5 */
static struct line_fit_pt *compute_lfps(int sz, const struct pt *pts, const uint8_t *im, int w, int h) {
  struct line_fit_pt *lfps = (struct line_fit_pt *)calloc((size_t)sz, sizeof(struct line_fit_pt));
  for (int i = 0; i < sz; i++) {
    const struct pt *p = &pts[i];
    if (i > 0) lfps[i] = lfps[i - 1];
    const double delta = 0.5;
    const double x = p->x * .5 + delta, y = p->y * .5 + delta;
    const int ix = (int)x, iy = (int)y;
    double W = 1;
    if (ix > 0 && ix + 1 < w && iy > 0 && iy + 1 < h) {
      const int grad_x = im[iy * w + ix + 1] - im[iy * w + ix - 1];
      const int grad_y = im[(iy + 1) * w + ix] - im[(iy - 1) * w + ix];
      W = sqrt((double)(grad_x * grad_x + grad_y * grad_y)) + 1;
    }
    const double fx = x, fy = y;
    lfps[i].Mx += W * fx;
    lfps[i].My += W * fy;
    lfps[i].Mxx += W * fx * fx;
    lfps[i].Mxy += W * fx * fy;
    lfps[i].Myy += W * fy * fy;
    lfps[i].W += W;
  }
  return lfps;
}

/* fit_line: covariance of the points [i0, i1] (cyclic), normal = eigenvector of the larger eigenvalue's complement */
static void fit_line(const struct line_fit_pt *lfps, int sz, int i0, int i1, double *lineparm, double *err, double *mse) {
  double Mx, My, Mxx, Myy, Mxy, W;
  int N;
  if (i0 < i1) {
    N = i1 - i0 + 1;
    Mx = lfps[i1].Mx; My = lfps[i1].My; Mxx = lfps[i1].Mxx; Mxy = lfps[i1].Mxy; Myy = lfps[i1].Myy; W = lfps[i1].W;
    if (i0 > 0) {
      Mx -= lfps[i0 - 1].Mx; My -= lfps[i0 - 1].My; Mxx -= lfps[i0 - 1].Mxx;
      Mxy -= lfps[i0 - 1].Mxy; Myy -= lfps[i0 - 1].Myy; W -= lfps[i0 - 1].W;
    }
  } else {
    Mx = lfps[sz - 1].Mx - lfps[i0 - 1].Mx; My = lfps[sz - 1].My - lfps[i0 - 1].My;
    Mxx = lfps[sz - 1].Mxx - lfps[i0 - 1].Mxx; Mxy = lfps[sz - 1].Mxy - lfps[i0 - 1].Mxy;
    Myy = lfps[sz - 1].Myy - lfps[i0 - 1].Myy; W = lfps[sz - 1].W - lfps[i0 - 1].W;
    Mx += lfps[i1].Mx; My += lfps[i1].My; Mxx += lfps[i1].Mxx; Mxy += lfps[i1].Mxy; Myy += lfps[i1].Myy; W += lfps[i1].W;
    N = sz - i0 + i1 + 1;
  }
  const double Ex = Mx / W, Ey = My / W;
  const double Cxx = Mxx / W - Ex * Ex, Cxy = Mxy / W - Ex * Ey, Cyy = Myy / W - Ey * Ey;
  const double eig_small = 0.5 * (Cxx + Cyy - sqrtf((float)((Cxx - Cyy) * (Cxx - Cyy) + 4 * Cxy * Cxy)));
  if (lineparm) {
    lineparm[0] = Ex;
    lineparm[1] = Ey;
    const double eig = 0.5 * (Cxx + Cyy + sqrtf((float)((Cxx - Cyy) * (Cxx - Cyy) + 4 * Cxy * Cxy)));
    const double nx1 = Cxx - eig, ny1 = Cxy, M1 = nx1 * nx1 + ny1 * ny1;
    const double nx2 = Cxy, ny2 = Cyy - eig, M2 = nx2 * nx2 + ny2 * ny2;
    double nx, ny, M;
    if (M1 > M2) { nx = nx1; ny = ny1; M = M1; } else { nx = nx2; ny = ny2; M = M2; }
    const double length = sqrtf((float)M);
    if (fabs(length) < 1e-12) {
      lineparm[2] = lineparm[3] = 0;
    } else {
      lineparm[2] = nx / length;
      lineparm[3] = ny / length;
    }
  }
  if (err) *err = N * eig_small;
  if (mse) *mse = eig_small;
}

static int err_compare_descending(const void *a_, const void *b_) {
  const double a = *(const double *)a_, b = *(const double *)b_;
  return (a < b) ? 1 : ((a == b) ? 0 : -1);
}

/* quad_segment_maxima: corner candidates = local maxima of the smoothed windowed line-fit error, then the best of the
 * C(<=10, 4) ordered choices */
static int quad_segment_maxima(const orc_config *c, int sz, const struct line_fit_pt *lfps, int indices[4]) {
  int ksz = sz / 12;
  if (ksz > 20) ksz = 20;
  if (ksz < 2) return 0;
  double *errs = (double *)malloc(sizeof(double) * (size_t)sz);
  for (int i = 0; i < sz; i++) fit_line(lfps, sz, (i + sz - ksz) % sz, (i + ksz) % sz, NULL, &errs[i], NULL);
  {
    double *y = (double *)malloc(sizeof(double) * (size_t)sz);
    const double sigma = 1, cutoff = 0.05;
    int fsz = (int)(sqrt(-log(cutoff) * 2 * sigma * sigma) + 1);
    fsz = 2 * fsz + 1;
    float f[32];
    for (int i = 0; i < fsz; i++) {
      const int j = i - fsz / 2;
      f[i] = (float)exp(-j * j / (2 * sigma * sigma));
    }
    for (int iy = 0; iy < sz; iy++) {
      double acc = 0;
      for (int i = 0; i < fsz; i++) acc += errs[(iy + i - fsz / 2 + sz) % sz] * f[i];
      y[iy] = acc;
    }
    memcpy(errs, y, sizeof(double) * (size_t)sz);
    free(y);
  }
  int *maxima = (int *)malloc(sizeof(int) * (size_t)sz);
  double *maxima_errs = (double *)malloc(sizeof(double) * (size_t)sz);
  int nmaxima = 0;
  for (int i = 0; i < sz; i++) {
    if (errs[i] > errs[(i + 1) % sz] && errs[i] > errs[(i + sz - 1) % sz]) {
      maxima[nmaxima] = i;
      maxima_errs[nmaxima] = errs[i];
      nmaxima++;
    }
  }
  free(errs);
  if (nmaxima < 4) {
    free(maxima);
    free(maxima_errs);
    return 0;
  }
  const int max_nmaxima = c->max_nmaxima;
  if (nmaxima > max_nmaxima) {
    double *copy = (double *)malloc(sizeof(double) * (size_t)nmaxima);
    memcpy(copy, maxima_errs, sizeof(double) * (size_t)nmaxima);
    qsort(copy, (size_t)nmaxima, sizeof(double), err_compare_descending);
    const double maxima_thresh = copy[max_nmaxima];
    int out = 0;
    for (int in = 0; in < nmaxima; in++) {
      if (maxima_errs[in] <= maxima_thresh) continue;
      maxima[out++] = maxima[in];
    }
    nmaxima = out;
    free(copy);
  }
  free(maxima_errs);
  int best_indices[4] = {0, 0, 0, 0};
  double best_error = HUGE_VALF;
  double err01, err12, err23, err30, mse01, mse12, mse23, mse30;
  double params01[4], params12[4];
  const double max_dot = c->cos_critical_rad;
  for (int m0 = 0; m0 < nmaxima - 3; m0++) {
    const int i0 = maxima[m0];
    for (int m1 = m0 + 1; m1 < nmaxima - 2; m1++) {
      const int i1 = maxima[m1];
      fit_line(lfps, sz, i0, i1, params01, &err01, &mse01);
      if (mse01 > c->max_line_fit_mse) continue;
      for (int m2 = m1 + 1; m2 < nmaxima - 1; m2++) {
        const int i2 = maxima[m2];
        fit_line(lfps, sz, i1, i2, params12, &err12, &mse12);
        if (mse12 > c->max_line_fit_mse) continue;
        const double dot = params01[2] * params12[2] + params01[3] * params12[3];
        if (fabs(dot) > max_dot) continue;
        for (int m3 = m2 + 1; m3 < nmaxima; m3++) {
          const int i3 = maxima[m3];
          fit_line(lfps, sz, i2, i3, NULL, &err23, &mse23);
          if (mse23 > c->max_line_fit_mse) continue;
          fit_line(lfps, sz, i3, i0, NULL, &err30, &mse30);
          if (mse30 > c->max_line_fit_mse) continue;
          const double err = err01 + err12 + err23 + err30;
          if (err < best_error) {
            best_error = err;
            best_indices[0] = i0; best_indices[1] = i1; best_indices[2] = i2; best_indices[3] = i3;
          }
        }
      }
    }
  }
  free(maxima);
  if (best_error == HUGE_VALF) return 0;
  for (int i = 0; i < 4; i++) indices[i] = best_indices[i];
  return best_error / sz < c->max_line_fit_mse;
}

struct quad {
  float p[4][2];
  int reversed_border;
};

static double sq(double v) { return v * v; }

static int fit_quad(const orc_config *c, const uint8_t *im, int w, int h, cluster *cl, struct quad *quad, int tag_width,
                    int normal_border, int reversed_border) {
  int res = 0;
  int sz = cl->n;
  if (sz < 24) return 0;
  struct pt *pts = cl->pts;
  uint16_t xmax = pts[0].x, xmin = pts[0].x, ymax = pts[0].y, ymin = pts[0].y;
  for (int i = 1; i < sz; i++) {
    if (pts[i].x > xmax) xmax = pts[i].x; else if (pts[i].x < xmin) xmin = pts[i].x;
    if (pts[i].y > ymax) ymax = pts[i].y; else if (pts[i].y < ymin) ymin = pts[i].y;
  }
  if ((xmax - xmin) * (ymax - ymin) < tag_width) return 0;
  const float cx = (float)((xmin + xmax) * 0.5 + 0.05118);
  const float cy = (float)((ymin + ymax) * 0.5 + -0.028581);
  float dot = 0;
  const float quadrants[2][2] = {{-1 * (2 << 15), 0}, {2 * (2 << 15), 2 << 15}};
  for (int i = 0; i < sz; i++) {
    struct pt *p = &pts[i];
    float dx = p->x - cx, dy = p->y - cy;
    dot += dx * p->gx + dy * p->gy;
    const float quadrant = quadrants[dy > 0][dx > 0];
    if (dy < 0) {
      dy = -dy;
      dx = -dx;
    }
    if (dx < 0) {
      const float tmp = dx;
      dx = dy;
      dy = -tmp;
    }
    p->slope = quadrant + dy / dx;
  }
  quad->reversed_border = dot < 0;
  if (!reversed_border && quad->reversed_border) return 0;
  if (!normal_border && !quad->reversed_border) return 0;
  ptsort(pts, sz);
  { /* remove duplicate points (a by-product of the segmentation) */
    int outpos = 1;
    const struct pt *last = &pts[0];
    for (int i = 1; i < sz; i++) {
      const struct pt *p = &pts[i];
      if (p->x != last->x || p->y != last->y) {
        if (i != outpos) pts[outpos] = *p;
        outpos++;
      }
      last = p;
    }
    cl->n = outpos;
    sz = outpos;
  }
  if (sz < 24) return 0;
  struct line_fit_pt *lfps = compute_lfps(sz, pts, im, w, h);
  int indices[4];
  if (!quad_segment_maxima(c, sz, lfps, indices)) goto finish;
  double lines[4][4];
  for (int i = 0; i < 4; i++) {
    const int i0 = indices[i], i1 = indices[(i + 1) & 3];
    double mse;
    fit_line(lfps, sz, i0, i1, lines[i], NULL, &mse);
    if (mse > c->max_line_fit_mse) {
      res = 0;
      goto finish;
    }
  }
  for (int i = 0; i < 4; i++) {
    const double A00 = lines[i][3], A01 = -lines[(i + 1) & 3][3];
    const double A10 = -lines[i][2], A11 = lines[(i + 1) & 3][2];
    const double B0 = -lines[i][0] + lines[(i + 1) & 3][0];
    const double B1 = -lines[i][1] + lines[(i + 1) & 3][1];
    const double det = A00 * A11 - A10 * A01;
    const double W00 = A11 / det, W01 = -A01 / det;
    if (fabs(det) < 0.001) {
      res = 0;
      goto finish;
    }
    const double L0 = W00 * B0 + W01 * B1;
    quad->p[i][0] = (float)(lines[i][0] + L0 * A00);
    quad->p[i][1] = (float)(lines[i][1] + L0 * A10);
    res = 1;
  }
  { /* reject quads that are too small */
    double area = 0, length[3], p;
    for (int i = 0; i < 3; i++) {
      const int a = i, b = (i + 1) % 3;
      length[i] = sqrt(sq(quad->p[b][0] - quad->p[a][0]) + sq(quad->p[b][1] - quad->p[a][1]));
    }
    p = (length[0] + length[1] + length[2]) / 2;
    area += sqrt(p * (p - length[0]) * (p - length[1]) * (p - length[2]));
    const int idxs[] = {2, 3, 0, 2};
    for (int i = 0; i < 3; i++) {
      const int a = idxs[i], b = idxs[i + 1];
      length[i] = sqrt(sq(quad->p[b][0] - quad->p[a][0]) + sq(quad->p[b][1] - quad->p[a][1]));
    }
    p = (length[0] + length[1] + length[2]) / 2;
    area += sqrt(p * (p - length[0]) * (p - length[1]) * (p - length[2]));
    if (area < 0.95 * tag_width * tag_width) {
      res = 0;
      goto finish;
    }
  }
  for (int i = 0; i < 4; i++) { /* reject quads whose cumulative angle change is not 2 pi */
    const int i0 = i, i1 = (i + 1) & 3, i2 = (i + 2) & 3;
    const double dx1 = quad->p[i1][0] - quad->p[i0][0], dy1 = quad->p[i1][1] - quad->p[i0][1];
    const double dx2 = quad->p[i2][0] - quad->p[i1][0], dy2 = quad->p[i2][1] - quad->p[i1][1];
    const double cos_dtheta = (dx1 * dx2 + dy1 * dy2) / sqrt((dx1 * dx1 + dy1 * dy1) * (dx2 * dx2 + dy2 * dy2));
    if ((cos_dtheta > c->cos_critical_rad || cos_dtheta < -c->cos_critical_rad) || dx1 * dy2 < dy1 * dx2) {
      res = 0;
      goto finish;
    }
  }
finish:
  free(lfps);
  return res;
}

/* refine_edges (apriltag.c): per edge, sample the full-resolution gradient along the normal and refit the line */
static void refine_edges(const orc_config *c, const uint8_t *im, int W, int H, struct quad *quad) {
  double lines[4][4];
  for (int edge = 0; edge < 4; edge++) {
    const int a = edge, b = (edge + 1) & 3;
    double nx = quad->p[b][1] - quad->p[a][1];
    double ny = -quad->p[b][0] + quad->p[a][0];
    const double mag = sqrt(nx * nx + ny * ny);
    nx /= mag;
    ny /= mag;
    if (quad->reversed_border) {
      nx = -nx;
      ny = -ny;
    }
    int nsamples = (int)(mag / 8);
    if (nsamples < 16) nsamples = 16;
    double Mx = 0, My = 0, Mxx = 0, Mxy = 0, Myy = 0, N = 0;
    for (int s = 0; s < nsamples; s++) {
      const double alpha = (1.0 + s) / (nsamples + 1);
      const double x0 = alpha * quad->p[a][0] + (1 - alpha) * quad->p[b][0];
      const double y0 = alpha * quad->p[a][1] + (1 - alpha) * quad->p[b][1];
      double Mn = 0, Mcount = 0;
      const double range = c->quad_decimate + 1;
      for (double n = -range; n <= range; n += 0.25) {
        const double grange = 1;
        const int x1 = (int)(x0 + (n + grange) * nx), y1 = (int)(y0 + (n + grange) * ny);
        if (x1 < 0 || x1 >= W || y1 < 0 || y1 >= H) continue;
        const int x2 = (int)(x0 + (n - grange) * nx), y2 = (int)(y0 + (n - grange) * ny);
        if (x2 < 0 || x2 >= W || y2 < 0 || y2 >= H) continue;
        const int g1 = im[(size_t)y1 * W + x1], g2 = im[(size_t)y2 * W + x2];
        if (g1 < g2) continue; /* gradient the wrong way round */
        const double weight = (g2 - g1) * (g2 - g1);
        Mn += weight * n;
        Mcount += weight;
      }
      if (Mcount == 0) continue;
      const double n0 = Mn / Mcount;
      const double bestx = x0 + n0 * nx, besty = y0 + n0 * ny;
      Mx += bestx; My += besty; Mxx += bestx * bestx; Mxy += bestx * besty; Myy += besty * besty; N++;
    }
    const double Ex = Mx / N, Ey = My / N;
    const double Cxx = Mxx / N - Ex * Ex, Cxy = Mxy / N - Ex * Ey, Cyy = Myy / N - Ey * Ey;
    const double normal_theta = .5 * atan2f((float)(-2 * Cxy), (float)(Cyy - Cxx));
    lines[edge][0] = Ex;
    lines[edge][1] = Ey;
    lines[edge][2] = cosf((float)normal_theta);
    lines[edge][3] = sinf((float)normal_theta);
  }
  for (int i = 0; i < 4; i++) {
    const double A00 = lines[i][3], A01 = -lines[(i + 1) & 3][3];
    const double A10 = -lines[i][2], A11 = lines[(i + 1) & 3][2];
    const double B0 = -lines[i][0] + lines[(i + 1) & 3][0];
    const double B1 = -lines[i][1] + lines[(i + 1) & 3][1];
    const double det = A00 * A11 - A10 * A01;
    if (fabs(det) > 0.001) {
      const double W00 = A11 / det, W01 = -A01 / det;
      const double L0 = W00 * B0 + W01 * B1;
      quad->p[(i + 1) & 3][0] = (float)(lines[i][0] + L0 * A00);
      quad->p[(i + 1) & 3][1] = (float)(lines[i][1] + L0 * A10);
    }
  }
}

/* apriltag_detector_detect */
int orc_classic_detect(const orc_config *c, const uint8_t *gray, orc_detection *out, int cap, int *nquads_out) {
  const int f = c->quad_decimate;
  if (nquads_out) *nquads_out = 0;
  if (f < 1 || c->width <= 0 || c->height <= 0 || c->width % f || c->height % f) return -1;
  const int W = c->width, H = c->height, w = W / f, h = H / f;
  if (w % 4 || h % 4 || w < 8 || h < 8) return -1; /* (upstream handles ragged tiles; the callers here never need them) */
  const size_t n = (size_t)w * h;
  uint8_t *quad_im = (uint8_t *)malloc(n), *thresh = (uint8_t *)malloc(n), *minmax = (uint8_t *)malloc((size_t)(w / 4) * (h / 4) * 2);
  orc_i_decimate(gray, W, f, quad_im, w, h);                   /* image_u8_decimate, integer factors */
  if (c->quad_sigma != 0) orc_i_gaussian_blur(quad_im, w, h, c->quad_sigma);
  orc_i_threshold(quad_im, w, h, c->min_white_black_diff, minmax, thresh);
  unionfind uf;
  uf.parent = (uint32_t *)malloc(n * sizeof(uint32_t));
  uf.size = (uint32_t *)calloc(n, sizeof(uint32_t));
  for (size_t i = 0; i < n; i++) uf.parent[i] = (uint32_t)i;
  connected_components(&uf, thresh, w, h);
  cluster_map m;
  memset(&m, 0, sizeof(m));
  m.nbuckets = (int)(0.2 * w * h);
  if (m.nbuckets < 16) m.nbuckets = 16;
  m.bucket = (int *)malloc((size_t)m.nbuckets * sizeof(int));
  for (int i = 0; i < m.nbuckets; i++) m.bucket[i] = -1;
  gradient_clusters(&m, &uf, thresh, w, h);

  /* fit_quads: family-derived limits (apriltag_quad_thresh.c) */
  int normal_border, reversed_border;
  orc_i_border_polarities(c, &normal_border, &reversed_border);
  const int tag_width = orc_i_min_tag_width(c);
  struct quad *quads = (struct quad *)malloc(((size_t)m.n + 1) * sizeof(struct quad));
  int nq = 0;
  for (int ci = 0; ci < m.n; ci++) {
    cluster *cl = &m.items[ci];
    if (cl->n < c->min_cluster_pixels) continue;
    if (cl->n > 2 * (2 * w + 2 * h)) continue; /* a cluster cannot be longer than twice the image perimeter */
    struct quad q;
    memset(&q, 0, sizeof(q));
    if (fit_quad(c, quad_im, w, h, cl, &q, tag_width, normal_border, reversed_border)) quads[nq++] = q;
  }
  if (f > 1) { /* centres of decimated pixels -> full-resolution coordinates */
    for (int i = 0; i < nq; i++)
      for (int j = 0; j < 4; j++) {
        quads[i].p[j][0] = (float)((quads[i].p[j][0] - 0.5) * f + 0.5);
        quads[i].p[j][1] = (float)((quads[i].p[j][1] - 0.5) * f + 0.5);
      }
  }
  if (nquads_out) *nquads_out = nq;

  /* quad_decode_task */
  orc_detection *dets = (orc_detection *)malloc(((size_t)nq * orc_i_family_slots(c) + 1) * sizeof(orc_detection));
  int nd = 0;
  for (int qi = 0; qi < nq; qi++) {
    struct quad *q = &quads[qi];
    if (c->refine_edges) refine_edges(c, gray, W, H, q);
    double corr[4][4];
    for (int i = 0; i < 4; i++) {
      corr[i][0] = (i == 0 || i == 3) ? -1 : 1;
      corr[i][1] = (i == 0 || i == 1) ? -1 : 1;
      corr[i][2] = q->p[i][0];
      corr[i][3] = q->p[i][1];
    }
    double Hm[9];
    if (orc_homography_compute(corr, Hm) != 0) continue;
    const double det = Hm[0] * (Hm[4] * Hm[8] - Hm[5] * Hm[7]) - Hm[1] * (Hm[3] * Hm[8] - Hm[5] * Hm[6]) +
                       Hm[2] * (Hm[3] * Hm[7] - Hm[4] * Hm[6]);
    if (!(fabs(det) > 1e-300)) continue;
    for (int fi = 0; fi < orc_i_family_slots(c); fi++) {
      const orc_family *fam = orc_i_family(c, fi);
      if (!fam || (fam->reversed_border != 0) != (q->reversed_border != 0)) continue;
      int id, hamming, rotation;
      const float margin = orc_i_quad_decode(c, fam, gray, W, H, Hm, &id, &hamming, &rotation);
      if (margin >= 0 && hamming < 255) orc_i_fill_detection(&dets[nd++], fi, id, hamming, margin, rotation, Hm);
    }
  }
  nd = orc_i_reconcile(dets, nd);
  const int ncopy = nd < cap ? nd : cap;
  if (out && ncopy > 0) memcpy(out, dets, (size_t)ncopy * sizeof(orc_detection));

  for (int ci = 0; ci < m.n; ci++) free(m.items[ci].pts);
  free(m.items); free(m.next); free(m.bucket);
  free(uf.parent); free(uf.size);
  free(quads); free(dets);
  free(quad_im); free(thresh); free(minmax);
  return nd;
}
