/*
 * TEST INFRASTRUCTURE -- CPU oracle, see apriltag_oracle.h for scope and parity status.
 *
 * Every stage cites the reference lines (relative to /root/reference) whose
 * behaviour it restates.  This is a restatement of *behaviour* in sequential C:
 * none of the reference's kernel structure (CUB passes, shared-memory staging,
 * block-based union-find) is reproduced.
 */
#include "apriltag_oracle.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "cuda_math_emul.h"
#include "oracle_internal.h"
#include "tag_families.h"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

float orc_emul_atan2f(float y, float x) { return orc_cuda_atan2f(y, x); }
float orc_emul_hypotf(float a, float b) { return orc_cuda_hypotf(a, b); }
uint64_t orc_tag36h11_code(int id) { return orc_tag36h11_codes[id]; }

/* Built-in families (libapriltag tagXXhYY_create(), apriltag_utils.cu:10-27): AprilTag 3 layouts, normal border,
 * added with bits_corrected = 2 (apriltags_cuda_detector.cu:140). */
static const orc_family k_families[ORC_NUM_FAMILIES] = {
    {"tag36h11", orc_tag36h11_NBITS, orc_tag36h11_NCODES, orc_tag36h11_WIDTH_AT_BORDER, orc_tag36h11_TOTAL_WIDTH, 0,
     orc_tag36h11_MIN_HAMMING, orc_tag36h11_codes, orc_tag36h11_bit_x, orc_tag36h11_bit_y, 2},
    {"tag25h9", orc_tag25h9_NBITS, orc_tag25h9_NCODES, orc_tag25h9_WIDTH_AT_BORDER, orc_tag25h9_TOTAL_WIDTH, 0,
     orc_tag25h9_MIN_HAMMING, orc_tag25h9_codes, orc_tag25h9_bit_x, orc_tag25h9_bit_y, 2},
    {"tag16h5", orc_tag16h5_NBITS, orc_tag16h5_NCODES, orc_tag16h5_WIDTH_AT_BORDER, orc_tag16h5_TOTAL_WIDTH, 0,
     orc_tag16h5_MIN_HAMMING, orc_tag16h5_codes, orc_tag16h5_bit_x, orc_tag16h5_bit_y, 2},
};
const orc_family *orc_family_get(int index) { return (index >= 0 && index < ORC_NUM_FAMILIES) ? &k_families[index] : NULL; }
int orc_family_index(const char *name) {
  for (int i = 0; i < ORC_NUM_FAMILIES; i++)
    if (strcmp(name, k_families[i].name) == 0) return i;
  return -1;
}
static uint32_t family_mask_of(const orc_config *c) { return c->family_mask ? c->family_mask : 1u; }

/* The families a configuration decodes, numbered as its detections number them: the caller's list, or the built-in
 * families family_mask selects at their built-in index (a slot the mask leaves out is NULL). */
int orc_i_family_slots(const orc_config *c) { return c->nfamilies > 0 ? c->nfamilies : ORC_NUM_FAMILIES; }
const orc_family *orc_i_family(const orc_config *c, int slot) {
  if (c->nfamilies > 0) return &c->families[slot];
  return ((family_mask_of(c) >> slot) & 1u) ? &k_families[slot] : NULL;
}
/* Border polarities over the families in use (apriltag_gpu.cu:169-177). */
void orc_i_border_polarities(const orc_config *c, int *normal_border, int *reversed_border) {
  *normal_border = *reversed_border = 0;
  for (int fi = 0; fi < orc_i_family_slots(c); fi++) {
    const orc_family *fam = orc_i_family(c, fi);
    if (!fam) continue;
    *normal_border |= !fam->reversed_border;
    *reversed_border |= fam->reversed_border != 0;
  }
}

void orc_default_config(orc_config *c, int width, int height, int format) {
  memset(c, 0, sizeof(*c));
  c->width = width;
  c->height = height;
  c->format = format;
  /* apriltag_detector_create() defaults as set by the node,
   * src/apriltags_cuda/src/apriltags_cuda_detector.cu:142-147 */
  c->quad_decimate = 2;
  c->quad_sigma = 0.0f;
  c->refine_edges = 1;
  c->decode_sharpening = 0.25;
  c->min_cluster_pixels = 5;
  c->max_nmaxima = 10;
  c->cos_critical_rad = cosf((float)(10 * M_PI / 180));
  c->max_line_fit_mse = 10.0f;
  c->min_white_black_diff = 5;
  c->fx = 1.0; c->fy = 1.0; c->cx = 0.0; c->cy = 0.0;
  c->max_stage = ORC_STAGE_DECODE;
  c->family_mask = 1; /* tag36h11, the family the node configures (apriltags_cuda_detector.hpp:213) */
}

/* ------------------------------------------------------------------------- */
/* Stage 1: gray + decimate (+ blur)                                          */
/* ------------------------------------------------------------------------- */

/* threshold.cu:16-40 (YUYV: gray[i] = in[2i]).  BGR follows the luma OpenCV's
 * COLOR_BGR2YUV_YUYV produces, which is what the node feeds the detector
 * (apriltags_cuda_detector.cu:399-404). */
void orc_i_to_gray(const orc_config *c, const uint8_t *in, uint8_t *gray) {
  const size_t N = (size_t)c->width * c->height;
  if (c->format == ORC_FMT_GRAY8) {
    memcpy(gray, in, N);
  } else if (c->format == ORC_FMT_YUYV) {
    for (size_t i = 0; i < N; i++) gray[i] = in[2 * i];
  } else {
    for (size_t i = 0; i < N; i++) {
      const int b = in[3 * i], g = in[3 * i + 1], r = in[3 * i + 2];
      gray[i] = (uint8_t)((4211 * r + 8258 * g + 1606 * b + (1 << 13) + (16 << 14)) >> 14);
    }
  }
}

/* threshold.cu:27-31: point subsample. */
void orc_i_decimate(const uint8_t *gray, int W, int f, uint8_t *out, int w, int h) {
  for (int y = 0; y < h; y++)
    for (int x = 0; x < w; x++) out[(size_t)y * w + x] = gray[(size_t)(y * f) * W + x * f];
}

/* Upstream image_u8_gaussian_blur / convolve (libapriltag common/image_u8.c;
 * RECALLED -- the reference GPU path ignores quad_sigma, SURVEY App. C). */
static void convolve1d(const uint8_t *x, uint8_t *y, int sz, const uint8_t *k, int ksz) {
  for (int i = 0; i < ksz / 2 && i < sz; i++) y[i] = x[i];
  for (int i = 0; i < sz - ksz; i++) {
    uint32_t acc = 0;
    for (int j = 0; j < ksz; j++) acc += (uint32_t)k[j] * x[i + j];
    y[ksz / 2 + i] = (uint8_t)(acc >> 8);
  }
  for (int i = sz - ksz + ksz / 2; i < sz; i++)
    if (i >= 0) y[i] = x[i];
}

static int blur_kernel(float quad_sigma, uint8_t *k) {
  const float sigma = fabsf(quad_sigma);
  int ksz = (int)(4 * sigma);
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
  for (int i = 0; i < ksz; i++) k[i] = (uint8_t)(dk[i] / acc * 255);
  return ksz;
}

void orc_i_gaussian_blur(uint8_t *im, int w, int h, float quad_sigma) {
  uint8_t k[32];
  const int ksz = blur_kernel(quad_sigma, k);
  if (!ksz) return;
  uint8_t *orig = NULL;
  if (quad_sigma < 0) {
    orig = (uint8_t *)malloc((size_t)w * h);
    memcpy(orig, im, (size_t)w * h);
  }
  uint8_t *xb = (uint8_t *)malloc(w > h ? w : h), *yb = (uint8_t *)malloc(w > h ? w : h);
  for (int y = 0; y < h; y++) {
    memcpy(xb, im + (size_t)y * w, w);
    convolve1d(xb, im + (size_t)y * w, w, k, ksz);
  }
  for (int x = 0; x < w; x++) {
    for (int y = 0; y < h; y++) xb[y] = im[(size_t)y * w + x];
    convolve1d(xb, yb, h, k, ksz);
    for (int y = 0; y < h; y++) im[(size_t)y * w + x] = yb[y];
  }
  free(xb);
  free(yb);
  if (orig) {
    for (size_t i = 0; i < (size_t)w * h; i++) {
      int v = 2 * orig[i] - im[i];
      if (v < 0) v = 0;
      if (v > 255) v = 255;
      im[i] = (uint8_t)v;
    }
    free(orig);
  }
}

/* ------------------------------------------------------------------------- */
/* Stage 2: adaptive threshold   threshold.cu:60-147                          */
/* ------------------------------------------------------------------------- */
void orc_i_threshold(const uint8_t *im, int w, int h, int min_white_black_diff, uint8_t *minmax_out,
                      uint8_t *out) {
  const int tw = w / 4, th = h / 4;
  uint8_t *mm = (uint8_t *)malloc((size_t)tw * th * 2);
  for (int ty = 0; ty < th; ty++)
    for (int tx = 0; tx < tw; tx++) { /* threshold.cu:60-80 */
      int mn = 255, mx = 0;
      for (int dy = 0; dy < 4; dy++)
        for (int dx = 0; dx < 4; dx++) {
          const int v = im[(size_t)(ty * 4 + dy) * w + tx * 4 + dx];
          if (v < mn) mn = v;
          if (v > mx) mx = v;
        }
      mm[2 * (ty * tw + tx)] = (uint8_t)mn;
      mm[2 * (ty * tw + tx) + 1] = (uint8_t)mx;
    }
  for (int ty = 0; ty < th; ty++)
    for (int tx = 0; tx < tw; tx++) { /* threshold.cu:84-118 */
      int mn = 255, mx = 0;
      for (int j = -1; j <= 1; j++)
        for (int i = -1; i <= 1; i++) {
          const int rx = tx + i, ry = ty + j;
          if (rx < 0 || rx >= tw || ry < 0 || ry >= th) continue;
          const int a = mm[2 * (ry * tw + rx)], b = mm[2 * (ry * tw + rx) + 1];
          if (a < mn) mn = a;
          if (b > mx) mx = b;
        }
      minmax_out[2 * (ty * tw + tx)] = (uint8_t)mn;
      minmax_out[2 * (ty * tw + tx) + 1] = (uint8_t)mx;
    }
  for (int y = 0; y < h; y++)
    for (int x = 0; x < w; x++) { /* threshold.cu:121-147 */
      const int mn = minmax_out[2 * ((y / 4) * tw + x / 4)], mx = minmax_out[2 * ((y / 4) * tw + x / 4) + 1];
      uint8_t r;
      if (mx - mn < min_white_black_diff) {
        r = 127;
      } else {
        const uint8_t t = (uint8_t)(mn + (mx - mn) / 2);
        r = im[(size_t)y * w + x] > t ? 255 : 0;
      }
      out[(size_t)y * w + x] = r;
    }
  free(mm);
}

/* ------------------------------------------------------------------------- */
/* Stage 3: connected components  labeling_allegretti_2019_BKE.cu:114-462     */
/* Semantics only: 255 is 8-connected, 0 is 4-connected, 127 is nobody's       */
/* neighbour.  Label = smallest pixel index in the component (any correct CCL */
/* matches the reference up to relabelling); size = pixel count at the root.  */
/* ------------------------------------------------------------------------- */
static uint32_t uf_find(uint32_t *p, uint32_t a) {
  uint32_t r = a;
  while (p[r] != r) r = p[r];
  while (p[a] != r) {
    const uint32_t n = p[a];
    p[a] = r;
    a = n;
  }
  return r;
}
static void uf_union(uint32_t *p, uint32_t a, uint32_t b) {
  a = uf_find(p, a);
  b = uf_find(p, b);
  if (a < b) p[b] = a;
  else if (b < a) p[a] = b;
}

static void label_components(const uint8_t *t, int w, int h, uint32_t *labels, uint32_t *sizes) {
  const size_t n = (size_t)w * h;
  for (size_t i = 0; i < n; i++) labels[i] = (uint32_t)i;
  for (int y = 0; y < h; y++)
    for (int x = 0; x < w; x++) {
      const uint32_t i = (uint32_t)(y * w + x);
      const uint8_t v = t[i];
      if (v == 127) continue;
      if (x > 0 && t[i - 1] == v) uf_union(labels, i, i - 1);
      if (y > 0 && t[i - w] == v) uf_union(labels, i, i - w);
      if (v == 255 && y > 0) {
        if (x > 0 && t[i - w - 1] == 255) uf_union(labels, i, i - w - 1);
        if (x + 1 < w && t[i - w + 1] == 255) uf_union(labels, i, i - w + 1);
      }
    }
  memset(sizes, 0, n * sizeof(uint32_t));
  for (size_t i = 0; i < n; i++) {
    labels[i] = uf_find(labels, (uint32_t)i);
    if (t[i] != 127) sizes[labels[i]]++;
  }
}

/* ------------------------------------------------------------------------- */
/* Stage 4: boundary points   apriltag_gpu.cu:226-360 (BlobDiff)              */
/* ------------------------------------------------------------------------- */
static const int kDx[4] = {1, 1, 0, -1};
static const int kDy[4] = {0, 1, 1, 1};

static int cmp_point(const void *a_, const void *b_) {
  const orc_point *a = (const orc_point *)a_, *b = (const orc_point *)b_;
  if (a->rep0 != b->rep0) return a->rep0 < b->rep0 ? -1 : 1;
  if (a->rep1 != b->rep1) return a->rep1 < b->rep1 ? -1 : 1;
  if (a->dir != b->dir) return a->dir < b->dir ? -1 : 1;
  if (a->by != b->by) return a->by < b->by ? -1 : 1;
  if (a->bx != b->bx) return a->bx < b->bx ? -1 : 1;
  return 0;
}

static void boundary_points(orc_result *r) {
  const int w = r->w, h = r->h;
  const uint8_t *t = r->thresh;
  const uint32_t *L = r->labels, *S = r->sizes;
  size_t cap = 1024, np = 0;
  orc_point *pts = (orc_point *)malloc(cap * sizeof(orc_point));
  for (int y = 1; y <= h - 2; y++)
    for (int x = 1; x <= w - 2; x++) { /* apriltag_gpu.cu:239,276-281 */
      const uint32_t i = (uint32_t)(y * w + x);
      const uint8_t v0 = t[i];
      const uint32_t rep0 = L[i];
      if (v0 == 127 || S[rep0] < 25) continue; /* :284 */
      for (int d = 0; d < 4; d++) {
        if (d == 3) { /* :339-357 duplicate suppression */
          const uint8_t vl = t[i - 1], v2 = t[i + w];
          if (vl != 127 && v2 != 127 && v2 != vl) {
            if (x != 1 && S[L[i - 1]] >= 25 && S[L[i + w]] >= 25) continue;
          }
        }
        const uint32_t j = (uint32_t)((y + kDy[d]) * w + x + kDx[d]);
        const uint8_t v1 = t[j];
        if (v0 + v1 != 255) continue; /* :305 */
        const uint32_t rep1 = L[j];
        if (S[rep1] < 25) continue; /* :306 */
        if (np == cap) {
          cap *= 2;
          pts = (orc_point *)realloc(pts, cap * sizeof(orc_point));
        }
        orc_point *p = &pts[np++];
        memset(p, 0, sizeof(*p));
        p->rep0 = rep0 < rep1 ? rep0 : rep1;
        p->rep1 = rep0 < rep1 ? rep1 : rep0;
        p->bx = (uint16_t)x;
        p->by = (uint16_t)y;
        p->x = (uint16_t)(2 * x + kDx[d]); /* points.h:111-116 */
        p->y = (uint16_t)(2 * y + kDy[d]);
        p->dir = (uint8_t)d;
        p->b2w = v1 > v0; /* :316 */
      }
    }
  /* C1 + C2 (apriltag_gpu.cu:788-825): order-preserving compaction of the dense
   * [dir][y][x] array followed by a stable sort on the blob pair. */
  qsort(pts, np, sizeof(orc_point), cmp_point);
  r->points = pts;
  r->num_points = (int)np;
}

/* ------------------------------------------------------------------------- */
/* Stage 5: per blob-pair extents + blob filter                               */
/* apriltag_gpu.cu:418-454 (extents), :522-575 (SelectBlobs), :871-905         */
/* ------------------------------------------------------------------------- */
static double extents_cx(const orc_cluster *e) { /* line_fit_filter.h:44-46 */
  return (double)((float)(e->min_x + e->max_x) * 0.5f) + 0.05118;
}
static double extents_cy(const orc_cluster *e) { /* line_fit_filter.h:47-49 */
  return (double)((float)(e->min_y + e->max_y) * 0.5f) + -0.028581;
}
static float extents_dot(const orc_cluster *e) { /* line_fit_filter.h:51-58 */
  const int64_t a = e->pxgx_plus_pygy_sum * 2 - (int64_t)((int32_t)(e->min_x + e->max_x) * e->gx_sum) -
                    (int64_t)((int32_t)(e->min_y + e->max_y) * e->gy_sum);
  const double d = (double)a * 0.5 - 0.05118 * (double)e->gx_sum + 0.028581 * (double)e->gy_sum;
  return (float)d;
}

int orc_i_min_tag_width(const orc_config *c) { /* apriltag_gpu.cu:169-181: min over the families */
  int m = 1000000;
  for (int f = 0; f < orc_i_family_slots(c); f++)
    if (orc_i_family(c, f) && orc_i_family(c, f)->width_at_border < m) m = orc_i_family(c, f)->width_at_border;
  m = (int)((float)m / (float)c->quad_decimate);
  if (m < 3) m = 3;
  return m;
}
static int min_tag_width(const orc_config *c) { return orc_i_min_tag_width(c); }

static void clusters_and_filter(const orc_config *c, orc_result *r) {
  const int np = r->num_points;
  orc_cluster *cl = (orc_cluster *)malloc(((size_t)np + 1) * sizeof(orc_cluster));
  int nc = 0;
  for (int i = 0; i < np;) {
    const orc_point *p0 = &r->points[i];
    orc_cluster e;
    memset(&e, 0, sizeof(e));
    e.rep0 = p0->rep0;
    e.rep1 = p0->rep1;
    e.min_x = e.max_x = p0->x;
    e.min_y = e.max_y = p0->y;
    e.start = (uint32_t)i;
    int j = i;
    for (; j < np && r->points[j].rep0 == e.rep0 && r->points[j].rep1 == e.rep1; j++) {
      const orc_point *p = &r->points[j];
      const int gx = p->b2w ? kDx[p->dir] : -kDx[p->dir]; /* points.h:120-125 */
      const int gy = p->b2w ? kDy[p->dir] : -kDy[p->dir];
      if (p->x < e.min_x) e.min_x = p->x;
      if (p->x > e.max_x) e.max_x = p->x;
      if (p->y < e.min_y) e.min_y = p->y;
      if (p->y > e.max_y) e.max_y = p->y;
      e.count++;
      e.gx_sum += gx;
      e.gy_sum += gy;
      e.pxgx_plus_pygy_sum += (int64_t)p->x * gx + (int64_t)p->y * gy;
    }
    cl[nc++] = e;
    i = j;
  }
  /* SelectBlobs (apriltag_gpu.cu:534-559).  The perimeter bound 2*(W+H) at
   * :871 is written for decimate 2; in quad-image units it is 4*(w+h). */
  const uint32_t min_px = (uint32_t)(c->min_cluster_pixels > 24 ? c->min_cluster_pixels : 24);
  const uint32_t max_px = (uint32_t)(4 * (r->w + r->h));
  const int tag_width = min_tag_width(c);
  int normal_border, reversed_border;
  orc_i_border_polarities(c, &normal_border, &reversed_border);
  uint32_t sel = 0;
  for (int i = 0; i < nc; i++) {
    orc_cluster *e = &cl[i];
    int ok = 1;
    if (e->count < min_px) ok = 0;
    if (e->count > max_px) ok = 0;
    if ((e->max_x - e->min_x) * (e->max_y - e->min_y) < tag_width) ok = 0;
    const int quad_reversed = extents_dot(e) < 0.0;
    if (!reversed_border && quad_reversed) ok = 0;
    if (!normal_border && !quad_reversed) ok = 0;
    e->selected = ok;
    e->sel_start = sel;
    if (ok) sel += e->count;
  }
  r->clusters = cl;
  r->num_clusters = nc;
  r->num_selected_points = (int)sel;
}

/* ------------------------------------------------------------------------- */
/* Stage 6: angle sort + prefix moments                                       */
/* apriltag_gpu.cu:380-412 (theta), :909-956 (select + sort), :631-687 (moments)*/
/* ------------------------------------------------------------------------- */
static int cmp_spoint(const void *a_, const void *b_) {
  const orc_spoint *a = (const orc_spoint *)a_, *b = (const orc_spoint *)b_;
  if (a->blob != b->blob) return a->blob < b->blob ? -1 : 1;
  if (a->theta != b->theta) return a->theta < b->theta ? -1 : 1;
  /* the radix sort is stable, ties keep the compaction order (dir, y, x) */
  if (a->dir != b->dir) return a->dir < b->dir ? -1 : 1;
  if (a->by != b->by) return a->by < b->by ? -1 : 1;
  if (a->bx != b->bx) return a->bx < b->bx ? -1 : 1;
  return 0;
}

static void sort_and_moments(orc_result *r) {
  const int ns = r->num_selected_points;
  r->spoints = (orc_spoint *)malloc(((size_t)ns + 1) * sizeof(orc_spoint));
  r->lfps = (orc_lfp *)malloc(((size_t)ns + 1) * sizeof(orc_lfp));
  int k = 0;
  for (int ci = 0; ci < r->num_clusters; ci++) {
    const orc_cluster *e = &r->clusters[ci];
    if (!e->selected) continue;
    const double cx = extents_cx(e), cy = extents_cy(e);
    for (uint32_t j = 0; j < e->count; j++) {
      const orc_point *p = &r->points[e->start + j];
      orc_spoint *s = &r->spoints[k++];
      memset(s, 0, sizeof(*s));
      s->blob = (uint32_t)ci;
      /* apriltag_gpu.cu:402-406 */
      const float fy = (float)((double)p->y - cy), fx = (float)((double)p->x - cx);
      const float theta = (float)(((double)orc_cuda_atan2f(fy, fx) + M_PI) * 8e6);
      long long ti = llrintf(theta);
      if (ti < 0) ti = 0;
      s->theta = (uint32_t)(ti & 0xfffffff);
      s->x = p->x; s->y = p->y; s->bx = p->bx; s->by = p->by; s->dir = p->dir;
    }
  }
  qsort(r->spoints, ns, sizeof(orc_spoint), cmp_spoint);
  /* TransformLineFitPoint + InclusiveScanByKey, apriltag_gpu.cu:631-687,984-987 */
  const int w = r->w, h = r->h;
  const uint8_t *im = r->quad_im;
  orc_lfp acc;
  memset(&acc, 0, sizeof(acc));
  for (int i = 0; i < ns; i++) {
    const orc_spoint *s = &r->spoints[i];
    if (i == 0 || r->spoints[i - 1].blob != s->blob) memset(&acc, 0, sizeof(acc));
    const int32_t ix2 = s->x + 1, iy2 = s->y + 1;
    const int32_t ix = ix2 / 2, iy = iy2 / 2;
    int32_t W = 1;
    if (ix > 0 && ix + 1 < w && iy > 0 && iy + 1 < h) {
      const int32_t gx = im[iy * w + ix + 1] - im[iy * w + ix - 1];
      const int32_t gy = im[(iy + 1) * w + ix] - im[(iy - 1) * w + ix];
      W = (int32_t)(orc_cuda_hypotf((float)gx, (float)gy) + 1);
    }
    acc.Mx += (int64_t)W * ix2;
    acc.My += (int64_t)W * iy2;
    acc.Mxx += (int64_t)W * ix2 * ix2;
    acc.Mxy += (int64_t)W * ix2 * iy2;
    acc.Myy += (int64_t)W * iy2 * iy2;
    acc.W += W;
    r->lfps[i] = acc;
  }
}

/* ------------------------------------------------------------------------- */
/* Stage 7: line-fit errors, smoothing, peaks   line_fit_filter.cu:22-36,      */
/* :217-278 (CalculateError), :504-525 (filter), :572-590 (peaks)              */
/* ------------------------------------------------------------------------- */
static orc_moments read_moments(const orc_lfp *lf, uint32_t count, uint32_t i0, uint32_t i1) {
  /* line_fit_filter.cu:745-796 (ReadMoments) == :230-274 */
  orc_moments m;
  memset(&m, 0, sizeof(m));
  if (i0 < i1) {
    m.N = (int32_t)(i1 - i0 + 1);
    const orc_lfp *a = &lf[i1];
    m.Mx = a->Mx; m.My = a->My; m.Mxx = a->Mxx; m.Mxy = a->Mxy; m.Myy = a->Myy; m.W = a->W;
    if (i0 > 0) {
      const orc_lfp *b = &lf[i0 - 1];
      m.Mx -= b->Mx; m.My -= b->My; m.Mxx -= b->Mxx; m.Mxy -= b->Mxy; m.Myy -= b->Myy; m.W -= b->W;
    }
  } else {
    const orc_lfp *b = &lf[i0 - 1], *z = &lf[count - 1], *a = &lf[i1];
    m.Mx = z->Mx - b->Mx + a->Mx;
    m.My = z->My - b->My + a->My;
    m.Mxx = z->Mxx - b->Mxx + a->Mxx;
    m.Mxy = z->Mxy - b->Mxy + a->Mxy;
    m.Myy = z->Myy - b->Myy + a->Myy;
    m.W = z->W - b->W + a->W;
    m.N = (int32_t)(count - i0 + i1 + 1);
  }
  return m;
}

/* Shared by FitLineError (line_fit_filter.cu:22-36) and FitLine (:798-872). */
static float eig_small_of(const orc_moments *m, float *hypot_out, int64_t *Cxx_o, int64_t *Cxy_o, int64_t *Cyy_o) {
  const int64_t Cxx = m->Mxx * m->W - m->Mx * m->Mx;
  const int64_t Cxy = m->Mxy * m->W - m->Mx * m->My;
  const int64_t Cyy = m->Myy * m->W - m->My * m->My;
  const float hyp = orc_cuda_hypotf((float)(Cxx - Cyy), (float)(2 * Cxy));
  const float eight_w2 = (float)((double)(m->W * m->W) * 8.0);
  const float eig = ((float)(Cxx + Cyy) - hyp) / eight_w2;
  if (hypot_out) *hypot_out = hyp;
  if (Cxx_o) { *Cxx_o = Cxx; *Cxy_o = Cxy; *Cyy_o = Cyy; }
  return eig;
}

static const float kFilter[7] = {/* line_fit_filter.h:122-128 */
    0.01110899634659290314f, 0.13533528149127960205f, 0.60653066635131835938f, 1.0f,
    0.60653066635131835938f, 0.13533528149127960205f, 0.01110899634659290314f};

static void errors_and_peaks(orc_result *r) {
  const int ns = r->num_selected_points;
  r->errs = (double *)calloc((size_t)ns + 1, sizeof(double));
  r->filtered_errs = (double *)calloc((size_t)ns + 1, sizeof(double));
  r->is_peak = (uint8_t *)calloc((size_t)ns + 1, 1);
  for (int ci = 0; ci < r->num_clusters; ci++) {
    const orc_cluster *e = &r->clusters[ci];
    if (!e->selected) continue;
    const uint32_t cnt = e->count, off = e->sel_start;
    const orc_lfp *lf = r->lfps + off;
    const uint32_t ksz = cnt / 12 < 20 ? cnt / 12 : 20; /* :112 */
    for (uint32_t i = 0; i < cnt; i++) {
      const uint32_t i0 = (i + 2 * cnt - ksz) % cnt, i1 = (i + cnt + ksz) % cnt; /* :220-221 */
      const orc_moments m = read_moments(lf, cnt, i0, i1);
      const float eig = eig_small_of(&m, NULL, NULL, NULL, NULL);
      r->errs[off + i] = (double)((float)m.N * eig); /* :35 */
    }
    for (uint32_t i = 0; i < cnt; i++) {
      double acc = 0.0;
      for (int j = 0; j < 7; j++) {
        const double ev = r->errs[off + (i + cnt + j - 3) % cnt];
        acc += ev * (double)kFilter[j]; /* :512-524 */
      }
      r->filtered_errs[off + i] = acc;
    }
    for (uint32_t i = 0; i < cnt; i++) {
      const double b = r->filtered_errs[off + (i + cnt - 1) % cnt], m = r->filtered_errs[off + i],
                   a = r->filtered_errs[off + (i + 1) % cnt];
      r->is_peak[off + i] = (m > b && m > a); /* :582 */
    }
  }
}

/* ------------------------------------------------------------------------- */
/* Stage 8: quad fit   line_fit_filter.cu:889-1061 (QuadFitCalculator),        */
/* :1088-1193 (DoFitQuads); peak selection apriltag_gpu.cu:1001-1078           */
/* ------------------------------------------------------------------------- */
typedef struct {
  float err;
  uint32_t idx;
} peak_t;
static int cmp_peak(const void *a_, const void *b_) {
  const peak_t *a = (const peak_t *)a_, *b = (const peak_t *)b_;
  if (a->err < b->err) return -1;
  if (a->err > b->err) return 1;
  return a->idx < b->idx ? -1 : (a->idx > b->idx);
}
static int cmp_u32(const void *a, const void *b) {
  const uint32_t x = *(const uint32_t *)a, y = *(const uint32_t *)b;
  return x < y ? -1 : x > y;
}

/* FitLine, line_fit_filter.cu:798-872 (device) and apriltag_detect.cu:38-90 (host). */
static void fit_line(const orc_moments *m, double *lp01, double *lp23, double *err, double *mse) {
  float hyp;
  int64_t Cxx, Cxy, Cyy;
  const float eig = eig_small_of(m, &hyp, &Cxx, &Cxy, &Cyy);
  if (lp01) {
    lp01[0] = (double)((float)m->Mx / (float)(m->W * 2));
    lp01[1] = (double)((float)m->My / (float)(m->W * 2));
  }
  if (lp23) {
    const float nx1 = (float)(Cxx - Cyy) - hyp;
    const float ny1 = (float)(2 * Cxy);
    const float M1 = nx1 * nx1 + ny1 * ny1;
    const float nx2 = (float)(2 * Cxy);
    const float ny2 = (float)(Cyy - Cxx) - hyp;
    const float M2 = nx2 * nx2 + ny2 * ny2;
    float nx, ny;
    if (M1 > M2) { nx = nx1; ny = ny1; } else { nx = nx2; ny = ny2; }
    const float len = orc_cuda_hypotf(nx, ny);
    lp23[0] = (double)(nx / len);
    lp23[1] = (double)(ny / len);
  }
  *err = (double)((float)m->N * eig);
  *mse = (double)eig;
}

#define ORC_DBL_MAX 1.7976931348623157e308

static void fit_quads(const orc_config *c, orc_result *r) {
  r->fitquads = (orc_fitquad *)calloc((size_t)r->num_clusters + 1, sizeof(orc_fitquad));
  int nq = 0;
  const double max_mse = (double)c->max_line_fit_mse;
  const double max_dot = (double)c->cos_critical_rad;
  for (int ci = 0; ci < r->num_clusters; ci++) {
    const orc_cluster *e = &r->clusters[ci];
    if (!e->selected) continue;
    const uint32_t cnt = e->count, off = e->sel_start;
    const orc_lfp *lf = r->lfps + off;
    /* C8-C10: compact peaks, sort by (blob, -filtered as f32), apriltag_gpu.cu:1001-1078 */
    peak_t *pk = (peak_t *)malloc((size_t)cnt * sizeof(peak_t));
    int npk = 0;
    for (uint32_t i = 0; i < cnt; i++)
      if (r->is_peak[off + i]) {
        pk[npk].err = (float)(-r->filtered_errs[off + i]); /* line_fit_filter.cu:585 */
        pk[npk].idx = i;
        npk++;
      }
    if (npk == 0) { free(pk); continue; }
    qsort(pk, npk, sizeof(peak_t), cmp_peak);
    const int nm = npk < 10 ? npk : 10;
    uint32_t idx[10];
    for (int i = 0; i < nm; i++) idx[i] = pk[i].idx;
    free(pk);
    qsort(idx, nm, sizeof(uint32_t), cmp_u32); /* line_fit_filter.cu:1104-1119 */

    orc_fitquad *q = &r->fitquads[nq++];
    q->blob = (uint32_t)ci;
    q->rep0 = e->rep0;
    q->rep1 = e->rep1;
    q->npeaks = npk;
    double best = ORC_DBL_MAX;
    int bm[4] = {0, 1, 2, 3};
    /* nested-loop order == Unrank order (line_fit_filter.cu:709-728); ties keep the
     * lowest rank (MinQuadError, :1071-1080, through an order-preserving BlockReduce) */
    for (int m0 = 0; m0 < nm - 3; m0++)
      for (int m1 = m0 + 1; m1 < nm - 2; m1++) {
        double e01, mse01, p01[2];
        orc_moments mo = read_moments(lf, cnt, idx[m0], idx[m1]);
        fit_line(&mo, NULL, p01, &e01, &mse01);
        if (mse01 > max_mse) continue; /* :964-966 */
        for (int m2 = m1 + 1; m2 < nm - 1; m2++) {
          double e12, mse12, p12[2];
          mo = read_moments(lf, cnt, idx[m1], idx[m2]);
          fit_line(&mo, NULL, p12, &e12, &mse12);
          if (mse12 > max_mse) continue; /* :1009 */
          const double dot = p01[0] * p12[0] + p01[1] * p12[1];
          if (fabs(dot) > max_dot) continue; /* :1017 */
          for (int m3 = m2 + 1; m3 < nm; m3++) {
            double e23, mse23, e30, mse30;
            mo = read_moments(lf, cnt, idx[m2], idx[m3]);
            fit_line(&mo, NULL, NULL, &e23, &mse23);
            if (mse23 > max_mse) continue;
            mo = read_moments(lf, cnt, idx[m3], idx[m0]);
            fit_line(&mo, NULL, NULL, &e30, &mse30);
            if (mse30 > max_mse) continue;
            const double tot = e01 + e12 + e23 + e30; /* :1047 */
            if (tot < best) {
              best = tot;
              bm[0] = m0; bm[1] = m1; bm[2] = m2; bm[3] = m3;
            }
          }
        }
      }
    q->err = best;
    q->valid = best < (double)(c->max_line_fit_mse * (float)cnt); /* :1165 */
    if (q->valid) {
      for (int i = 0; i < 4; i++) q->indices[i] = idx[bm[i]];
      for (int i = 0; i < 4; i++)
        q->moments[i] = read_moments(lf, cnt, q->indices[i], q->indices[(i + 1) & 3]); /* :1188-1191 */
    }
  }
  r->num_fitquads = nq;
}

/* ------------------------------------------------------------------------- */
/* Stage 9: corners   apriltag_detect.cu:98-241 (UpdateFitQuads), :260-282     */
/* ------------------------------------------------------------------------- */
static void quad_corners(const orc_config *c, orc_result *r) {
  r->corners = (orc_quadcorners *)calloc((size_t)r->num_fitquads + 1, sizeof(orc_quadcorners));
  int n = 0;
  const int mtw = min_tag_width(c);
  int normal_border, reversed_border;
  orc_i_border_polarities(c, &normal_border, &reversed_border);
  for (int qi = 0; qi < r->num_fitquads; qi++) {
    const orc_fitquad *q = &r->fitquads[qi];
    if (!q->valid) continue;
    orc_quadcorners qc;
    memset(&qc, 0, sizeof(qc));
    qc.blob = q->blob;
    qc.rep0 = q->rep0;
    qc.rep1 = q->rep1;
    qc.reversed_border = reversed_border && !normal_border; /* one polarity across the families */
    double lines[4][4];
    for (int i = 0; i < 4; i++) {
      double err, mse;
      fit_line(&q->moments[i], lines[i], lines[i] + 2, &err, &mse);
    }
    int bad = 0;
    for (int i = 0; i < 4; i++) { /* :125-166 */
      const double A00 = lines[i][3], A01 = -lines[(i + 1) & 3][3];
      const double A10 = -lines[i][2], A11 = lines[(i + 1) & 3][2];
      const double B0 = -lines[i][0] + lines[(i + 1) & 3][0];
      const double B1 = -lines[i][1] + lines[(i + 1) & 3][1];
      const double det = A00 * A11 - A10 * A01;
      const double W00 = A11 / det, W01 = -A01 / det;
      if (fabs(det) < 0.001) { bad = 1; break; }
      const double L0 = W00 * B0 + W01 * B1;
      qc.corners[i][0] = (float)(lines[i][0] + L0 * A00);
      qc.corners[i][1] = (float)(lines[i][1] + L0 * A10);
    }
    if (bad) continue;
    { /* :171-207 area */
      float area = 0;
      float length[3], p;
      for (int i = 0; i < 3; i++) {
        const int a = i, b = (i + 1) % 3;
        length[i] = orc_cuda_hypotf(qc.corners[b][0] - qc.corners[a][0], qc.corners[b][1] - qc.corners[a][1]);
      }
      p = (length[0] + length[1] + length[2]) / 2;
      area += sqrtf(p * (p - length[0]) * (p - length[1]) * (p - length[2]));
      static const int idxs[4] = {2, 3, 0, 2};
      for (int i = 0; i < 3; i++) {
        const int a = idxs[i], b = idxs[i + 1];
        length[i] = orc_cuda_hypotf(qc.corners[b][0] - qc.corners[a][0], qc.corners[b][1] - qc.corners[a][1]);
      }
      p = (length[0] + length[1] + length[2]) / 2;
      area += sqrtf(p * (p - length[0]) * (p - length[1]) * (p - length[2]));
      if ((double)area < 0.95 * mtw * mtw) continue;
    }
    { /* :209-238 angles + winding */
      int reject = 0;
      for (int i = 0; i < 4; i++) {
        const int i0 = i, i1 = (i + 1) & 3, i2 = (i + 2) & 3;
        const float dx1 = qc.corners[i1][0] - qc.corners[i0][0];
        const float dy1 = qc.corners[i1][1] - qc.corners[i0][1];
        const float dx2 = qc.corners[i2][0] - qc.corners[i1][0];
        const float dy2 = qc.corners[i2][1] - qc.corners[i1][1];
        const float cos_dtheta = (dx1 * dx2 + dy1 * dy2) / sqrtf((dx1 * dx1 + dy1 * dy1) * (dx2 * dx2 + dy2 * dy2));
        if (fabsf(cos_dtheta) > c->cos_critical_rad || dx1 * dy2 < dy1 * dx2) { reject = 1; break; }
      }
      if (reject) continue;
    }
    /* AdjustPixelCenters, :260-282 */
    const float f = (float)c->quad_decimate;
    if (f > 1) {
      for (int j = 0; j < 4; j++) {
        qc.corners[j][0] = (qc.corners[j][0] - 0.5f) * f + 0.5f;
        qc.corners[j][1] = (qc.corners[j][1] - 0.5f) * f + 0.5f;
      }
    }
    r->corners[n++] = qc;
  }
  r->num_corners = n;
}

/* ------------------------------------------------------------------------- */
/* Stage 10: refine edges   apriltag_detect.cu:307-564                         */
/* ------------------------------------------------------------------------- */
void orc_redistort(double *x, double *y, const orc_config *c) { /* :307-331 */
  const double k1 = c->k1, k2 = c->k2, p1 = c->p1, p2 = c->p2, k3 = c->k3;
  const double xP = (*x - c->cx) / c->fx;
  const double yP = (*y - c->cy) / c->fy;
  const double rSq = xP * xP + yP * yP;
  const double linCoef = 1 + k1 * rSq + k2 * rSq * rSq + k3 * rSq * rSq * rSq;
  const double xPP = xP * linCoef + 2 * p1 * xP * yP + p2 * (rSq + 2 * xP * xP);
  const double yPP = yP * linCoef + p1 * (rSq + 2 * yP * yP) + 2 * p2 * xP * yP;
  *x = xPP * c->fx + c->cx;
  *y = yPP * c->fy + c->cy;
}

int orc_undistort(double *u, double *v, const orc_config *c) { /* :335-402 */
  int converged = 1;
  const double k1 = c->k1, k2 = c->k2, p1 = c->p1, p2 = c->p2, k3 = c->k3;
  const double xPP = (*u - c->cx) / c->fx;
  const double yPP = (*v - c->cy) / c->fy;
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
  } while (fabs(xP - prev_x) > 1e-6 || fabs(yP - prev_y) > 1e-6);
  *u = xP * c->fx + c->cx;
  *v = yP * c->fy + c->cy;
  return converged;
}

static void refine_edges(const orc_config *c, const uint8_t *im, int W, int H, float p[4][2], int reversed_border) {
  double lines[4][4];
  for (int edge = 0; edge < 4; edge++) {
    const int a = edge, b = (edge + 1) & 3;
    float nx = p[b][1] - p[a][1];
    float ny = -p[b][0] + p[a][0];
    const float mag = sqrtf(nx * nx + ny * ny);
    nx /= mag;
    ny /= mag;
    if (reversed_border) { nx = -nx; ny = -ny; }
    int nsamples = (int)(mag / 8);
    if (nsamples < 16) nsamples = 16;
    double Mx = 0, My = 0, Mxx = 0, Mxy = 0, Myy = 0, N = 0;
    for (int s = 0; s < nsamples; s++) {
      const double alpha = (1.0 + s) / (nsamples + 1);
      const double x0 = alpha * p[a][0] + (1 - alpha) * p[b][0];
      const double y0 = alpha * p[a][1] + (1 - alpha) * p[b][1];
      double Mn = 0, Mcount = 0;
      const double range = (double)((float)c->quad_decimate) + 1;
      for (double n = -range; n <= range; n += 0.25) {
        const double grange = 1;
        const int x1 = (int)(x0 + (n + grange) * nx);
        const int y1 = (int)(y0 + (n + grange) * ny);
        if (x1 < 0 || x1 >= W || y1 < 0 || y1 >= H) continue;
        const int x2 = (int)(x0 + (n - grange) * nx);
        const int y2 = (int)(y0 + (n - grange) * ny);
        if (x2 < 0 || x2 >= W || y2 < 0 || y2 >= H) continue;
        const int g1 = im[(size_t)y1 * W + x1];
        const int g2 = im[(size_t)y2 * W + x2];
        if (g1 < g2) continue;
        const double weight = (double)((g2 - g1) * (g2 - g1));
        Mn += weight * n;
        Mcount += weight;
      }
      if (Mcount == 0) continue;
      const double n0 = Mn / Mcount;
      double bestx = x0 + n0 * nx;
      double besty = y0 + n0 * ny;
      orc_undistort(&bestx, &besty, c);
      Mx += bestx;
      My += besty;
      Mxx += bestx * bestx;
      Mxy += bestx * besty;
      Myy += besty * besty;
      N++;
    }
    const double Ex = Mx / N, Ey = My / N;
    const double Cxx = Mxx / N - Ex * Ex;
    const double Cxy = Mxy / N - Ex * Ey;
    const double Cyy = Myy / N - Ey * Ey;
    /* :523-525: single-precision libm on the host; the engine uses the device
     * routines, so agreement here is to float rounding, not bit-exact. */
    const double normal_theta = .5 * atan2f((float)(-2 * Cxy), (float)(Cyy - Cxx));
    nx = cosf((float)normal_theta);
    ny = sinf((float)normal_theta);
    lines[edge][0] = Ex;
    lines[edge][1] = Ey;
    lines[edge][2] = nx;
    lines[edge][3] = ny;
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
      double px = lines[i][0] + L0 * A00;
      double py = lines[i][1] + L0 * A10;
      orc_redistort(&px, &py, c);
      p[(i + 1) & 3][0] = (float)px;
      p[(i + 1) & 3][1] = (float)py;
    }
  }
}

/* ------------------------------------------------------------------------- */
/* Stage 11: decode.  quad_decode_index lives in the un-vendored libapriltag   */
/* fork (declared at apriltag_detect.cu:27-29, called at :613).  RECALLED from  */
/* upstream AprilTag 3 apriltag.c: quad_update_homographies, homography_compute2,*/
/* quad_decode, graymodel_*, value_for_pixel, sharpen, quick_decode_codeword,    */
/* rotate90, and the detection construction in quad_decode_task.               */
/* ------------------------------------------------------------------------- */
int orc_homography_compute(const double c[4][4], double Hout[9]) {
  double A[72];
  for (int i = 0; i < 4; i++) {
    double *r0 = &A[(2 * i) * 9], *r1 = &A[(2 * i + 1) * 9];
    r0[0] = c[i][0]; r0[1] = c[i][1]; r0[2] = 1; r0[3] = 0; r0[4] = 0; r0[5] = 0;
    r0[6] = -c[i][0] * c[i][2]; r0[7] = -c[i][1] * c[i][2]; r0[8] = c[i][2];
    r1[0] = 0; r1[1] = 0; r1[2] = 0; r1[3] = c[i][0]; r1[4] = c[i][1]; r1[5] = 1;
    r1[6] = -c[i][0] * c[i][3]; r1[7] = -c[i][1] * c[i][3]; r1[8] = c[i][3];
  }
  const double epsilon = 1e-10;
  for (int col = 0; col < 8; col++) {
    double max_val = 0;
    int max_val_idx = -1;
    for (int row = col; row < 8; row++) {
      const double val = fabs(A[row * 9 + col]);
      if (val > max_val) { max_val = val; max_val_idx = row; }
    }
    if (max_val_idx < 0) return -1;
    if (max_val < epsilon) return -1;
    if (max_val_idx != col) {
      for (int i = col; i < 9; i++) {
        const double tmp = A[col * 9 + i];
        A[col * 9 + i] = A[max_val_idx * 9 + i];
        A[max_val_idx * 9 + i] = tmp;
      }
    }
    for (int i = col + 1; i < 8; i++) {
      const double f = A[i * 9 + col] / A[col * 9 + col];
      A[i * 9 + col] = 0;
      for (int j = col + 1; j < 9; j++) A[i * 9 + j] -= f * A[col * 9 + j];
    }
  }
  for (int col = 7; col >= 0; col--) {
    double sum = 0;
    for (int i = col + 1; i < 8; i++) sum += A[col * 9 + i] * A[i * 9 + 8];
    A[col * 9 + 8] = (A[col * 9 + 8] - sum) / A[col * 9 + col];
  }
  for (int i = 0; i < 8; i++) Hout[i] = A[i * 9 + 8];
  Hout[8] = 1;
  return 0;
}

void orc_i_h_project(const double *H, double x, double y, double *ox, double *oy);
static void h_project(const double *H, double x, double y, double *ox, double *oy) { orc_i_h_project(H, x, y, ox, oy); }
void orc_i_h_project(const double *H, double x, double y, double *ox, double *oy) {
  const double xx = H[0] * x + H[1] * y + H[2];
  const double yy = H[3] * x + H[4] * y + H[5];
  const double zz = H[6] * x + H[7] * y + H[8];
  *ox = xx / zz;
  *oy = yy / zz;
}

typedef struct {
  double A[3][3], B[3], C[3];
} graymodel;
static void gm_add(graymodel *g, double x, double y, double gray) {
  g->A[0][0] += x * x; g->A[0][1] += x * y; g->A[0][2] += x;
  g->A[1][1] += y * y; g->A[1][2] += y; g->A[2][2] += 1;
  g->B[0] += x * gray; g->B[1] += y * gray; g->B[2] += gray;
}
static void gm_solve(graymodel *g) { /* mat33_sym_solve: chol + lower-tri inverse */
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
static double gm_interp(const graymodel *g, double x, double y) { return g->C[0] * x + g->C[1] * y + g->C[2]; }

static double value_for_pixel(const uint8_t *im, int W, int H, double px, double py) {
  const int x1 = (int)floor(px - 0.5);
  const int x2 = (int)ceil(px - 0.5);
  const double x = px - 0.5 - x1;
  const int y1 = (int)floor(py - 0.5);
  const int y2 = (int)ceil(py - 0.5);
  const double y = py - 0.5 - y1;
  if (x1 < 0 || x2 >= W || y1 < 0 || y2 >= H) return -1;
  return im[(size_t)y1 * W + x1] * (1 - x) * (1 - y) + im[(size_t)y1 * W + x2] * x * (1 - y) +
         im[(size_t)y2 * W + x1] * (1 - x) * y + im[(size_t)y2 * W + x2] * x * y;
}

/* rotate90 (libapriltag apriltag.c): the codeword of the tag turned by 90 degrees */
static uint64_t rotate90(uint64_t w, int nbits) {
  int p = nbits;
  uint64_t l = 0;
  if (nbits % 4 == 1) {
    p = nbits - 1;
    l = 1;
  }
  w = ((w >> l) << (p / 4 + l)) | (w >> (3 * p / 4 + l) << l) | (w & l);
  w &= ((1ULL << nbits) - 1);
  return w;
}

int orc_decode_codeword_family(const orc_family *fam, uint64_t rcode, int *hamming, int *rotation) {
  /* quick_decode_codeword: the first rotation with a code within max_hamming bits, and at that rotation the lowest
   * id within reach.  The hit need not be unique: tag16h5 (minimum distance 5) at max_hamming 3 has words within 3
   * bits of two codes.  libapriltag's hash table answers with the lowest id there too: quick_decode_init inserts the
   * codes in id order, each with every word within max_hamming bits, and an insert only takes an empty slot, so on a
   * word's probe chain the lowest id's entry comes first and the lookup returns it. */
  for (int ridx = 0; ridx < 4; ridx++) {
    for (int id = 0; id < fam->ncodes; id++) {
      const int d = __builtin_popcountll(rcode ^ fam->codes[id]);
      if (d <= fam->max_hamming) {
        *hamming = d;
        *rotation = ridx;
        return id;
      }
    }
    rcode = rotate90(rcode, fam->nbits);
  }
  *hamming = 255;
  *rotation = 0;
  return -1;
}
int orc_decode_codeword(uint64_t rcode, int *hamming, int *rotation) {
  return orc_decode_codeword_family(&k_families[0], rcode, hamming, rotation);
}

/* returns decision margin (<0: rejected) */
float orc_i_quad_decode(const orc_config *c, const orc_family *fam, const uint8_t *im, int W, int H, const double *Hm, int *id,
                        int *hamming, int *rotation) {
  const int wb = fam->width_at_border, tw = fam->total_width;
  const float patterns[] = {
      -0.5f, 0.5f, 0, 1, 1, 0.5f, 0.5f, 0, 1, 0, wb + 0.5f, .5f, 0, 1, 1, wb - 0.5f, .5f, 0, 1, 0,
      0.5f, -0.5f, 1, 0, 1, 0.5f, 0.5f, 1, 0, 0, 0.5f, wb + 0.5f, 1, 0, 1, 0.5f, wb - 0.5f, 1, 0, 0};
  graymodel whitemodel, blackmodel;
  memset(&whitemodel, 0, sizeof(whitemodel));
  memset(&blackmodel, 0, sizeof(blackmodel));
  for (int pi = 0; pi < 8; pi++) {
    const float *pat = &patterns[pi * 5];
    const int is_white = (int)pat[4];
    for (int i = 0; i < wb; i++) {
      const double tagx01 = (pat[0] + i * pat[2]) / (wb);
      const double tagy01 = (pat[1] + i * pat[3]) / (wb);
      const double tagx = 2 * (tagx01 - 0.5);
      const double tagy = 2 * (tagy01 - 0.5);
      double px, py;
      h_project(Hm, tagx, tagy, &px, &py);
      const int ix = (int)px, iy = (int)py;
      if (ix < 0 || iy < 0 || ix >= W || iy >= H) continue;
      const int v = im[(size_t)iy * W + ix];
      if (is_white) gm_add(&whitemodel, tagx, tagy, v);
      else gm_add(&blackmodel, tagx, tagy, v);
    }
  }
  gm_solve(&whitemodel);
  gm_solve(&blackmodel);
  if ((gm_interp(&whitemodel, 0, 0) - gm_interp(&blackmodel, 0, 0) < 0) != fam->reversed_border) return -1;

  float black_score = 0, white_score = 0;
  float black_score_count = 1, white_score_count = 1;
  double values[144];
  memset(values, 0, sizeof(values));
  const int min_coord = (wb - tw) / 2;
  for (int i = 0; i < fam->nbits; i++) {
    const int bit_x = fam->bit_x[i], bit_y = fam->bit_y[i];
    const double tagx01 = (bit_x + 0.5) / (wb);
    const double tagy01 = (bit_y + 0.5) / (wb);
    const double tagx = 2 * (tagx01 - 0.5);
    const double tagy = 2 * (tagy01 - 0.5);
    double px, py;
    h_project(Hm, tagx, tagy, &px, &py);
    const double v = value_for_pixel(im, W, H, px, py);
    if (v == -1) continue;
    const double thresh = (gm_interp(&blackmodel, tagx, tagy) + gm_interp(&whitemodel, tagx, tagy)) / 2.0;
    values[tw * (bit_y - min_coord) + bit_x - min_coord] = v - thresh;
  }
  { /* sharpen */
    double sharpened[144];
    static const double kernel[9] = {0, -1, 0, -1, 4, -1, 0, -1, 0};
    for (int y = 0; y < tw; y++)
      for (int x = 0; x < tw; x++) {
        sharpened[y * tw + x] = 0;
        for (int i = 0; i < 3; i++)
          for (int j = 0; j < 3; j++) {
            if ((y + i - 1) < 0 || (y + i - 1) > tw - 1 || (x + j - 1) < 0 || (x + j - 1) > tw - 1) continue;
            sharpened[y * tw + x] += values[(y + i - 1) * tw + (x + j - 1)] * kernel[i * 3 + j];
          }
      }
    for (int i = 0; i < tw * tw; i++) values[i] = values[i] + c->decode_sharpening * sharpened[i];
  }
  uint64_t rcode = 0;
  for (int i = 0; i < fam->nbits; i++) {
    const int bit_x = fam->bit_x[i], bit_y = fam->bit_y[i];
    rcode = (rcode << 1);
    const double v = values[(bit_y - min_coord) * tw + bit_x - min_coord];
    if (v > 0) {
      white_score += (float)v;
      white_score_count++;
      rcode |= 1;
    } else {
      black_score -= (float)v;
      black_score_count++;
    }
  }
  *id = orc_decode_codeword_family(fam, rcode, hamming, rotation);
  return fminf(white_score / white_score_count, black_score / black_score_count);
}

/* the apriltag_detection_t quad_decode_task builds from a decoded quad (libapriltag apriltag.c, RECALLED) */
void orc_i_fill_detection(orc_detection *d, int family, int id, int hamming, float margin, int rotation, const double *Hm) {
  /* cos/sin(rotation * M_PI / 2.0) as libm returns them for k = 0..3 */
  static const double kc[4] = {1.0, 6.123233995736766e-17, -1.0, -1.8369701987210297e-16};
  static const double ks[4] = {0.0, 1.0, 1.2246467991473532e-16, -1.0};
  memset(d, 0, sizeof(*d));
  d->id = id;
  d->hamming = hamming;
  d->decision_margin = margin;
  d->rotation = rotation;
  d->family = family;
  const double cc = kc[rotation], ss = ks[rotation];
  /* H * R, R = [c -s 0; s c 0; 0 0 1] */
  for (int row = 0; row < 3; row++) {
    d->H[row * 3 + 0] = Hm[row * 3 + 0] * cc + Hm[row * 3 + 1] * ss;
    d->H[row * 3 + 1] = Hm[row * 3 + 0] * -ss + Hm[row * 3 + 1] * cc;
    d->H[row * 3 + 2] = Hm[row * 3 + 2];
  }
  h_project(d->H, 0, 0, &d->c[0], &d->c[1]);
  for (int i = 0; i < 4; i++) {
    const int tcx = (i == 1 || i == 2) ? 1 : -1;
    const int tcy = (i < 2) ? 1 : -1;
    h_project(d->H, tcx, tcy, &d->p[i][0], &d->p[i][1]);
  }
}

static void decode_quads(const orc_config *c, orc_result *r) {
  r->detections = (orc_detection *)calloc((size_t)r->num_corners * orc_i_family_slots(c) + 1, sizeof(orc_detection));
  r->refined = (orc_quadcorners *)calloc((size_t)r->num_corners + 1, sizeof(orc_quadcorners));
  int nd = 0;
  for (int qi = 0; qi < r->num_corners; qi++) {
    float p[4][2];
    memcpy(p, r->corners[qi].corners, sizeof(p));
    if (c->refine_edges) refine_edges(c, r->gray, r->W, r->H, p, r->corners[qi].reversed_border);
    r->refined[qi] = r->corners[qi]; /* the quad as handed to quad_decode_index, apriltag_detect.cu:613 */
    memcpy(r->refined[qi].corners, p, sizeof(p));
    double corr[4][4];
    for (int i = 0; i < 4; i++) {
      corr[i][0] = (i == 0 || i == 3) ? -1 : 1;
      corr[i][1] = (i == 0 || i == 1) ? -1 : 1;
      corr[i][2] = p[i][0];
      corr[i][3] = p[i][1];
    }
    double Hm[9];
    if (orc_homography_compute(corr, Hm) != 0) continue;
    { /* quad_update_homographies also needs H to be invertible (matd_inverse) */
      const double det = Hm[0] * (Hm[4] * Hm[8] - Hm[5] * Hm[7]) - Hm[1] * (Hm[3] * Hm[8] - Hm[5] * Hm[6]) +
                         Hm[2] * (Hm[3] * Hm[7] - Hm[4] * Hm[6]);
      if (!(fabs(det) > 1e-300)) continue;
    }
    for (int fi = 0; fi < orc_i_family_slots(c); fi++) { /* quad_decode_task: every family of the matching polarity */
      const orc_family *fam = orc_i_family(c, fi);
      if (!fam || (fam->reversed_border != 0) != (r->corners[qi].reversed_border != 0)) continue;
      int id, hamming, rotation;
      const float margin = orc_i_quad_decode(c, fam, r->gray, r->W, r->H, Hm, &id, &hamming, &rotation);
      if (margin >= 0 && hamming < 255) {
        orc_detection *d = &r->detections[nd++];
        orc_i_fill_detection(d, fi, id, hamming, margin, rotation, Hm);
        d->rep0 = r->corners[qi].rep0;
        d->rep1 = r->corners[qi].rep1;
      }
    }
  }
  r->num_detections = nd;
}

/* ------------------------------------------------------------------------- */
/* Stage 12: reconcile + sort   reconcile_detections (libapriltag, RECALLED),  */
/* apriltag_detect.cu:284-288,660-662                                          */
/* ------------------------------------------------------------------------- */
static int seg_intersect(const double *a0, const double *a1, const double *b0, const double *b1) {
  const double d1x = a1[0] - a0[0], d1y = a1[1] - a0[1];
  const double d2x = b1[0] - b0[0], d2y = b1[1] - b0[1];
  const double den = d1x * d2y - d1y * d2x;
  if (den == 0) return 0;
  const double t = ((b0[0] - a0[0]) * d2y - (b0[1] - a0[1]) * d2x) / den;
  const double u = ((b0[0] - a0[0]) * d1y - (b0[1] - a0[1]) * d1x) / den;
  return t >= 0 && t <= 1 && u >= 0 && u <= 1;
}
static int poly_contains(const double p[4][2], const double *q) {
  int c = 0;
  for (int i = 0, j = 3; i < 4; j = i++) {
    if (((p[i][1] > q[1]) != (p[j][1] > q[1])) &&
        (q[0] < (p[j][0] - p[i][0]) * (q[1] - p[i][1]) / (p[j][1] - p[i][1]) + p[i][0]))
      c = !c;
  }
  return c;
}
static int polys_overlap(const double a[4][2], const double b[4][2]) {
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++)
      if (seg_intersect(a[i], a[(i + 1) & 3], b[j], b[(j + 1) & 3])) return 1;
  double ca[2] = {0, 0}, cb[2] = {0, 0};
  for (int i = 0; i < 4; i++) {
    ca[0] += a[i][0] / 4; ca[1] += a[i][1] / 4;
    cb[0] += b[i][0] / 4; cb[1] += b[i][1] / 4;
  }
  return poly_contains(a, cb) || poly_contains(b, ca);
}
static int prefer_smaller(int pref, double q0, double q1) {
  if (pref) return pref;
  if (q0 < q1) return -1;
  if (q1 < q0) return 1;
  return 0;
}
static int cmp_det(const void *a_, const void *b_) {
  const orc_detection *a = (const orc_detection *)a_, *b = (const orc_detection *)b_;
  if (a->id != b->id) return a->id - b->id;
  if (a->c[0] != b->c[0]) return a->c[0] < b->c[0] ? -1 : 1;
  if (a->c[1] != b->c[1]) return a->c[1] < b->c[1] ? -1 : 1;
  return a->family - b->family;
}
int orc_i_reconcile(orc_detection *d, int n) {
  for (int i0 = 0; i0 < n; i0++) {
    for (int i1 = i0 + 1; i1 < n; i1++) {
      if (d[i0].id != d[i1].id || d[i0].family != d[i1].family) continue;
      if (!polys_overlap(d[i0].p, d[i1].p)) continue;
      int pref = 0;
      pref = prefer_smaller(pref, d[i0].hamming, d[i1].hamming);
      pref = prefer_smaller(pref, -d[i0].decision_margin, -d[i1].decision_margin);
      for (int i = 0; i < 4; i++) {
        pref = prefer_smaller(pref, d[i0].p[i][0], d[i1].p[i][0]);
        pref = prefer_smaller(pref, d[i0].p[i][1], d[i1].p[i][1]);
      }
      if (pref < 0) {
        d[i1] = d[n - 1];
        n--;
        i1--;
      } else {
        d[i0] = d[n - 1];
        n--;
        i0--;
        break;
      }
    }
  }
  qsort(d, n, sizeof(orc_detection), cmp_det);
  return n;
}
static void reconcile(orc_result *r) { r->num_detections = orc_i_reconcile(r->detections, r->num_detections); }

/* ------------------------------------------------------------------------- */
orc_result *orc_detect(const orc_config *c, const uint8_t *image) {
  const int f = c->quad_decimate;
  if (f < 1 || c->width <= 0 || c->height <= 0) return NULL;
  if (c->width % f || c->height % f) return NULL;
  const int w = c->width / f, h = c->height / f;
  if (w % 4 || h % 4 || w < 8 || h < 8) return NULL; /* threshold.cu:156-157 in quad-image terms */
  if (c->max_nmaxima != 10) return NULL;             /* line_fit_filter.cu:1205 */
  orc_result *r = (orc_result *)calloc(1, sizeof(orc_result));
  r->W = c->width; r->H = c->height; r->w = w; r->h = h;
  const size_t N = (size_t)r->W * r->H, n = (size_t)w * h;
  r->gray = (uint8_t *)malloc(N);
  r->quad_im = (uint8_t *)malloc(n);
  r->minmax = (uint8_t *)malloc((size_t)(w / 4) * (h / 4) * 2);
  r->thresh = (uint8_t *)malloc(n);
  orc_i_to_gray(c, image, r->gray);
  orc_i_decimate(r->gray, r->W, f, r->quad_im, w, h);
  if (c->quad_sigma != 0) orc_i_gaussian_blur(r->quad_im, w, h, c->quad_sigma);
  orc_i_threshold(r->quad_im, w, h, c->min_white_black_diff, r->minmax, r->thresh);
  if (c->max_stage <= ORC_STAGE_THRESHOLD) return r;
  r->labels = (uint32_t *)malloc(n * sizeof(uint32_t));
  r->sizes = (uint32_t *)malloc(n * sizeof(uint32_t));
  label_components(r->thresh, w, h, r->labels, r->sizes);
  if (c->max_stage <= ORC_STAGE_LABELS) return r;
  boundary_points(r);
  if (c->max_stage <= ORC_STAGE_POINTS) return r;
  clusters_and_filter(c, r);
  sort_and_moments(r);
  if (c->max_stage <= ORC_STAGE_BLOBS) return r;
  errors_and_peaks(r);
  if (c->max_stage <= ORC_STAGE_LINEFIT) return r;
  fit_quads(c, r);
  quad_corners(c, r);
  if (c->max_stage <= ORC_STAGE_QUADS) return r;
  decode_quads(c, r);
  reconcile(r);
  return r;
}

void orc_free_result(orc_result *r) {
  if (!r) return;
  free(r->gray); free(r->quad_im); free(r->minmax); free(r->thresh); free(r->labels); free(r->sizes);
  free(r->points); free(r->clusters); free(r->spoints); free(r->lfps); free(r->errs); free(r->filtered_errs);
  free(r->is_peak); free(r->fitquads); free(r->corners); free(r->detections); free(r->refined);
  free(r);
}
