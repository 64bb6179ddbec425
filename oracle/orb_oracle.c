/*
 * orb_oracle.c -- CPU restatement (plain C) of the reference's per-frame ORB front-end.
 *
 * TEST INFRASTRUCTURE ONLY (see orb_oracle.h).  Build with -O2 -ffp-contract=off (the reference is built
 * Release for plain x86-64, i.e. SSE2 and no FMA contraction).
 *
 * Each function cites the reference lines it follows, relative to /root/reference/src/ORB_SLAM2/.
 * The OpenCV primitives (un-vendored dependency; README asks for OpenCV 4.2, goldens are cv2 4.13.0)
 * restate OpenCV's published fixed-point algorithms and are pinned against cv2 in tests/.
 */
#include "orb_oracle.h"

#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* cvRound: SSE cvtss2si / cvtsd2si == round-half-to-even in the default rounding mode */
static inline int cv_round_f(float v) { return (int)lrintf(v); }
static inline int cv_round_d(double v) { return (int)lrint(v); }
static inline int cv_floor_f(float v) {
  int i = (int)v;
  return i - (i > v);
}
static inline int cv_floor_d(double v) {
  int i = (int)v;
  return i - (i > v);
}
static inline int cv_ceil_d(double v) {
  int i = (int)v;
  return i + (i < v);
}
static inline int cv_ceil_f(float v) {
  int i = (int)v;
  return i + (i < v);
}
static inline int imin(int a, int b) { return a < b ? a : b; }
static inline int imax(int a, int b) { return a > b ? a : b; }

/* ------------------------------------------------------------------------------------------------ */
/* src/ORBExtractor.cc:283-289: mvfScaledFactors.push_back(std::pow(scaleFactor, level)) (float^int -> double) */
void oracle_scale_factors(float scale_factor, int n_levels, float *sf) {
  for (int l = 0; l < n_levels; ++l) sf[l] = (float)pow((double)scale_factor, (double)l);
}

/* src/ORBExtractor.cc:291-301 */
void oracle_level_quotas(int n_features, float scale_factor, int n_levels, int *quota) {
  float scale = 1.0f / scale_factor;
  int sum = 0;
  /* int*float -> float, divided by a double */
  int nfeats = cv_round_d((double)((float)n_features * (1 - scale)) / (1 - pow((double)scale, (double)n_levels)));
  for (int l = 0; l < n_levels - 1; ++l) {
    quota[l] = nfeats;
    sum += nfeats;
    nfeats = cv_round_f((float)nfeats * scale);
  }
  quota[n_levels - 1] = imax(0, n_features - sum);
}

/* src/ORBExtractor.cc:305-317 */
int oracle_level_sizes(int width, int height, const float *sf, int n_levels, int *lw, int *lh) {
  lw[0] = width;
  lh[0] = height;
  for (int i = 1; i < n_levels; ++i) {
    lw[i] = cv_round_f((float)width / sf[i]);
    lh[i] = cv_round_f((float)height / sf[i]);
    if (lw[i] < 2 * 19 || lh[i] < 2 * 19) return -1;
  }
  return 0;
}

/* src/ORBExtractor.cc:217-236 */
void oracle_umax(int *umax) {
  const int R = 15;
  int v, v0;
  int vmax = cv_floor_f((float)R * sqrtf(2.f) / 2 + 1);
  int vmin = cv_ceil_d((double)((float)R * sqrtf(2.f) / 2));
  const double hp2 = R * R;
  for (v = 0; v <= vmax; ++v) umax[v] = cv_round_d(sqrt(hp2 - v * v));
  for (v = R, v0 = 0; v >= vmin; --v) {
    while (umax[v0] == umax[v0 + 1]) ++v0;
    umax[v] = v0;
    ++v0;
  }
}

/* ------------------------------------------------------------------------------------------------ */
/* cv::resize INTER_LINEAR 8UC1 (call site src/ORBExtractor.cc:316).  OpenCV imgproc/resize.cpp: coefficient
 * tables with 11-bit fixed point (INTER_RESIZE_COEF_SCALE = 2048), HResizeLinear into int32, VResizeLinear
 * ((b0*(S0>>4))>>16 + (b1*(S1>>4))>>16 + 2) >> 2.  An exact 2x2 decimation is re-routed to INTER_AREA. */
static short sat_s16(int v) { return (short)(v < -32768 ? -32768 : (v > 32767 ? 32767 : v)); }

void oracle_resize_linear_u8(const uint8_t *src, int sw, int sh, size_t sstride, uint8_t *dst, int dw, int dh,
                             size_t dstride) {
  if (dw == sw && dh == sh) {
    for (int y = 0; y < dh; ++y) memcpy(dst + (size_t)y * dstride, src + (size_t)y * sstride, (size_t)dw);
    return;
  }
  if (dw * 2 == sw && dh * 2 == sh) { /* INTER_LINEAR with iscale 2x2 -> INTER_AREA fast path */
    for (int y = 0; y < dh; ++y) {
      const uint8_t *s0 = src + (size_t)(2 * y) * sstride, *s1 = s0 + sstride;
      for (int x = 0; x < dw; ++x)
        dst[(size_t)y * dstride + x] = (uint8_t)((s0[2 * x] + s0[2 * x + 1] + s1[2 * x] + s1[2 * x + 1] + 2) >> 2);
    }
    return;
  }
  double inv_scale_x = (double)dw / sw, inv_scale_y = (double)dh / sh;
  double scale_x = 1. / inv_scale_x, scale_y = 1. / inv_scale_y;
  int *xofs = (int *)malloc(sizeof(int) * (size_t)dw);
  short *ialpha = (short *)malloc(sizeof(short) * 2 * (size_t)dw);
  int *row0 = (int *)malloc(sizeof(int) * (size_t)dw), *row1 = (int *)malloc(sizeof(int) * (size_t)dw);
  for (int dx = 0; dx < dw; ++dx) {
    float fx = (float)((dx + 0.5) * scale_x - 0.5);
    int sx = cv_floor_f(fx);
    fx -= sx;
    if (sx < 0) {
      fx = 0;
      sx = 0;
    }
    if (sx >= sw - 1) {
      fx = 0;
      sx = sw - 1;
    }
    xofs[dx] = sx;
    ialpha[2 * dx] = sat_s16(cv_round_f((1.f - fx) * 2048.f));
    ialpha[2 * dx + 1] = sat_s16(cv_round_f(fx * 2048.f));
  }
  for (int dy = 0; dy < dh; ++dy) {
    float fy = (float)((dy + 0.5) * scale_y - 0.5);
    int sy = cv_floor_f(fy);
    fy -= sy;
    short b0 = sat_s16(cv_round_f((1.f - fy) * 2048.f)), b1 = sat_s16(cv_round_f(fy * 2048.f));
    int y0 = imin(imax(sy, 0), sh - 1), y1 = imin(imax(sy + 1, 0), sh - 1); /* rows are clamped, not re-weighted */
    const uint8_t *s0 = src + (size_t)y0 * sstride, *s1 = src + (size_t)y1 * sstride;
    for (int dx = 0; dx < dw; ++dx) {
      int sx = xofs[dx], sx1 = imin(sx + 1, sw - 1);
      int a0 = ialpha[2 * dx], a1 = ialpha[2 * dx + 1];
      row0[dx] = s0[sx] * a0 + s0[sx1] * a1;
      row1[dx] = s1[sx] * a0 + s1[sx1] * a1;
    }
    uint8_t *d = dst + (size_t)dy * dstride;
    for (int dx = 0; dx < dw; ++dx) {
      int v = (((b0 * (row0[dx] >> 4)) >> 16) + ((b1 * (row1[dx] >> 4)) >> 16) + 2) >> 2;
      d[dx] = (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
    }
  }
  free(xofs);
  free(ialpha);
  free(row0);
  free(row1);
}

/* cv::GaussianBlur 7x7 sigma 2, 8UC1, REFLECT_101 (call site src/ORBExtractor.cc:319).  OpenCV's fixed-point
 * path: 8.8 kernel {18,34,48,56,48,34,18} (sum 256), horizontal pass into u16, vertical into u32, round >>16. */
static inline int refl101(int i, int n) {
  if (n == 1) return 0;
  while (i < 0 || i >= n) {
    if (i < 0) i = -i;
    if (i >= n) i = 2 * (n - 1) - i;
  }
  return i;
}

void oracle_gaussian_blur7_u8(const uint8_t *src, int w, int h, size_t sstride, uint8_t *dst, size_t dstride) {
  static const uint32_t k[7] = {18, 34, 48, 56, 48, 34, 18};
  uint16_t *tmp = (uint16_t *)malloc(sizeof(uint16_t) * (size_t)w * (size_t)h);
  for (int y = 0; y < h; ++y) {
    const uint8_t *s = src + (size_t)y * sstride;
    for (int x = 0; x < w; ++x) {
      uint32_t acc = 0;
      for (int i = 0; i < 7; ++i) acc += s[refl101(x + i - 3, w)] * k[i];
      tmp[(size_t)y * w + x] = (uint16_t)acc;
    }
  }
  for (int y = 0; y < h; ++y) {
    const uint16_t *r[7];
    for (int j = 0; j < 7; ++j) r[j] = tmp + (size_t)refl101(y + j - 3, h) * w;
    uint8_t *d = dst + (size_t)y * dstride;
    for (int x = 0; x < w; ++x) {
      uint32_t acc = 0;
      for (int j = 0; j < 7; ++j) acc += (uint32_t)r[j][x] * k[j];
      d[x] = (uint8_t)((acc + 32768u) >> 16);
    }
  }
  free(tmp);
}

/* cv::FAST TYPE_9_16 (call sites src/ORBExtractor.cc:365,367). Bresenham ring of radius 3, clockwise from (0,3). */
static const int ring_dx[16] = {0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1};
static const int ring_dy[16] = {3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3};

int oracle_fast9_arc_value(const uint8_t *p, size_t stride) {
  int d[16];
  int v = p[0];
  for (int k = 0; k < 16; ++k) d[k] = v - p[(ptrdiff_t)ring_dy[k] * (ptrdiff_t)stride + ring_dx[k]];
  int best = -256;
  for (int s = 0; s < 16; ++s) {
    int mn = 256, mx = -256;
    for (int i = 0; i < 9; ++i) {
      int q = d[(s + i) & 15];
      if (q < mn) mn = q;
      if (q > mx) mx = q;
    }
    /* all nine darker than centre by mn, or all nine brighter by -mx */
    if (mn > best) best = mn;
    if (-mx > best) best = -mx;
  }
  return best;
}

int oracle_fast9_nms(const uint8_t *img, int w, int h, size_t stride, int threshold, int *xs, int *ys, int *scores,
                     int cap) {
  if (w < 7 || h < 7) return 0;
  /* score map: cornerScore (= m - 1) at detected corners, 0 elsewhere, only inside [3,w-3) x [3,h-3) */
  uint8_t *sc = (uint8_t *)calloc((size_t)w * (size_t)h, 1);
  for (int y = 3; y < h - 3; ++y)
    for (int x = 3; x < w - 3; ++x) {
      const uint8_t *p = img + (size_t)y * stride + x;
      /* cheap exact pre-test (as cv::FAST does): any arc of 9 contains at least 2 of the 4 compass pixels */
      int v = p[0], hi = v + threshold, lo = v - threshold;
      int a = p[3 * (ptrdiff_t)stride], b = p[3], c = p[-3 * (ptrdiff_t)stride], d = p[-3];
      if ((a > hi) + (b > hi) + (c > hi) + (d > hi) < 2 && (a < lo) + (b < lo) + (c < lo) + (d < lo) < 2) continue;
      int m = oracle_fast9_arc_value(p, stride);
      if (m > threshold) sc[(size_t)y * w + x] = (uint8_t)(m - 1);
    }
  int n = 0;
  for (int y = 3; y < h - 3; ++y)
    for (int x = 3; x < w - 3; ++x) {
      int s = sc[(size_t)y * w + x];
      if (!s) {
        /* a detected corner always has score >= threshold >= 0; score 0 can only arise at threshold 0 (m == 1),
         * where it can never beat its neighbours strictly unless they are ... also 0: strict '>' fails. */
        continue;
      }
      const uint8_t *c = sc + (size_t)y * w + x;
      if (s > c[-1] && s > c[1] && s > c[-w - 1] && s > c[-w] && s > c[-w + 1] && s > c[w - 1] && s > c[w] &&
          s > c[w + 1]) {
        if (n < cap) {
          xs[n] = x;
          ys[n] = y;
          scores[n] = s;
        }
        ++n;
      }
    }
  free(sc);
  return n;
}

/* cv::undistortPoints with P = K (call site src/Camera.cc:36): 5 fixed-point iterations, double, no early exit */
void oracle_undistort_points(float *xy, int n, float fx_, float fy_, float cx_, float cy_, const float *dist,
                             int n_dist) {
  double fx = fx_, fy = fy_, cx = cx_, cy = cy_;
  double k1 = n_dist > 0 ? dist[0] : 0, k2 = n_dist > 1 ? dist[1] : 0, p1 = n_dist > 2 ? dist[2] : 0,
         p2 = n_dist > 3 ? dist[3] : 0, k3 = n_dist > 4 ? dist[4] : 0;
  double ifx = 1. / fx, ify = 1. / fy;
  for (int i = 0; i < n; ++i) {
    double x = ((double)xy[2 * i] - cx) * ifx, y = ((double)xy[2 * i + 1] - cy) * ify;
    double x0 = x, y0 = y;
    for (int it = 0; it < 5; ++it) {
      double r2 = x * x + y * y;
      double icdist = 1. / (1 + ((k3 * r2 + k2) * r2 + k1) * r2);
      double dx = 2 * p1 * x * y + p2 * (r2 + 2 * x * x);
      double dy = p1 * (r2 + 2 * y * y) + 2 * p2 * x * y;
      x = (x0 - dx) * icdist;
      y = (y0 - dy) * icdist;
    }
    xy[2 * i] = (float)(x * fx + cx);
    xy[2 * i + 1] = (float)(y * fy + cy);
  }
}

/* ------------------------------------------------------------------------------------------------ */
/* src/ORBExtractor.cc:331-375 */
int oracle_fast_cells(const uint8_t *img, int w_img, int h_img, size_t stride, int ini_th, int min_th, int *xs,
                      int *ys, int *scores, int cap, int *n_fallback_cells) {
  const int border = 19;
  int maxBX = w_img - border + 3, maxBY = h_img - border + 3, minBX = border - 3, minBY = border - 3;
  int w = maxBX - minBX, h = maxBY - minBY;
  int nCols = w / 30, nRows = h / 30;
  if (nCols <= 0 || nRows <= 0) return -1; /* the reference divides by zero here */
  int wCell = w / nCols, hCell = h / nRows; /* ceil() of an integer quotient is a no-op (:342-343) */
  int cell_cap = 64 * 64;
  int *cx = (int *)malloc(sizeof(int) * 3 * (size_t)cell_cap), *cy = cx + cell_cap, *cs = cy + cell_cap;
  int n = 0, nfb = 0;
  for (int i = 0; i < nRows; ++i) {
    int iniY = minBY + i * hCell, maxY = iniY + hCell + 6;
    if (iniY >= maxBY - 6) continue;
    if (maxY > maxBY) maxY = maxBY;
    for (int j = 0; j < nCols; ++j) {
      int iniX = minBX + j * wCell, maxX = iniX + wCell + 6;
      if (iniX >= maxBX - 6) continue;
      if (maxX > maxBX) maxX = maxBX;
      const uint8_t *patch = img + (size_t)iniY * stride + iniX;
      int c = oracle_fast9_nms(patch, maxX - iniX, maxY - iniY, stride, ini_th, cx, cy, cs, cell_cap);
      if (c == 0) {
        c = oracle_fast9_nms(patch, maxX - iniX, maxY - iniY, stride, min_th, cx, cy, cs, cell_cap);
        ++nfb;
      }
      for (int k = 0; k < c; ++k) {
        if (n < cap) {
          xs[n] = cx[k] + j * wCell;
          ys[n] = cy[k] + i * hCell;
          scores[n] = cs[k];
        }
        ++n;
      }
    }
  }
  free(cx);
  if (n_fallback_cells) *n_fallback_cells = nfb;
  return n;
}

/* ------------------------------------------------------------------------------------------------ */
/* src/ORBExtractor.cc:19-192 + include/ORB_SLAM2/ORBExtractor.h:55-62.  The multimap<count, node, greater> is
 * restated as a flat list of live nodes ordered by (count desc, insertion sequence asc). */
typedef struct qnode {
  double r0, r1, c0, c1;
  int *idx;
  int n;
  long seq;
  int is_root;
} qnode;

static int q_is_in(const qnode *nd, float x, float y) { /* ORBExtractor.h:55-62, strict */
  return ((double)x > nd->c0 && (double)x < nd->c1 && (double)y > nd->r0 && (double)y < nd->r1);
}

static void q_child(const qnode *parent, double r0, double r1, double c0, double c1, const float *xs,
                    const float *ys, qnode *out) { /* :39-53 */
  out->r0 = r0;
  out->r1 = r1;
  out->c0 = c0;
  out->c1 = c1;
  out->is_root = 0;
  out->n = 0;
  out->idx = (int *)malloc(sizeof(int) * (size_t)(parent->n > 0 ? parent->n : 1));
  for (int k = 0; k < parent->n; ++k) {
    int id = parent->idx[k];
    if (q_is_in(out, xs[id], ys[id])) out->idx[out->n++] = id;
  }
}

int oracle_quadtree_select(int roi_w, int roi_h, int n, const float *xs, const float *ys, const float *resp,
                           int need_i, int *out_idx, long *n_pops) {
  unsigned need = (unsigned)need_i;
  size_t live_cap = (size_t)need_i + 16, n_live = 0;
  qnode *live = (qnode *)malloc(sizeof(qnode) * live_cap);
  long seq = 0, pops = 0;
  qnode root;
  root.r0 = 0;
  root.r1 = roi_h;
  root.c0 = 0;
  root.c1 = roi_w;
  root.n = n;
  root.is_root = 1;
  root.seq = seq++;
  root.idx = (int *)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
  for (int i = 0; i < n; ++i) root.idx[i] = i; /* :26-27, no filtering for the root */
  live[n_live++] = root;
  unsigned n_nodes = 1;
  while (n_nodes < need && n_live > 0) { /* :151 */
    size_t best = 0;
    for (size_t i = 1; i < n_live; ++i)
      if (live[i].n > live[best].n || (live[i].n == live[best].n && live[i].seq < live[best].seq)) best = i;
    qnode cur = live[best];
    live[best] = live[--n_live];
    ++pops;
    qnode kids[64];
    int n_kids = 0;
    if (cur.is_root) { /* initSplit :81-96 */
      const double w = cur.c1, h = cur.r1;
      const int nIni = (int)round(w / h);
      const float hX = (float)((double)w / nIni);
      double cols[66];
      int nc = 0;
      cols[nc++] = cur.c0;
      for (size_t k = 1; k < (size_t)(nIni > 0 ? nIni : 0) && nc < 64; ++k) cols[nc++] = (double)((float)k * hX);
      cols[nc++] = cur.c1;
      for (int i = 0; i < nIni && i < 63; ++i) q_child(&cur, cur.r0, cur.r1, cols[i], cols[i + 1], xs, ys, &kids[n_kids++]);
    } else { /* split :60-72 */
      double rows[3] = {cur.r0, (cur.r0 + cur.r1) / 2, cur.r1};
      double cols[3] = {cur.c0, (cur.c0 + cur.c1) / 2, cur.c1};
      for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j) q_child(&cur, rows[i], rows[i + 1], cols[j], cols[j + 1], xs, ys, &kids[n_kids++]);
    }
    n_nodes -= 1;
    for (int k = 0; k < n_kids; ++k) {
      if (kids[k].n == 0) {
        free(kids[k].idx);
        continue;
      }
      kids[k].seq = seq++;
      if (n_live == live_cap) {
        live_cap *= 2;
        live = (qnode *)realloc(live, sizeof(qnode) * live_cap);
      }
      live[n_live++] = kids[k];
      n_nodes += 1;
    }
    free(cur.idx);
  }
  /* nodes2kpoints :182-192: first min(need, |M|) nodes in multimap order */
  size_t take = n_live < (size_t)need ? n_live : (size_t)need;
  uint8_t *sel = (uint8_t *)calloc((size_t)(n > 0 ? n : 1), 1);
  uint8_t *used = (uint8_t *)calloc(n_live > 0 ? n_live : 1, 1);
  for (size_t t = 0; t < take; ++t) {
    size_t best = (size_t)-1;
    for (size_t i = 0; i < n_live; ++i) {
      if (used[i]) continue;
      if (best == (size_t)-1 || live[i].n > live[best].n || (live[i].n == live[best].n && live[i].seq < live[best].seq))
        best = i;
    }
    used[best] = 1;
    size_t max_idx = 0; /* getFeature :103-117 */
    float max_resp = 0.0f;
    for (int k = 0; k < live[best].n; ++k) {
      int id = live[best].idx[k];
      if (resp[id] > max_resp) {
        max_idx = (size_t)id;
        max_resp = resp[id];
      }
    }
    if ((int)max_idx < n) sel[max_idx] = 1; /* n == 0 && need == 1 reads kps[0] out of range in the reference */
  }
  int n_out = 0;
  for (int i = 0; i < n; ++i)
    if (sel[i]) out_idx[n_out++] = i;
  for (size_t i = 0; i < n_live; ++i) free(live[i].idx);
  free(live);
  free(sel);
  free(used);
  if (n_pops) *n_pops = pops;
  return n_out;
}

/* ------------------------------------------------------------------------------------------------ */
/* src/ORBExtractor.cc:465-487 */
double oracle_ic_angle(const uint8_t *img, size_t stride, int x, int y) {
  static int umax[16];
  static int init = 0;
  if (!init) {
    oracle_umax(umax);
    init = 1;
  }
  const int R = 15;
  int m10 = 0, m01 = 0;
  const uint8_t *c = img + (size_t)y * stride + x;
  for (int dx = -R; dx <= R; ++dx) m10 += dx * c[dx];
  for (int dy = 1; dy <= R; ++dy) {
    int vsum = 0, d = umax[dy];
    for (int dx = -d; dx <= d; ++dx) {
      int up = c[(ptrdiff_t)dy * (ptrdiff_t)stride + dx], down = c[-(ptrdiff_t)dy * (ptrdiff_t)stride + dx];
      m10 += dx * (up + down);
      vsum += (up - down);
    }
    m01 += vsum * dy;
  }
  return atan2((double)m01, (double)m10);
}

/* src/ORBExtractor.cc:427-456 and rotateTemplate :534-540 */
void oracle_brief(const uint8_t *blurred, size_t stride, float px, float py, double theta, const float *pattern,
                  uint8_t *desc) {
  double c = cos(theta), s = sin(theta);
  for (int b = 0; b < 256; ++b) {
    const float *t = pattern + 4 * b;
    float p1x = (float)((double)t[0] * c - (double)t[1] * s);
    float p1y = (float)((double)t[0] * s + (double)t[1] * c);
    float p2x = (float)((double)t[2] * c - (double)t[3] * s);
    float p2y = (float)((double)t[2] * s + (double)t[3] * c);
    uint8_t v1 = blurred[(size_t)cv_round_f(py + p1y) * stride + (size_t)cv_round_f(px + p1x)];
    uint8_t v2 = blurred[(size_t)cv_round_f(py + p2y) * stride + (size_t)cv_round_f(px + p2x)];
    if ((b & 7) == 0) desc[b >> 3] = 0;
    desc[b >> 3] |= (uint8_t)((v1 < v2) << (b & 7));
  }
}

/* ------------------------------------------------------------------------------------------------ */
int oracle_pyramid_build(oracle_pyramid *p, const uint8_t *img, int w, int h, size_t stride, int n_features,
                         int n_levels, float scale_factor) {
  memset(p, 0, sizeof(*p));
  if (n_levels < 1 || n_levels > ORACLE_MAX_LEVELS) return -2;
  p->n_levels = n_levels;
  oracle_scale_factors(scale_factor, n_levels, p->sf);
  oracle_level_quotas(n_features, scale_factor, n_levels, p->quota);
  if (oracle_level_sizes(w, h, p->sf, n_levels, p->w, p->h) != 0) return -1;
  for (int l = 0; l < n_levels; ++l) {
    size_t sz = (size_t)p->w[l] * (size_t)p->h[l];
    p->img[l] = (uint8_t *)malloc(sz);
    p->blur[l] = (uint8_t *)malloc(sz);
    if (l == 0)
      for (int y = 0; y < h; ++y) memcpy(p->img[0] + (size_t)y * w, img + (size_t)y * stride, (size_t)w);
    else /* every level is resized from level 0 (:316), never cascaded */
      oracle_resize_linear_u8(p->img[0], w, h, (size_t)w, p->img[l], p->w[l], p->h[l], (size_t)p->w[l]);
  }
  for (int l = 0; l < n_levels; ++l)
    oracle_gaussian_blur7_u8(p->img[l], p->w[l], p->h[l], (size_t)p->w[l], p->blur[l], (size_t)p->w[l]);
  return 0;
}

void oracle_pyramid_free(oracle_pyramid *p) {
  for (int l = 0; l < p->n_levels; ++l) {
    free(p->img[l]);
    free(p->blur[l]);
    p->img[l] = p->blur[l] = NULL;
  }
}

/* src/ORBExtractor.cc:499-508 (extract), :376-386 (quadtree + border shift), :397-415 (computeBRIEF vector form) */
int oracle_extract(const oracle_pyramid *p, int ini_th, int min_th, const float *pattern, oracle_keypoint *kps,
                   uint8_t *desc, double *angles_rad, int *level_counts) {
  int n_out = 0;
  for (int l = 0; l < p->n_levels; ++l) {
    int w = p->w[l], h = p->h[l];
    int cap = w * h / 4 + 16;
    int *xs = (int *)malloc(sizeof(int) * 3 * (size_t)cap), *ys = xs + cap, *sc = ys + cap;
    int n = oracle_fast_cells(p->img[l], w, h, (size_t)w, ini_th, min_th, xs, ys, sc, cap, NULL);
    if (n < 0) {
      free(xs);
      return -1;
    }
    float *fx = (float *)malloc(sizeof(float) * 3 * (size_t)(n + 1)), *fy = fx + n + 1, *fr = fy + n + 1;
    for (int i = 0; i < n; ++i) {
      fx[i] = (float)xs[i];
      fy[i] = (float)ys[i];
      fr[i] = (float)sc[i];
    }
    int need = p->quota[l];
    int *sel = (int *)malloc(sizeof(int) * (size_t)(need + 1));
    int ns = oracle_quadtree_select(w - 32, h - 32, n, fx, fy, fr, need, sel, NULL);
    for (int k = 0; k < ns; ++k) {
      oracle_keypoint *kp = &kps[n_out];
      float x = fx[sel[k]] + 16.f, y = fy[sel[k]] + 16.f;
      double theta = oracle_ic_angle(p->img[l], (size_t)w, cv_round_f(x), cv_round_f(y));
      oracle_brief(p->blur[l], (size_t)w, x, y, theta, pattern, desc + 32 * (size_t)n_out);
      kp->angle = (float)(theta / M_PI * 180);
      kp->x = x * p->sf[l];
      kp->y = y * p->sf[l];
      kp->size = 7.f;
      kp->response = fr[sel[k]];
      kp->octave = l;
      kp->class_id = -1;
      if (angles_rad) angles_rad[n_out] = theta;
      ++n_out;
    }
    if (level_counts) level_counts[l] = ns;
    free(sel);
    free(fx);
    free(xs);
  }
  return n_out;
}

/* ------------------------------------------------------------------------------------------------ */
/* src/ORBMatcher.cc:941-956 */
static int desc_distance(const uint8_t *a, const uint8_t *b) {
  int dist = 0;
  for (int i = 0; i < 8; ++i) {
    uint32_t pa, pb;
    memcpy(&pa, a + 4 * i, 4);
    memcpy(&pb, b + 4 * i, 4);
    uint32_t v = pa ^ pb;
    v = v - ((v >> 1) & 0x55555555u);
    v = (v & 0x33333333u) + ((v >> 2) & 0x33333333u);
    dist += (int)((((v + (v >> 4)) & 0xF0F0F0Fu) * 0x1010101u) >> 24);
  }
  return dist;
}

/* src/ORBMatcher.cc:1002-1011 (getPitch) + :893-905 (SAD): 11x11 patches, each minus its own centre, L1 norm */
static float sad_11(const uint8_t *li, size_t ls, int lx, int ly, const uint8_t *ri, size_t rs, int rx, int ry) {
  float lc = (float)li[(size_t)ly * ls + (size_t)lx], rc = (float)ri[(size_t)ry * rs + (size_t)rx];
  double acc = 0; /* cv::norm accumulates CV_32F L1 in double */
  for (int dy = -5; dy <= 5; ++dy)
    for (int dx = -5; dx <= 5; ++dx) {
      float a = (float)li[(size_t)(ly + dy) * ls + (size_t)(lx + dx)] - lc;
      float b = (float)ri[(size_t)(ry + dy) * rs + (size_t)(rx + dx)] - rc;
      acc += fabs((double)(a - b));
    }
  return (float)acc;
}

/* src/ORBMatcher.cc:841-881 */
static float pixel_sad_match(const oracle_pyramid *left, const oracle_pyramid *right, const oracle_keypoint *lk,
                             const oracle_keypoint *rk) {
  const int L = 5;
  const uint8_t *li = left->img[lk->octave], *ri = right->img[rk->octave];
  size_t ls = (size_t)left->w[lk->octave], rs = (size_t)right->w[rk->octave];
  int lx = cv_floor_f(lk->x / left->sf[lk->octave]), ly = cv_floor_f(lk->y / left->sf[lk->octave]);
  int rx = cv_floor_f(rk->x / right->sf[rk->octave]), ry = cv_floor_f(rk->y / right->sf[rk->octave]);
  float scores[11];
  float min_score = 3.402823466e+38F;
  int best = 0;
  for (int l = -L; l < L + 1; ++l) {
    float s = sad_11(li, ls, lx, ly, ri, rs, rx + l, ry);
    if (s < min_score) {
      min_score = s;
      best = l;
    }
    scores[l + L] = s;
  }
  float delta = 0;
  best += L;
  if (best > 0 && best < 11 - 1) {
    float s1 = scores[best - 1], s2 = scores[best], s3 = scores[best + 1];
    delta = (float)(0.5 * (double)(s1 - s3) / (double)(s1 + s3 - 2 * s2));
    if (delta < 1 && delta > -1)
      delta *= right->sf[rk->octave];
    else
      delta = 0;
  }
  return delta;
}

int oracle_search_by_stereo(const oracle_pyramid *left, const oracle_pyramid *right, const oracle_keypoint *kl,
                            const uint8_t *dl, int nl, const oracle_keypoint *kr, const uint8_t *dr, int nr, float fx,
                            float bf, double *u_right, double *depth, int *match_idx) {
  int rows = left->h[0], cols = left->w[0];
  for (int i = 0; i < nl; ++i) {
    u_right[i] = -1.0;
    depth[i] = -1.0;
    if (match_idx) match_idx[i] = -1;
  }
  /* createRowIndexDB :915-932 -- stored as [minRow, maxRow) per right keypoint; a row's list is ascending idx */
  int *rmin = (int *)malloc(sizeof(int) * 2 * (size_t)(nr + 1)), *rmax = rmin + nr + 1;
  for (int j = 0; j < nr; ++j) {
    float r = (float)(2.0 * (double)right->sf[kr[j].octave]);
    unsigned row = (unsigned)cv_round_f(kr[j].y);
    rmax[j] = imin(rows, cv_round_f((float)row + r + 1));
    rmin[j] = imax(0, cv_round_f((float)row - r));
  }
  int n_matches = 0;
  for (int i = 0; i < nl; ++i) {
    const oracle_keypoint *lk = &kl[i];
    float maxU = lk->x - 0;
    float minU = lk->x - fx > 0.f ? lk->x - fx : 0.f;
    int row = cv_round_f(lk->y);
    int best_j = -1, best_d = 0x7fffffff;
    for (int j = 0; j < nr; ++j) { /* ascending index == order inside rowIdxDB[row] */
      if (row < rmin[j] || row >= rmax[j]) continue;
      float xr = kr[j].x;
      if (!(xr < maxU && xr > minU)) continue;
      int d = desc_distance(dl + 32 * (size_t)i, dr + 32 * (size_t)j);
      if (d < best_d) {
        best_d = d;
        best_j = j;
      }
    }
    if (best_j < 0) continue;
    if (best_d > 75) continue; /* mnMeanThreshold :1088 */
    const oracle_keypoint *rk = &kr[best_j];
    if (lk->octave > rk->octave + 1 || lk->octave < rk->octave - 1) continue;
    /* Drop the match when the left 11x11 window or the right 11x21 window (11 shifts of 11 columns) leaves its level
     * image, as stereo_kernel does: the reference throws in cv::Mat::rowRange there (DESIGN section 2).  Only undistorted
     * left keypoints can get that close to the border. */
    {
      int lo = lk->octave, ro = rk->octave;
      int lx = cv_floor_f(lk->x / left->sf[lo]), ly = cv_floor_f(lk->y / left->sf[lo]);
      int rx = cv_floor_f(rk->x / right->sf[ro]), ry = cv_floor_f(rk->y / right->sf[ro]);
      if (lx - 5 < 0 || ly - 5 < 0 || lx + 5 >= left->w[lo] || ly + 5 >= left->h[lo] || rx - 10 < 0 || ry - 5 < 0 || rx + 10 >= right->w[ro] ||
          ry + 5 >= right->h[ro])
        continue;
    }
    float dU = pixel_sad_match(left, right, lk, rk);
    float rightU = rk->x + dU;
    rightU = rightU > 0.f ? rightU : 0.f;
    float lim = (float)cols - 1;
    rightU = rightU < lim ? rightU : lim;
    float delta = lk->x - rightU;
    if (delta <= 0) {
      rightU = rk->x;
      delta = lk->x - rightU;
      if (delta <= 0) continue;
    }
    u_right[i] = rightU;
    depth[i] = bf / (lk->x - rightU);
    if (match_idx) match_idx[i] = best_j;
    ++n_matches;
  }
  free(rmin);
  return n_matches;
}

/* src/Frame.cc:125-159 */
void oracle_rgbd_lookup(const void *depth_raw, int is_float, int w, int h, size_t stride_elems, float depth_scale,
                        const oracle_keypoint *kps_raw, const oracle_keypoint *kps_undist, int n, float bf,
                        double *u_right, double *depth) {
  (void)w;
  (void)h;
  float inv = (float)(1.0 / (double)depth_scale); /* Mat /= s  ==  convertTo(-1, 1./s), computed in float */
  for (int i = 0; i < n; ++i) {
    int yy = (int)kps_raw[i].y, xx = (int)kps_raw[i].x; /* at<float>(float, float): truncation */
    float raw = is_float ? ((const float *)depth_raw)[(size_t)yy * stride_elems + (size_t)xx]
                         : (float)((const uint16_t *)depth_raw)[(size_t)yy * stride_elems + (size_t)xx];
    float d = raw * inv;
    u_right[i] = -1;
    depth[i] = -1;
    if (d > 0) {
      depth[i] = d;
      u_right[i] = kps_undist[i].x - bf / d;
    }
  }
}

/* ---------------------------------------------------------------------------------------------------------------
 * Tracking-side area matchers (SURVEY section 8(f) rank 2)
 * --------------------------------------------------------------------------------------------------------------- */

/* VirtualFrame::initGrid, src/Frame.cc:53-69.  Keypoints whose cell lies outside the grid index mGrids out of range in
 * the reference; they are left out here.  CSR: start[rows*cols+1], entries[n] (keypoint order inside a cell). */
void oracle_init_grid(const oracle_keypoint *kps, int n, float min_u, float min_v, float max_u, float max_v, int *rows_out,
                      int *cols_out, int *start, int cap_cells, int *entries) {
  int rows = cv_ceil_f((float)(max_v - min_v) / 48u);
  int cols = cv_ceil_f((float)(max_u - min_u) / 64u);
  *rows_out = rows;
  *cols_out = cols;
  if (rows <= 0 || cols <= 0 || rows * cols > cap_cells) return;
  int nc = rows * cols;
  for (int c = 0; c <= nc; ++c) start[c] = 0;
  for (int pass = 0; pass < 2; ++pass) {
    for (int i = 0; i < n; ++i) {
      long r = cv_floor_f(kps[i].y / 48u), c = cv_floor_f(kps[i].x / 64u);
      if (r < 0 || r >= rows || c < 0 || c >= cols) continue;
      if (pass == 0)
        ++start[r * cols + c + 1];
      else
        entries[start[r * cols + c]++] = i;
    }
    if (pass == 0)
      for (int c = 0; c < nc; ++c) start[c + 1] += start[c];
    else {
      for (int c = nc; c > 0; --c) start[c] = start[c - 1];
      start[0] = 0;
    }
  }
}

/* VirtualFrame::findFeaturesInArea, src/Frame.cc:286-311 (getScaledFactor2: include/ORB_SLAM2/Frame.h:207).
 * A window that leaves the grid (negative maxX/maxY, or a cell index beyond the grid) is undefined behaviour in the
 * reference (size_t loop counters over mGrids); here the cell range is clipped to the grid. */
int oracle_find_features_in_area(const oracle_keypoint *kps, const int *start, const int *entries, int rows, int cols,
                                 const float *sf, float max_u, float max_v, float x, float y, float radius, int octave,
                                 int min_level, int max_level, int *out) {
  float sf2 = (float)pow((double)sf[octave], 2);
  radius = radius * sf2;
  int min_x = cv_round_f(x - radius), max_x = cv_round_f(x + radius);
  int min_y = cv_round_f(y - radius), max_y = cv_round_f(y + radius);
  if (min_x < 0) min_x = 0;
  if (max_x > (int)max_u) max_x = (int)max_u;
  if (min_y < 0) min_y = 0;
  if (max_y > (int)max_v) max_y = (int)max_v;
  if (max_x < 0 || max_y < 0) return 0;
  int c0 = cv_floor_f((float)min_x / 64u), c1 = cv_floor_f((float)max_x / 64u);
  int r0 = cv_floor_f((float)min_y / 48u), r1 = cv_floor_f((float)max_y / 48u);
  if (c1 > cols - 1) c1 = cols - 1;
  if (r1 > rows - 1) r1 = rows - 1;
  int n = 0;
  for (int r = r0; r <= r1; ++r)
    for (int c = c0; c <= c1; ++c)
      for (int e = start[r * cols + c]; e < start[r * cols + c + 1]; ++e) {
        int id = entries[e], o = kps[id].octave;
        if (o <= max_level && o >= min_level) out[n++] = id;
      }
  return n;
}

/* ORBMatcher::getBestMatch, src/ORBMatcher.cc:967-990: the running second-best is only updated by candidates that are
 * NOT a new minimum, and the displaced minimum is not demoted into it. */
int oracle_best_match(const uint8_t *desc, const uint8_t *cand_desc, const int *cand_idx, int n, int *best_dist,
                      float *ratio) {
  int min_d = INT_MAX, second_d = INT_MAX, min_idx = 0;
  for (int k = 0; k < n; ++k) {
    int d = desc_distance(desc, cand_desc + 32 * (size_t)cand_idx[k]);
    if (d < min_d) {
      min_d = d;
      min_idx = cand_idx[k];
    } else if (d < second_d)
      second_d = d;
  }
  *ratio = (float)min_d / (float)second_d;
  *best_dist = min_d;
  return min_idx;
}

/* The inner step shared by both ORBMatcher::searchByProjection overloads (src/ORBMatcher.cc:296-343 and :575-591):
 * candidates in the area, minus the excluded keypoints (:322-331), then getBestMatch.  best_idx = -1 / n_cand = 0 when
 * nothing is left (the reference `continue`s). */
void oracle_search_in_area(const oracle_keypoint *kps, const uint8_t *desc, int n_kps, const int *start,
                           const int *entries, int rows, int cols, const float *sf, float max_u, float max_v,
                           const oracle_area_query *q, const uint8_t *q_desc, int n_q, const uint8_t *exclude,
                           int *best_idx, int *best_dist, float *ratio, int *n_cand) {
  int *cand = (int *)malloc(sizeof(int) * (size_t)(n_kps > 0 ? n_kps : 1));
  for (int i = 0; i < n_q; ++i) {
    int n = oracle_find_features_in_area(kps, start, entries, rows, cols, sf, max_u, max_v, q[i].x, q[i].y, q[i].radius,
                                         q[i].octave, q[i].min_level, q[i].max_level, cand);
    if (exclude) {
      int m = 0;
      for (int k = 0; k < n; ++k)
        if (!exclude[cand[k]]) cand[m++] = cand[k];
      n = m;
    }
    n_cand[i] = n;
    best_idx[i] = -1;
    best_dist[i] = INT_MAX;
    ratio[i] = 0.f;
    if (n == 0) continue;
    best_idx[i] = oracle_best_match(q_desc + 32 * (size_t)i, desc, cand, n, &best_dist[i], &ratio[i]);
  }
  free(cand);
}

/* ORBMatcher::verifyAngle, src/ORBMatcher.cc:1013-1051 (mnBinNum = 30, mnBinChoose = 3): keeps the matches of the three
 * fullest bins of the angle-difference histogram, emitted in ascending bin order, original order inside a bin.
 * Arrays are rewritten in place; returns the new count. */
int oracle_verify_angle(int n, int *query_idx, int *train_idx, float *distance, const oracle_keypoint *kps1,
                        const oracle_keypoint *kps2) {
  enum { kBins = 30, kChoose = 3 };
  int *bin = (int *)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
  int count[kBins] = {0};
  for (int i = 0; i < n; ++i) {
    float diff = kps1[query_idx[i]].angle - kps2[train_idx[i]].angle;
    diff = diff >= 0 ? diff : 360 + diff;
    int b = (int)(diff / (360 / kBins));
    if (b == 30) b = 0;
    bin[i] = b;
    ++count[b];
  }
  int good[kBins] = {0};
  for (int k = 0; k < kChoose; ++k) {
    int max_size = 0, max_id = 0, init = 0;
    for (int b = 0; b < kBins; ++b) {
      if (good[b]) continue;
      if (count[b] > max_size) {
        max_id = b;
        max_size = count[b];
        init = 1;
      }
    }
    if (init) good[max_id] = 1;
  }
  int *qi = (int *)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1)), *ti = (int *)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
  float *di = (float *)malloc(sizeof(float) * (size_t)(n > 0 ? n : 1));
  int m = 0;
  for (int b = 0; b < kBins; ++b) {
    if (!good[b]) continue;
    for (int i = 0; i < n; ++i)
      if (bin[i] == b) {
        qi[m] = query_idx[i];
        ti[m] = train_idx[i];
        di[m] = distance[i];
        ++m;
      }
  }
  for (int i = 0; i < m; ++i) {
    query_idx[i] = qi[i];
    train_idx[i] = ti[i];
    distance[i] = di[i];
  }
  free(bin);
  free(qi);
  free(ti);
  free(di);
  return m;
}

/* ---------------------------------------------------------------------------------------------------------------
 * Result serialisation (SURVEY section 8(f) rank 4): orbslam2.KeyFrameData, proto3 wire format
 * (proto/Keyframe.proto:7-17,45-64), the bytes KeyFrame::serializeToProtobuf (src/KeyFrame.cc:553-647) produces for
 * a keyframe made from a fresh frame: no BoW yet (empty but present messages 10, 11), pose Tcw, no connections,
 * children or loop edges, and -1 for every keypoint's map point.
 * --------------------------------------------------------------------------------------------------------------- */
static size_t pb_varint(uint8_t *o, uint64_t v) {
  size_t n = 0;
  while (v >= 0x80) {
    o[n++] = (uint8_t)(v | 0x80);
    v >>= 7;
  }
  o[n++] = (uint8_t)v;
  return n;
}
static size_t pb_f32(uint8_t *o, float f) {
  memcpy(o, &f, 4);
  return 4;
}
static uint32_t f32_bits(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  return u;
}

size_t oracle_serialize_keyframe(const oracle_keypoint *kps, const uint8_t *desc, const double *u_right,
                                 const double *depth, int n, uint64_t id, float max_u, float max_v, float min_u,
                                 float min_v, const float *pose_rt /*[12] R row-major + t, NULL = identity*/,
                                 int with_map_points, uint8_t *out, size_t cap) {
  size_t need = 128 + (size_t)n * (28 + 4 + 4 + 36 + 10); /* a KeyPoint entry is at most 2 + 5 + 5 + 11 + 5 bytes */
  if (cap < need) return 0;
  uint8_t *o = out;
  if (id) { /* proto3: scalar fields equal to zero are not written */
    *o++ = 0x08;
    o += pb_varint(o, id);
  }
  const float b[4] = {max_u, max_v, min_u, min_v};
  for (int k = 0; k < 4; ++k)
    if (f32_bits(b[k])) {
      *o++ = (uint8_t)(((2 + k) << 3) | 5);
      o += pb_f32(o, b[k]);
    }
  for (int i = 0; i < n; ++i) { /* repeated KeyPoint keypoints = 6 */
    uint8_t m[32];
    size_t l = 0;
    if (f32_bits(kps[i].x)) {
      m[l++] = 0x0D;
      l += pb_f32(m + l, kps[i].x);
    }
    if (f32_bits(kps[i].y)) {
      m[l++] = 0x15;
      l += pb_f32(m + l, kps[i].y);
    }
    if (kps[i].octave) {
      m[l++] = 0x18;
      l += pb_varint(m + l, (uint64_t)(int64_t)kps[i].octave); /* int32: negative values sign-extend to 10 bytes */
    }
    if (f32_bits(kps[i].angle)) {
      m[l++] = 0x25;
      l += pb_f32(m + l, kps[i].angle);
    }
    *o++ = 0x32;
    o += pb_varint(o, l);
    memcpy(o, m, l);
    o += l;
  }
  if (n) { /* repeated float right_u = 7, depths = 8: packed; the writer narrows the doubles to float (:575-576) */
    *o++ = 0x3A;
    o += pb_varint(o, 4u * (uint64_t)n);
    for (int i = 0; i < n; ++i) o += pb_f32(o, (float)u_right[i]);
    *o++ = 0x42;
    o += pb_varint(o, 4u * (uint64_t)n);
    for (int i = 0; i < n; ++i) o += pb_f32(o, (float)depth[i]);
  }
  for (int i = 0; i < n; ++i) { /* repeated Descriptor descriptors = 9 { bytes data = 1 } */
    *o++ = 0x4A;
    *o++ = 34;
    *o++ = 0x0A;
    *o++ = 32;
    memcpy(o, desc + 32 * (size_t)i, 32);
    o += 32;
  }
  *o++ = 0x52; /* bow_vector = 10: mutable_bow_vector() makes the empty message present (:586) */
  *o++ = 0;
  *o++ = 0x5A; /* feature_vector = 11 (:593) */
  *o++ = 0;
  {            /* Pose pose = 12 { repeated float rotation = 1 [9]; repeated float translation = 2 [3] } (:602-608) */
    static const float eye[12] = {1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0};
    const float *rt = pose_rt ? pose_rt : eye;
    *o++ = 0x62;
    *o++ = 52;
    *o++ = 0x0A;
    *o++ = 36;
    for (int k = 0; k < 9; ++k) o += pb_f32(o, rt[k]);
    *o++ = 0x12;
    *o++ = 12;
    for (int k = 0; k < 3; ++k) o += pb_f32(o, rt[9 + k]);
  }
  if (with_map_points && n) { /* repeated int64 map_points = 16: -1 per keypoint without a map point (:641-646) */
    o += pb_varint(o, (16u << 3) | 2u);
    o += pb_varint(o, 10u * (uint64_t)n);
    for (int i = 0; i < n; ++i) {
      memset(o, 0xFF, 9);
      o[9] = 0x01;
      o += 10;
    }
  }
  return (size_t)(o - out);
}

/* ---------------------------------------------------------------------------------------------------------------
 * Bag-of-words transform (SURVEY section 8(f) rank 3).  PARITY UNPINNED: DBoW3 (https://github.com/rmsalinas/DBow3,
 * un-vendored, find_package(DBoW3) in CMakeLists.txt:15, no version pin) is not under /root/reference and the reference
 * ships no vocabulary, so this restates DBoW3's published algorithm -- Vocabulary::transform(features, BowVector&,
 * FeatureVector&, levelsup) and the per-feature descent, BowVector::addWeight / normalize(L1), FeatureVector::addFeature
 * -- anchored on the reference's call site include/ORB_SLAM2/Frame.h:224-231 (levelsup = 4) and on the vocabulary text
 * format the reference's README prescribes (ORB-SLAM2's ORBvoc.txt: "k L scoring weighting", then one node per line
 * "parent isLeaf d0..d31 weight"; node ids and word ids are assigned in line order).
 * Supported: TF_IDF / TF weighting with a scoring that normalises L1 (ORBvoc.txt: TF_IDF, L1_NORM).
 * --------------------------------------------------------------------------------------------------------------- */

/* Descent of one descriptor: at every level the child with the smallest Hamming distance, the first one among equals
 * (strict <, children in id order).  nid = the node reached at level L - levelsup (root if that is <= 0). */
void oracle_bow_descend(const oracle_vocab *v, const uint8_t *desc, int levelsup, int32_t *word_id, double *weight,
                        int32_t *nid) {
  const int nid_level = v->L - levelsup;
  int32_t node = 0, at = 0;
  int level = 0;
  do {
    ++level;
    const int c0 = v->child_start[node], c1 = v->child_start[node + 1];
    double best = 1.7976931348623157e308;
    for (int c = c0; c < c1; ++c) {
      const int32_t id = v->child_ids[c];
      const double d = (double)desc_distance(desc, v->desc + 32 * (size_t)id);
      if (d < best) {
        best = d;
        node = id;
      }
    }
    if (level == nid_level) at = node;
  } while (v->child_start[node] != v->child_start[node + 1]);
  *word_id = v->word_id[node];
  *weight = v->weight[node];
  *nid = nid_level <= 0 ? 0 : at;
}

/* Vocabulary::transform for n descriptors.  Outputs: the BowVector as (ids ascending, values) and the FeatureVector as
 * a CSR (node ids ascending, start[m+1], feature indices in insertion order).  Returns the BowVector size. */
int oracle_bow_transform(const oracle_vocab *v, const uint8_t *desc, int n, int levelsup, int32_t *bow_ids,
                         double *bow_vals, int32_t *fv_nodes, int32_t *fv_start, int32_t *fv_feats, int *fv_count) {
  int m = 0;
  int32_t *f_node = (int32_t *)malloc(sizeof(int32_t) * (size_t)(n > 0 ? n : 1));
  int *f_ok = (int *)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
  for (int i = 0; i < n; ++i) {
    int32_t id, nid;
    double w;
    oracle_bow_descend(v, desc + 32 * (size_t)i, levelsup, &id, &w, &nid);
    f_node[i] = nid;
    f_ok[i] = w > 0;
    if (!(w > 0)) continue; /* stopped word */
    /* BowVector::addWeight: std::map lower_bound, += if present, insert otherwise */
    int lo = 0, hi = m;
    while (lo < hi) {
      int mid = (lo + hi) >> 1;
      if (bow_ids[mid] < id) lo = mid + 1; else hi = mid;
    }
    if (lo < m && bow_ids[lo] == id)
      bow_vals[lo] += w;
    else {
      memmove(bow_ids + lo + 1, bow_ids + lo, sizeof(int32_t) * (size_t)(m - lo));
      memmove(bow_vals + lo + 1, bow_vals + lo, sizeof(double) * (size_t)(m - lo));
      bow_ids[lo] = id;
      bow_vals[lo] = w;
      ++m;
    }
  }
  /* BowVector::normalize(L1): the sum runs over the map in key order */
  double norm = 0.0;
  for (int k = 0; k < m; ++k) norm += fabs(bow_vals[k]);
  if (norm > 0.0)
    for (int k = 0; k < m; ++k) bow_vals[k] /= norm;
  /* FeatureVector (std::map<NodeId, std::vector<unsigned>>): node ids ascending, features in insertion order */
  int nn = 0, total = 0;
  for (int i = 0; i < n; ++i) {
    if (!f_ok[i]) continue;
    int seen = 0;
    for (int k = 0; k < nn; ++k) seen |= fv_nodes[k] == f_node[i];
    if (!seen) fv_nodes[nn++] = f_node[i];
  }
  for (int a = 1; a < nn; ++a) { /* insertion sort of the distinct node ids */
    int32_t x = fv_nodes[a];
    int b = a - 1;
    while (b >= 0 && fv_nodes[b] > x) {
      fv_nodes[b + 1] = fv_nodes[b];
      --b;
    }
    fv_nodes[b + 1] = x;
  }
  for (int k = 0; k < nn; ++k) {
    fv_start[k] = total;
    for (int i = 0; i < n; ++i)
      if (f_ok[i] && f_node[i] == fv_nodes[k]) fv_feats[total++] = i;
  }
  fv_start[nn] = total;
  *fv_count = nn;
  free(f_node);
  free(f_ok);
  return m;
}

/* The matching loop of ORBMatcher::searchByBow, src/ORBMatcher.cc:170-255, without the MapPoint objects: the caller
 * passes what the loop derives from them -- kf_query_ok[pkId] ("this keyframe feature takes part", :195-212) and
 * frame_cand_ok[pId] ("this frame feature may be matched", :216-233).  Merge-join of the two FeatureVectors (:181-186);
 * for every keyframe feature of a common node, in the keyframe's list order: candidates = the frame's features of the
 * node that pass the mask, then getBestMatch (:238).  One output row per visited keyframe feature that has candidates
 * (the reference's ++nMatch, :239): kf_idx, best_idx, best_dist, ratio.  The caller thresholds (:240-245: rejected iff
 * dist > mnMinThreshold || ratio > mfRatio -- a NaN ratio is accepted) and runs verifyAngle.  Returns the row count. */
int oracle_search_by_bow(const int32_t *f_nodes, const int32_t *f_start, const int32_t *f_feats, int f_n_nodes,
                         const uint8_t *f_desc, const uint8_t *frame_cand_ok, const int32_t *k_nodes,
                         const int32_t *k_start, const int32_t *k_feats, int k_n_nodes, const uint8_t *k_desc,
                         const uint8_t *kf_query_ok, int32_t *kf_idx, int32_t *best_idx, int32_t *best_dist,
                         float *ratio, int32_t *n_cand) {
  int rows = 0, fi = 0, ki = 0;
  int cap = 0;
  for (int j = 0; j < f_n_nodes; ++j) cap = imax(cap, f_start[j + 1] - f_start[j]);
  int *cand = (int *)malloc(sizeof(int) * (size_t)(cap > 0 ? cap : 1));
  while (fi < f_n_nodes && ki < k_n_nodes) {
    if (f_nodes[fi] > k_nodes[ki])
      ++ki;
    else if (f_nodes[fi] < k_nodes[ki])
      ++fi;
    else {
      for (int e = k_start[ki]; e < k_start[ki + 1]; ++e) {
        const int pk = k_feats[e];
        if (kf_query_ok && !kf_query_ok[pk]) continue;
        int n = 0;
        for (int t = f_start[fi]; t < f_start[fi + 1]; ++t)
          if (!frame_cand_ok || frame_cand_ok[f_feats[t]]) cand[n++] = f_feats[t];
        if (n == 0) continue;
        kf_idx[rows] = pk;
        n_cand[rows] = n;
        best_idx[rows] = oracle_best_match(k_desc + 32 * (size_t)pk, f_desc, cand, n, &best_dist[rows], &ratio[rows]);
        ++rows;
      }
      ++fi;
      ++ki;
    }
  }
  free(cand);
  return rows;
}
