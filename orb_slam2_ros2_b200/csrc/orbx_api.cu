// orbx_api.cu -- host layer behind the C ABI of include/orbx.h: per-context tables, device buffers, launch sequences.
//
// The per-config tables restate ORBExtractor::initPyramid's bookkeeping (src/ORBExtractor.cc:283-317) and the FAST cell
// grid of extractFast (:334-362) once per context -- the reference recomputes them per frame and keeps part of them in
// process-wide statics (:511-524); here nothing is static, so contexts with different configurations can coexist.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <new>
#include <sstream>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "../../include/orbx_pattern.h"
#include "orbx_internal.h"

using namespace orbx;

namespace
{

inline int cv_round(float v) { return (int)lrintf(v); }  // cvRound: round half to even (default FP environment)
inline int cv_round(double v) { return (int)lrint(v); }
inline int cv_floor(float v)
{
  int i = (int)v;
  return i - (i > v);
}

template <typename T> int dev_alloc(orbx_ctx *c, T **ptr, size_t count)
{
  void *q = nullptr;
  cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 256);
  if (e != cudaSuccess) return fail(c, ORBX_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e));
  c->allocs.push_back(q);
  *ptr = (T *)q;
  return ORBX_OK;
}

template <typename T> int dev_upload(orbx_ctx *c, const T **ptr, const std::vector<T> &v)
{
  T *d = nullptr;
  int rc = dev_alloc(c, &d, v.size() ? v.size() : 1);
  if (rc) return rc;
  if (!v.empty()) ORBX_CUDA(c, cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  *ptr = d;
  return ORBX_OK;
}

// cv::resize INTER_LINEAR coefficient tables (OpenCV imgproc/resize.cpp): 11-bit fixed point, computed in float
void build_resize_axis(int src_n, int dst_n, bool zero_at_border, std::vector<int> &ofs, std::vector<short2> &coef)
{
  const double scale = 1.0 / ((double)dst_n / (double)src_n);
  for (int d = 0; d < dst_n; ++d)
  {
    float f = (float)((d + 0.5) * scale - 0.5);
    int s = cv_floor(f);
    f -= (float)s;
    if (zero_at_border)
    { // columns: taps are re-weighted at the border; rows are clamped by the kernel instead
      if (s < 0)
      {
        f = 0.f;
        s = 0;
      }
      if (s >= src_n - 1)
      {
        f = 0.f;
        s = src_n - 1;
      }
    }
    int a0 = cv_round((1.f - f) * 2048.f), a1 = cv_round(f * 2048.f);
    a0 = a0 < -32768 ? -32768 : (a0 > 32767 ? 32767 : a0);
    a1 = a1 < -32768 ? -32768 : (a1 > 32767 ? 32767 : a1);
    ofs.push_back(s);
    coef.push_back(make_short2((short)a0, (short)a1));
  }
}

int build_tables(orbx_ctx *c)
{
  const orbx_config &g = c->cfg;
  const int nl = g.n_levels;
  c->levels.assign(nl, Level());
  std::vector<int> tab_ofs;
  std::vector<short2> tab_coef;
  std::vector<uint4> tab_pair;
  std::vector<long long> strips; // 24.40 fixed point

  // scale factors (:283-289), per-level quotas (:291-301), level sizes (:305-317)
  std::vector<float> sf(nl);
  for (int l = 0; l < nl; ++l) sf[l] = (float)std::pow((double)g.scale_factor, (double)l);
  {
    const float scale = 1.0f / g.scale_factor;
    int sum = 0;
    int nfeats = cv_round((double)((float)g.n_features * (1 - scale)) / (1 - std::pow((double)scale, (double)nl)));
    for (int l = 0; l < nl - 1; ++l)
    {
      c->levels[l].quota = nfeats;
      sum += nfeats;
      nfeats = cv_round((float)nfeats * scale);
    }
    c->levels[nl - 1].quota = std::max(0, g.n_features - sum);
  }
  size_t pyr_off = 0;
  int cell_index = 0, sel_off = 0;
  size_t slot_off = 0, scratch_off = 0;
  int max_quota = 0, max_ini = 0;
  c->tiles.clear();
  c->cells.clear();
  for (int l = 0; l < nl; ++l)
  {
    Level &L = c->levels[l];
    L.sf = sf[l];
    L.w = l == 0 ? g.width : cv_round((float)g.width / sf[l]);
    L.h = l == 0 ? g.height : cv_round((float)g.height / sf[l]);
    if (L.w < 2 * 19 || L.h < 2 * 19) return fail(c, ORBX_ERR_IMAGE_SIZE, "pyramid level smaller than 2*19 px");
    L.pitch = (L.w + 15) & ~15;
    L.pyr_off = (int)pyr_off;
    pyr_off += (size_t)L.pitch * L.h;
    pyr_off = (pyr_off + 255) & ~(size_t)255;
    L.area2x = (l > 0 && L.w * 2 == g.width && L.h * 2 == g.height) ? 1 : 0;
    if (l > 0)
    {
      L.tab_x = (int)tab_ofs.size();
      build_resize_axis(g.width, L.w, true, tab_ofs, tab_coef);
      L.tab_y = (int)tab_ofs.size();
      build_resize_axis(g.height, L.h, false, tab_ofs, tab_coef);
      // pyramid_levels_kernel fetches the taps of two adjacent columns with one aligned 8-byte window when that always works
      L.pair_window = 1;
      auto eff = [&](int gx) { const int sx = tab_ofs[L.tab_x + gx]; return sx + 1 > g.width - 1 ? g.width - 2 : sx; };
      for (int gx = 0; gx + 1 < L.w; ++gx)
      {
        const int a = eff(gx), b = eff(gx + 1);
        if (std::max(a, b) + 1 - (std::min(a, b) & ~3) > 7) L.pair_window = 0;
      }
      // One entry per pair of columns (rx, rx + 1), rx = -4 + 2 j, of the tile grid incl. the 3-px halo (REFLECT_101):
      // value = src[sx] * ax + src[min(sx + 1, W - 1)] * ay; the second tap is always read at +1: in the last column (sx == W - 1,
      // where the table has ay == 0) the pair moves one pixel left with the weights swapped.
      L.tab_pair = (int)tab_pair.size();
      const uint32_t pitch0 = (uint32_t)c->levels[0].pitch;
      auto column = [&](int rx, uint32_t &sx, uint32_t &coef) {
        sx = 0, coef = 0; // columns beyond the level + halo: weight 0 -> value 0
        if (rx >= L.w + kHalo) return;
        const int gx = rx < 0 ? -rx : (rx >= L.w ? 2 * (L.w - 1) - rx : rx);
        sx = (uint32_t)tab_ofs[L.tab_x + gx];
        uint32_t ax = (uint32_t)tab_coef[L.tab_x + gx].x, ay = (uint32_t)tab_coef[L.tab_x + gx].y;
        if (sx + 1u > (uint32_t)(g.width - 1)) sx = (uint32_t)(g.width - 2), ay = ax + ay, ax = 0;
        coef = ax | (ay << 16);
      };
      const int n_tx = (L.w + kTileW - 1) / kTileW;
      for (int j = 0; j < n_tx * (kTileW / 2) + 4; ++j)
      {
        uint32_t sxa, sxb, ca, cb;
        column(-4 + 2 * j, sxa, ca);
        column(-3 + 2 * j, sxb, cb);
        uint32_t base_a, base_b;
        if (L.pair_window)
        { // both tap pairs inside the aligned 8 bytes that start at the lower column's word, never beyond the row's pitch
          const uint32_t lo = ca == 0u ? sxb : (cb == 0u ? sxa : std::min(sxa, sxb));
          base_a = base_b = std::min(lo & ~3u, pitch0 - 8u);
        }
        else
          base_a = std::min(sxa & ~3u, pitch0 - 8u), base_b = std::min(sxb & ~3u, pitch0 - 8u);
        if (ca == 0u && cb == 0u && !tab_pair.empty() && (int)tab_pair.size() > L.tab_pair)
          base_a = base_b = tab_pair.back().x & 0xffffu; // columns beyond the level: weight 0, any window inside the tile's source box
        const uint32_t oa = ca == 0u ? 0u : sxa - base_a, ob = cb == 0u ? 0u : sxb - base_b;
        if (oa > 6u || ob > 6u) return fail(c, ORBX_ERR_INVALID_ARG, "resize window does not fit 8 bytes");
        tab_pair.push_back(make_uint4(base_a | ((oa | ((oa + 1u) << 4)) << 16), base_b | ((ob | ((ob + 1u) << 4)) << 16), ca, cb));
      }
    }
    {
      // level-0 source rectangle of every tile (pyramid_levels_kernel stages it through TMA when the level's box fits)
      const size_t first_tile = c->tiles.size();
      int box_w = 0, box_h = 0;
      for (int y0 = 0; y0 < L.h; y0 += kTileH)
        for (int x0 = 0; x0 < L.w; x0 += kTileW)
        {
          Tile t{l, x0, y0, 0};
          if (l > 0 && !L.area2x)
          {
            uint32_t b_lo = 0xffffffffu, b_hi = 0;
            for (int q = 0; q < kTileW / 2 + 4; ++q)
            {
              const uint4 e = tab_pair[(size_t)L.tab_pair + (x0 >> 1) + q];
              b_lo = std::min(b_lo, std::min(e.x & 0xffffu, e.y & 0xffffu));
              b_hi = std::max(b_hi, std::max(e.x & 0xffffu, e.y & 0xffffu));
            }
            const int sx0 = (int)(b_lo & ~15u);
            const int gy_lo = std::max(y0 - kHalo, 0), gy_hi = std::min(y0 + kTileH + kHalo - 1, L.h - 1);
            const int sy0 = std::min(std::max(tab_ofs[L.tab_y + gy_lo], 0), g.height - 1);
            const int sy1 = std::min(std::max(tab_ofs[L.tab_y + gy_hi] + 1, 0), g.height - 1);
            box_w = std::max(box_w, (int)b_hi + 8 - sx0);
            box_h = std::max(box_h, sy1 - sy0 + 1);
            t.src = sx0 | (sy0 << 16);
          }
          c->tiles.push_back(t);
        }
      box_w = (box_w + 15) & ~15;
      L.src_box_w = L.src_box_h = 0;
      if (box_w > 0 && box_w <= 256 && box_h <= 256 && box_w * box_h <= kPyrBoxBytesHost && !std::getenv("ORBX_PYR_NO_TMA"))
        L.src_box_w = box_w, L.src_box_h = box_h;
      else
        for (size_t i = first_tile; i < c->tiles.size(); ++i) c->tiles[i].src = 0;
    }
    if (l == 0) c->n_tiles0 = (int)c->tiles.size();

    // FAST cell grid (:334-362)
    const int maxBX = L.w - kEdge, maxBY = L.h - kEdge;
    const int w = maxBX - kEdge, h = maxBY - kEdge;
    L.roi_w = w;
    L.roi_h = h;
    L.n_cols = w / 30;
    L.n_rows = h / 30;
    if (L.n_cols <= 0 || L.n_rows <= 0) return fail(c, ORBX_ERR_IMAGE_SIZE, "pyramid level too small for one 30-px FAST cell");
    L.w_cell = w / L.n_cols; // ceil() of an integer quotient (:342-343)
    L.h_cell = h / L.n_rows;
    L.cell_base = cell_index;
    L.list_cap = 0;
    for (int i = 0; i < L.n_rows; ++i)
    {
      const int iniY = kEdge + i * L.h_cell;
      int maxY = iniY + L.h_cell + 6;
      if (iniY >= maxBY - 6) continue;
      if (maxY > maxBY) maxY = maxBY;
      for (int j = 0; j < L.n_cols; ++j)
      {
        const int iniX = kEdge + j * L.w_cell;
        int maxX = iniX + L.w_cell + 6;
        if (iniX >= maxBX - 6) continue;
        if (maxX > maxBX) maxX = maxBX;
        Cell ce;
        ce.level = l;
        ce.x0 = iniX;
        ce.y0 = iniY;
        ce.pw = maxX - iniX;
        ce.ph = maxY - iniY;
        if (ce.pw > kMaxPatch || ce.ph > kMaxPatch) return fail(c, ORBX_ERR_INVALID_ARG, "FAST cell patch exceeds 65 px");
        const int zw = std::max(0, ce.pw - 6), zh = std::max(0, ce.ph - 6);
        ce.cap = std::max(1, ((zw + 1) / 2) * ((zh + 1) / 2)); // strict 8-neighbour maxima cannot be denser than this
        ce.slot = (int)slot_off;
        ce.box_h = 0;
        slot_off += (size_t)ce.cap;
        L.list_cap += ce.cap;
        c->cells.push_back(ce);
        ++cell_index;
      }
    }
    L.n_level_cells = cell_index - L.cell_base;
    L.fast_box_h = 1;
    for (int ci = L.cell_base; ci < cell_index; ++ci) L.fast_box_h = std::max(L.fast_box_h, c->cells[ci].ph);
    for (int ci = L.cell_base; ci < cell_index; ++ci) c->cells[ci].box_h = L.fast_box_h; // the kernel issues its TMA load right after the cell record

    // quadtree root fan-out (initSplit :81-96)
    L.n_ini = (int)std::round((double)w / (double)h);
    if (L.n_ini > kMaxStrips) return fail(c, ORBX_ERR_INVALID_ARG, "aspect ratio too extreme (more than 255 root strips)");
    if (L.n_ini < 0) L.n_ini = 0;
    L.strip_off = (int)strips.size();
    {
      // cols = {0, (float)(1 * hX), (float)(2 * hX), ..., w} with hX = (float)(w / nIni) (:86-90); floats below 4096 have at
      // most 23 fractional bits, so the 24.40 fixed-point image is exact
      const float hX = (float)((double)w / (double)L.n_ini);
      strips.push_back(0);
      for (int k = 1; k < L.n_ini; ++k) strips.push_back((long long)std::llround(std::ldexp((double)((float)k * hX), 40)));
      strips.push_back((long long)w << 40);
    }
    L.sel_off = sel_off;
    sel_off += std::max(1, L.quota);
    L.scratch_off = (int)scratch_off;
    scratch_off += (size_t)L.list_cap * 4 + 8; // corner list + descent keys + 2 index arrays (u32 each)
    scratch_off += ((size_t)g.n_features + kMaxStrips + 8) * 8; // node bounds (4 x int64 per node, node_cap <= nFeatures + strips + 8)
    scratch_off = (scratch_off + 3) & ~(size_t)3;
    max_quota = std::max(max_quota, L.quota);
    max_ini = std::max(max_ini, L.n_ini);
  }
  if (g.width > 4080 || g.height > 4080) return fail(c, ORBX_ERR_INVALID_ARG, "images larger than 4080 px are not supported");

  Params &p = c->p;
  std::memset(&p, 0, sizeof(p));
  p.n_levels = nl;
  p.n_features = g.n_features;
  p.ini_th = g.ini_th_fast;
  p.min_th = g.min_th_fast;
  p.n_tiles = (int)c->tiles.size();
  p.n_tiles0 = c->n_tiles0;
  p.n_cells = (int)c->cells.size();
  p.width = g.width;
  p.height = g.height;
  p.pyr_img_stride = pyr_off;
  p.cell_entries = slot_off;
  p.sel_entries = sel_off;
  p.qt_scratch_img_stride = scratch_off;
  p.qt_node_cap = max_quota + max_ini + 8;
  {
    // FAST kernel: one warp per cell, each with its own slice of dynamic shared memory sized for the largest cell
    int zw = 1, zh = 1, box_h = 1;
    int area = 1;
    for (auto &ce : c->cells)
      zw = std::max(zw, ce.pw - 6), zh = std::max(zh, ce.ph - 6), box_h = std::max(box_h, ce.box_h), area = std::max(area, (ce.pw - 6) * (ce.ph - 6));
    auto up = [](int v, int a) { return (v + a - 1) / a * a; };
    // TMA box rows of 80 bytes.  Stage 1 may read up to 13 rows (+ a word) past the zone's patch: that lands in the warp's own map /
    // candidate area behind the patch (>= 1.1 KB), never outside the slice, and the flags of such rows are masked out.
    int off = up(box_h * 80, 16);
    p.fast_off_bar = off;
    off += 16;
    p.fast_map_pitch = up(zw + 2, 4);
    p.fast_off_map = off;
    off += up((zh + 2) * p.fast_map_pitch + 16, 16);
    p.fast_off_cand = off;
    off += up(area * 2, 16); // worst case: every zone pixel is a stage-1 candidate
    p.fast_off_mask = off;
    off += up(zh * 8, 16); // keep masks (one 64-bit mask per zone row)
    p.fast_off_lut = off;
    off += 64;             // the 32-entry flag-bit -> code table of the candidate expansion
    p.fast_warp_bytes = up(off, 128);
    if ((size_t)(kFastThreads / 32) * (size_t)p.fast_warp_bytes > 200 * 1024) return fail(c, ORBX_ERR_INVALID_ARG, "FAST cells too large for shared memory");
  }
  p.qt_fast = 1;
  if (const char *e = std::getenv("ORBX_QT_FAST")) p.qt_fast = std::atoi(e) != 0;
  if (p.qt_node_cap >= 60000) return fail(c, ORBX_ERR_INVALID_ARG, "n_features too large for the quadtree node pool");
  // shared-memory budget of the quadtree kernel: node pool + buckets + big-node list + keys / u16 index arrays of up to 3584 corners
  {
    int max_list = 0;
    for (auto &L : c->levels) max_list = std::max(max_list, L.list_cap);
    p.qt_big_cap = max_list / 256 + kMaxStrips + 16;
    int max_cells = 0;
    for (auto &L : c->levels) max_cells = std::max(max_cells, L.n_level_cells);
    p.qt_cell_cap = max_cells + 1;
    // Corners kept in shared memory: 3584 (4 CTAs per SM at the KITTI configuration) for images up to ~1 MP; larger images
    // produce proportionally more corners per level (~1 per 140-200 px on textured input), so they trade occupancy for a
    // list that fits: up to 160 KB per CTA.  Denser levels still work, through the global-scratch path.
    int cap = std::min(3584, std::max(2048, max_list)); // >= 2048: the second u16 index array doubles as up to 1000 int scatter cursors
    if ((long long)g.width * g.height / 140 > 3584)
    {
      const size_t fixed = quadtree_smem_bytes(0, p.qt_node_cap, p.qt_big_cap, p.qt_cell_cap);
      const size_t budget = 160 * 1024;
      if (budget > fixed + 9 * 3584) cap = std::min(max_list, (int)((budget - fixed) / 9) & ~255);
    }
    const size_t bytes = quadtree_smem_bytes(cap, p.qt_node_cap, p.qt_big_cap, p.qt_cell_cap);
    if (bytes > 200 * 1024) return fail(c, ORBX_ERR_INVALID_ARG, "n_features too large for the quadtree shared-memory pool");
    p.qt_smem_cap = cap;
    c->qt_smem = bytes;
  }
  p.fx = g.fx;
  p.fy = g.fy;
  p.cx = g.cx;
  p.cy = g.cy;
  p.bf = g.bf;
  p.depth_scale_inv = (float)(1.0 / (double)(g.depth_scale != 0.f ? g.depth_scale : 1.f)); // Mat /= s == convertTo(.., 1./s)
  for (int i = 0; i < 5; ++i) p.dist[i] = g.dist[i];
  p.undistort = g.dist[0] != 0.f ? 1 : 0; // Camera::undistortPoints returns early when k1 == 0 (src/Camera.cc:31)
  p.in_bpp = 1;
  {
    // VirtualFrame ctor (include/ORB_SLAM2/Frame.h:33-43): undistort (0,0) and (width,height); grid size (src/Frame.cc:55-56)
    float b[4] = {0.f, 0.f, (float)g.width, (float)g.height};
    if (p.undistort)
      for (int i = 0; i < 2; ++i)
      { // cv::undistortPoints with P = K: 5 fixed-point iterations in double
        const double fx = g.fx, fy = g.fy, cx = g.cx, cy = g.cy, k1 = g.dist[0], k2 = g.dist[1], p1 = g.dist[2], p2 = g.dist[3], k3 = g.dist[4];
        double x = ((double)b[2 * i] - cx) * (1. / fx), y = ((double)b[2 * i + 1] - cy) * (1. / fy);
        const double x0 = x, y0 = y;
        for (int it = 0; it < 5; ++it)
        {
          const double r2 = x * x + y * y, icd = 1. / (1 + ((k3 * r2 + k2) * r2 + k1) * r2);
          const double dx = 2 * p1 * x * y + p2 * (r2 + 2 * x * x), dy = p1 * (r2 + 2 * y * y) + 2 * p2 * x * y;
          x = (x0 - dx) * icd;
          y = (y0 - dy) * icd;
        }
        b[2 * i] = (float)(x * fx + cx);
        b[2 * i + 1] = (float)(y * fy + cy);
      }
    c->min_u = b[0];
    c->min_v = b[1];
    c->max_u = b[2];
    c->max_v = b[3];
    const float fr = (float)(c->max_v - c->min_v) / 48.f, fc = (float)(c->max_u - c->min_u) / 64.f;
    p.grid_rows = std::max(1, (int)std::ceil(fr));
    p.grid_cols = std::max(1, (int)std::ceil(fc));
    if ((long long)p.grid_rows * p.grid_cols > 10000) return fail(c, ORBX_ERR_INVALID_ARG, "undistorted image bounds are degenerate");
  }

  // pattern: float pairs -> int8 (the template file holds integers, :262)
  std::vector<char4> pat(256);
  for (int b = 0; b < 256; ++b)
  {
    float v[4];
    for (int k = 0; k < 4; ++k) v[k] = g.pattern ? g.pattern[4 * b + k] : (float)ORBX_BIT_PATTERN_31[4 * b + k];
    for (int k = 0; k < 4; ++k)
      if (v[k] != std::floor(v[k]) || std::fabs(v[k]) > 127.f) return fail(c, ORBX_ERR_INVALID_ARG, "BRIEF pattern entries must be integers in [-127,127]");
    pat[b] = make_char4((signed char)v[0], (signed char)v[1], (signed char)v[2], (signed char)v[3]);
  }
  // the rotated pattern must stay inside the 19-px border (mnBorderSize, :523)
  for (int b = 0; b < 256; ++b)
  {
    const double r1 = std::hypot((double)pat[b].x, (double)pat[b].y), r2 = std::hypot((double)pat[b].z, (double)pat[b].w);
    if (r1 > 18.5 || r2 > 18.5) return fail(c, ORBX_ERR_INVALID_ARG, "BRIEF pattern radius exceeds the 19-px border");
  }

  int rc;
  if ((rc = dev_upload(c, &p.levels, c->levels))) return rc;
  if ((rc = dev_upload(c, &p.tiles, c->tiles))) return rc;
  if ((rc = dev_upload(c, &p.cells, c->cells))) return rc;
  if ((rc = dev_upload(c, &p.tab_ofs, tab_ofs))) return rc;
  if ((rc = dev_upload(c, &p.tab_coef, tab_coef))) return rc;
  if ((rc = dev_upload(c, &p.tab_pair, tab_pair))) return rc;
  if ((rc = dev_upload(c, &p.strips_fx, strips))) return rc;
  if ((rc = dev_upload(c, &p.pattern, pat))) return rc;

  // algorithmic bytes (SURVEY.md section 8d): per image P + 60 N; stereo step 2*60 N + 352 N + 16 N
  int64_t P = 0;
  for (auto &L : c->levels) P += (int64_t)L.w * L.h;
  const int64_t N = g.n_features;
  c->alg_bytes_image = P + 60 * N;
  c->alg_bytes_stereo = 2 * c->alg_bytes_image + 120 * N + 352 * N + 16 * N;
  return ORBX_OK;
}

int alloc_buffers(orbx_ctx *c)
{
  Params &p = c->p;
  const size_t ni = (size_t)c->n_img_max, nf = (size_t)c->cfg.max_batch, N = (size_t)c->cfg.n_features;
  int rc;
  if ((rc = dev_alloc(c, &p.pyr, ni * p.pyr_img_stride))) return rc;
  if ((rc = dev_alloc(c, &p.blur, ni * p.pyr_img_stride))) return rc;
  if ((rc = dev_alloc(c, &p.cell_list, ni * p.cell_entries))) return rc;
  if ((rc = dev_alloc(c, &p.cell_cnt, ni * (size_t)p.n_cells))) return rc;
  if ((rc = dev_alloc(c, &p.sel, ni * (size_t)p.sel_entries))) return rc;
  if ((rc = dev_alloc(c, &p.sel_cnt, ni * (size_t)p.n_levels))) return rc;
  if ((rc = dev_alloc(c, &p.qt_scratch, ni * p.qt_scratch_img_stride))) return rc;
  if ((rc = dev_alloc(c, &p.kps, ni * N))) return rc;
  if ((rc = dev_alloc(c, &p.kps_und, ni * N))) return rc;
  if ((rc = dev_alloc(c, &p.desc, ni * N * 32))) return rc;
  if ((rc = dev_alloc(c, &p.n_kps, ni))) return rc;
  if ((rc = dev_alloc(c, &p.rtab, ni * N))) return rc;
  {
    // a right keypoint covers at most 2 * (2 * sf) + 2 rows (createRowIndexDB, src/ORBMatcher.cc:924-927)
    const float sf_max = c->levels.back().sf;
    p.row_cap = (int)std::min<size_t>((size_t)1 << 30, N * (size_t)(4.f * sf_max + 4.f));
    if ((rc = dev_alloc(c, &p.row_start, nf * ((size_t)c->cfg.height + 1)))) return rc;
    if ((rc = dev_alloc(c, &p.row_entries, nf * (size_t)p.row_cap))) return rc;
  }
  if ((rc = dev_alloc(c, &p.u_right, ni * N))) return rc; // sized per image so that mono batches can use it too
  if ((rc = dev_alloc(c, &p.depth, ni * N))) return rc;
  if ((rc = dev_alloc(c, &p.n_matches, ni))) return rc;
  if ((rc = dev_alloc(c, &p.grid_start, ni * ((size_t)p.grid_rows * p.grid_cols + 1)))) return rc;
  if ((rc = dev_alloc(c, &p.grid_entries, ni * N))) return rc;
  c->in_pitch = ((size_t)c->cfg.width + 15) & ~(size_t)15;
  if ((rc = dev_alloc(c, &c->d_in, ni * c->in_pitch * (size_t)c->cfg.height))) return rc;
  if ((rc = dev_alloc(c, &c->d_depth_in, nf * (size_t)c->cfg.width * (size_t)c->cfg.height * 4))) return rc;
  if ((rc = dev_alloc(c, &p.qt_stats, 16))) return rc;
  ORBX_CUDA(c, cudaMemset(p.qt_stats, 0, 16 * sizeof(unsigned long long)));
  ORBX_CUDA(c, cudaMemset(p.n_kps, 0, ni * sizeof(int)));
  ORBX_CUDA(c, cudaMemset(p.n_matches, 0, ni * sizeof(int)));
  return ORBX_OK;
}

} // namespace

namespace orbx
{

int fail(orbx_ctx *c, int code, const std::string &msg)
{
  if (c) c->last_error = msg;
  return code;
}

int require_owner(orbx_ctx *c, const orbx_ctx *owner_ctx, int owner_device, const char *what)
{
  if (owner_ctx != c || owner_device != c->device) return fail(c, ORBX_ERR_INVALID_ARG, std::string(what) + " belongs to another context");
  return ORBX_OK;
}

int resident_ctas(orbx_ctx *c, const void *kernel, int threads, size_t smem, const char *what, int *n)
{
  int per_sm = 0, n_sm = 0;
  ORBX_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
  ORBX_CUDA(c, cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, c->device));
  if (per_sm < 1) return fail(c, ORBX_ERR_CUDA, std::string(what) + " does not fit an SM");
  *n = per_sm * n_sm;
  return ORBX_OK;
}

int IoStaging::place()
{
  if (int rc = buf.reserve(c, total)) return rc;
  for (const Slice &x : slices)
  {
    x.set(buf.p + x.off);
    if (x.from) ORBX_CUDA(c, cudaMemcpyAsync(buf.p + x.off, x.from, x.bytes, cudaMemcpyHostToDevice, c->stream));
  }
  return ORBX_OK;
}

int IoStaging::finish()
{
  if (on_device) return ORBX_OK;
  for (const Slice &x : slices)
    if (x.to) ORBX_CUDA(c, cudaMemcpyAsync(x.to, buf.p + x.off, x.bytes, cudaMemcpyDeviceToHost, c->stream));
  ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
  return ORBX_OK;
}

int bow_buffers(orbx_ctx *c)
{
  if (c->bow_ready) return ORBX_OK;
  // one frame per image: a mono / RGB-D batch leaves up to n_img_max = 2 * max_batch frames resident
  const size_t F = (size_t)c->n_img_max, N = (size_t)c->cfg.n_features;
  int rc;
  if ((rc = bow_configure(c, (int)N, ORBX_ERR_CAPACITY))) return rc;
  BowArgs &b = c->bow;
  if ((rc = dev_alloc(c, &b.f_word, F * N))) return rc;
  if ((rc = dev_alloc(c, &b.f_nid, F * N))) return rc;
  if ((rc = dev_alloc(c, &b.f_weight, F * N))) return rc;
  if ((rc = dev_alloc(c, &b.bow_ids, F * N))) return rc;
  if ((rc = dev_alloc(c, &b.bow_vals, F * N))) return rc;
  if ((rc = dev_alloc(c, &b.n_bow, F))) return rc;
  if ((rc = dev_alloc(c, &b.fv_nodes, F * N))) return rc;
  if ((rc = dev_alloc(c, &b.fv_start, F * (N + 1)))) return rc;
  if ((rc = dev_alloc(c, &b.fv_feats, F * N))) return rc;
  if ((rc = dev_alloc(c, &b.n_fv, F))) return rc;
  c->bow_ready = true;
  return ORBX_OK;
}

void append_g(std::string &t, double v)
{
  char buf[64];
  t.append(buf, (size_t)std::snprintf(buf, sizeof(buf), "%g", v));
  t.push_back(' ');
}

BowArgs bow_at(const BowArgs &b, size_t frame0, size_t N)
{
  BowArgs a = b;
  a.f_word += frame0 * N, a.f_nid += frame0 * N, a.f_weight += frame0 * N;
  a.bow_ids += frame0 * N, a.bow_vals += frame0 * N, a.n_bow += frame0;
  a.fv_nodes += frame0 * N, a.fv_start += frame0 * (N + 1), a.fv_feats += frame0 * N, a.n_fv += frame0;
  return a;
}

SerArgs ser_args(const orbx_ctx *c, int image_stride, uint8_t *out, size_t stride, int64_t *sizes, uint64_t id0, const float *pose, int with_map_points)
{
  SerArgs a{};
  a.out = out, a.stride = stride, a.sizes = (long long *)sizes, a.id0 = id0, a.pose = pose, a.with_map_points = with_map_points;
  a.image_stride = image_stride;
  a.max_u = c->max_u, a.max_v = c->max_v, a.min_u = c->min_u, a.min_v = c->min_v;
  return a;
}

int DeviceBuffer::reserve(orbx_ctx *c, size_t want)
{
  if (want <= bytes) return ORBX_OK;
  if (p) ORBX_CUDA(c, cudaDeviceSynchronize());
  cudaFree(p);
  p = nullptr, bytes = 0;
  ORBX_CUDA(c, cudaMalloc((void **)&p, want));
  bytes = want;
  return ORBX_OK;
}

// Params whose per-image buffers start at image `img0` (and per-frame buffers at frame `frame0`)
Params params_at(const orbx_ctx *c, int img0, int frame0)
{
  Params p = c->p;
  p.img0 = img0;
  const size_t N = (size_t)c->cfg.n_features, i = (size_t)img0, f = (size_t)frame0;
  p.pyr += i * p.pyr_img_stride;
  p.blur += i * p.pyr_img_stride;
  p.cell_list += i * p.cell_entries;
  p.cell_cnt += i * (size_t)p.n_cells;
  p.sel += i * (size_t)p.sel_entries;
  p.sel_cnt += i * (size_t)p.n_levels;
  p.qt_scratch += i * p.qt_scratch_img_stride;
  p.kps += i * N;
  p.kps_und += i * N;
  p.desc += i * N * 32;
  p.n_kps += i;
  p.rtab += i * N;
  p.row_start += f * ((size_t)c->cfg.height + 1);
  p.row_entries += f * (size_t)p.row_cap;
  p.u_right += f * N;
  p.depth += f * N;
  p.n_matches += f;
  p.grid_start += f * ((size_t)p.grid_rows * p.grid_cols + 1);
  p.grid_entries += f * N;
  return p;
}

// records the frames now resident in the device slots (what frame-level consumers may read) and bumps frame_epoch
static void set_resident(orbx_ctx *c, int images, int frames, int stereo)
{
  c->last_images = images;
  c->last_frames = frames;
  c->last_stereo = stereo;
  ++c->frame_epoch;
}

// frame f of the resident frames reads image f * image_stride(c)
static int image_stride(const orbx_ctx *c) { return c->last_stereo ? 2 : 1; }

// The residency rule of the frame-level consumers: ORBX_OK when the images / frames / BoW of [0, end) are resident (one index
// i: end = i + 1LL), ORBX_ERR_STATE otherwise.  A BoW is resident from the orbx_bow_transform* call that covered its frame
// until the next call that produces frames.
static int require_images(orbx_ctx *c, int64_t end)
{
  if (end <= c->last_images) return ORBX_OK;
  return fail(c, ORBX_ERR_STATE, "no image with that index has been processed");
}
static int require_frames(orbx_ctx *c, int64_t end)
{
  if (end <= c->last_frames) return ORBX_OK;
  return fail(c, ORBX_ERR_STATE, "no frame with that index has been processed by the most recent stereo / RGB-D call");
}
int require_bow(orbx_ctx *c, int64_t end)
{
  if (c->bow_epoch == c->frame_epoch && end <= c->bow_frames) return ORBX_OK;
  return fail(c, ORBX_ERR_STATE, "the bag of words of that frame is not resident: call orbx_bow_transform* on the most recent call's frames first");
}

// the pipeline streams wait for the work enqueued so far on the context's stream
static int fork_pipes(orbx_ctx *c)
{
  ORBX_CUDA(c, cudaEventRecord(c->fork_ev, c->stream));
  for (int i = 0; i < c->kPipe; ++i) ORBX_CUDA(c, cudaStreamWaitEvent(c->pipe[i], c->fork_ev, 0));
  return ORBX_OK;
}

// NVTX range around the enqueue of one stage (host side; profilers correlate the launches inside it)
struct NvtxRange
{
  explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// ORBExtractor ctor + extract for n_images device-resident images on stream s; with `ev`, ev[0 .. 5] are recorded at the
// boundaries of the first five stages of orbx_stage_name
static int run_extract(orbx_ctx *c, const Params &p, int n_images, cudaStream_t s, cudaEvent_t *ev = nullptr)
{
  if (ev) ORBX_CUDA(c, cudaEventRecord(ev[0], s));
  {
    NvtxRange q("orbx:pyramid_blur");
    launch_pyramid_level0(p, n_images, s);
    if (ev) ORBX_CUDA(c, cudaEventRecord(ev[1], s));
    launch_pyramid_levels(p, c->maps_src, n_images, s);
  }
  if (ev) ORBX_CUDA(c, cudaEventRecord(ev[2], s));
  {
    NvtxRange q("orbx:fast_cells");
    launch_fast(p, c->maps, n_images, s);
  }
  if (ev) ORBX_CUDA(c, cudaEventRecord(ev[3], s));
  {
    NvtxRange q("orbx:quadtree");
    launch_quadtree(p, n_images, c->qt_smem, s);
  }
  if (ev) ORBX_CUDA(c, cudaEventRecord(ev[4], s));
  {
    NvtxRange q("orbx:orient_brief");
    launch_orient_brief(p, c->maps_blur, n_images, s);
  }
  if (ev) ORBX_CUDA(c, cudaEventRecord(ev[5], s));
  c->launches += 5;
  ORBX_CUDA(c, cudaGetLastError());
  return ORBX_OK;
}

// the Params of a stereo batch whose first frame is device slot d0, reading its images at d_left / d_right
static Params stereo_params(const orbx_ctx *c, int d0, const uint8_t *d_left, const uint8_t *d_right, size_t stride, size_t frame_stride)
{
  Params p = params_at(c, 2 * d0, d0);
  p.stereo = 1;
  p.in_left = d_left;
  p.in_right = d_right;
  p.in_stride = stride;
  p.in_frame_stride = frame_stride;
  return p;
}

// the kernels of a stereo batch for device slots [frame0, frame0 + nf) on stream s (inputs: frame 0 of the range at d_left /
// d_right); with `ev`, ev[0 .. ORBX_N_STAGES] are recorded on s at the stage boundaries of orbx_stage_name
static int run_stereo_range(orbx_ctx *c, cudaStream_t s, int frame0, int nf, const uint8_t *d_left, const uint8_t *d_right, size_t stride, size_t frame_stride,
                            cudaEvent_t *ev = nullptr)
{
  const Params p = stereo_params(c, frame0, d_left, d_right, stride, frame_stride);
  NvtxRange r("orbx:stereo_range");
  ORBX_CUDA(c, cudaMemsetAsync(p.n_matches, 0, (size_t)nf * sizeof(int), s));
  int rc = run_extract(c, p, 2 * nf, s, ev);
  if (rc) return rc;
  {
    NvtxRange q("orbx:frame_index"); // createRowIndexDB of the right keypoints + initGrid of the left ones, one launch
    launch_frame_index(p, nf, 2, true, s);
  }
  if (ev) ORBX_CUDA(c, cudaEventRecord(ev[6], s));
  {
    NvtxRange q("orbx:stereo_match");
    launch_stereo(p, nf, s);
  }
  if (ev) ORBX_CUDA(c, cudaEventRecord(ev[7], s));
  c->launches += 2;
  ORBX_CUDA(c, cudaGetLastError());
  return ORBX_OK;
}

static void drop_graph(orbx_ctx *c)
{
  if (c->graph1_exec) cudaGraphExecDestroy(c->graph1_exec);
  if (c->graph1) cudaGraphDestroy(c->graph1);
  c->graph1_exec = nullptr;
  c->graph1 = nullptr;
  c->graph1_pyr = nullptr;
}

// one stereo frame in device slot 0: a single graph launch when the context's graph is enabled and `s` can be captured
static int run_stereo_single(orbx_ctx *c, cudaStream_t s, const uint8_t *d_left, const uint8_t *d_right, size_t stride, size_t frame_stride)
{
  // the legacy / per-thread default streams cannot be captured
  const bool can = c->use_graph && s != nullptr && s != cudaStreamLegacy && s != cudaStreamPerThread;
  if (!can) return run_stereo_range(c, s, 0, 1, d_left, d_right, stride, frame_stride);
  if (!c->graph1_exec)
  {
    const int64_t before = c->launches;
    if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) != cudaSuccess)
    { // e.g. the caller is capturing this stream already: plain launches
      (void)cudaGetLastError();
      return run_stereo_range(c, s, 0, 1, d_left, d_right, stride, frame_stride);
    }
    const int rc = run_stereo_range(c, s, 0, 1, d_left, d_right, stride, frame_stride);
    const cudaError_t e = cudaStreamEndCapture(s, &c->graph1);
    c->graph1_kernels = (int)(c->launches - before);
    c->launches = before;
    if (rc != ORBX_OK || e != cudaSuccess || cudaGraphInstantiate(&c->graph1_exec, c->graph1, 0) != cudaSuccess)
    {
      (void)cudaGetLastError();
      drop_graph(c);
      c->use_graph = 0;
      return run_stereo_range(c, s, 0, 1, d_left, d_right, stride, frame_stride);
    }
    size_t n = 0;
    cudaGraphGetNodes(c->graph1, nullptr, &n);
    std::vector<cudaGraphNode_t> nodes(n);
    cudaGraphGetNodes(c->graph1, nodes.data(), &n);
    for (auto nd : nodes)
    {
      cudaGraphNodeType t;
      cudaKernelNodeParams kp;
      if (cudaGraphNodeGetType(nd, &t) == cudaSuccess && t == cudaGraphNodeTypeKernel && cudaGraphKernelNodeGetParams(nd, &kp) == cudaSuccess &&
          kp.func == pyramid_kernel_symbol(c->p.in_bpp))
        c->graph1_pyr = nd;
    }
    if (!c->graph1_pyr)
    {
      drop_graph(c);
      c->use_graph = 0;
      return run_stereo_range(c, s, 0, 1, d_left, d_right, stride, frame_stride);
    }
    c->graph1_left = d_left, c->graph1_right = d_right, c->graph1_stride = stride, c->graph1_fs = frame_stride;
  }
  else if (d_left != c->graph1_left || d_right != c->graph1_right || stride != c->graph1_stride || frame_stride != c->graph1_fs)
  {
    // only the pyramid kernel reads the caller's images: patch that node's Params in the instantiated graph
    cudaKernelNodeParams kp;
    ORBX_CUDA(c, cudaGraphKernelNodeGetParams(c->graph1_pyr, &kp));
    Params p = stereo_params(c, 0, d_left, d_right, stride, frame_stride);
    void *args[1] = {&p};
    kp.kernelParams = args;
    kp.extra = nullptr;
    ORBX_CUDA(c, cudaGraphExecKernelNodeSetParams(c->graph1_exec, c->graph1_pyr, &kp));
    c->graph1_left = d_left, c->graph1_right = d_right, c->graph1_stride = stride, c->graph1_fs = frame_stride;
  }
  ORBX_CUDA(c, cudaGraphLaunch(c->graph1_exec, s));
  c->launches += c->graph1_kernels;
  return ORBX_OK;
}

int run_stereo_chunks(orbx_ctx *c, int64_t n_frames, const uint8_t *left, size_t left_stride, const uint8_t *right, size_t right_stride, size_t frame_stride,
                      bool on_device, bool piped, const ChunkOut &out)
{
  const size_t W = (size_t)c->cfg.width * (size_t)c->p.in_bpp, H = (size_t)c->cfg.height; // row bytes
  if (std::min(left_stride, right_stride) < W || frame_stride < std::max(left_stride, right_stride) * (H - 1) + W)
    return fail(c, ORBX_ERR_INVALID_ARG, "stride / frame_stride smaller than the image");
  // Densely stacked rows that fit the staging pitch are copied as ONE linear transfer per side and read on the device
  // with the caller's stride (the kernels gather bytes, so rows need no alignment); 2-D pitched copies of odd-width
  // rows run at a fraction of the PCIe rate.
  const bool linear = left_stride == right_stride && frame_stride == left_stride * H && left_stride <= c->in_pitch;
  const size_t fs = linear ? frame_stride : c->in_pitch * H, dstride = linear ? left_stride : c->in_pitch;
  uint8_t *dl = c->d_in, *dr = c->d_in + (size_t)c->cfg.max_batch * c->in_pitch * H;
  // A slot is always driven by the same pipeline stream, so reusing it is ordered by that stream while the H2D copy of one
  // chunk, the kernels of another and the D2H copy of a third overlap across streams.
  const int chunk = c->chunk(), n_slots = std::max(1, c->cfg.max_batch / chunk);
  if (piped)
  {
    int rc = fork_pipes(c);
    if (rc) return rc;
  }
  int k = 0;
  for (int64_t f0 = 0; f0 < n_frames; f0 += chunk, ++k)
  {
    const int nf = (int)std::min<int64_t>(chunk, n_frames - f0);
    const int slot = k % n_slots, d0 = slot * chunk;
    cudaStream_t s = piped ? c->pipe[slot % c->kPipe] : c->stream;
    const uint8_t *in_l = left + (size_t)f0 * frame_stride, *in_r = right + (size_t)f0 * frame_stride;
    size_t in_stride = left_stride, in_fs = frame_stride;
    if (!on_device)
    { // device inputs are read in place: only the intermediate buffers cycle through the slots
      uint8_t *sl = dl + (size_t)d0 * fs, *sr = dr + (size_t)d0 * fs;
      if (linear)
      {
        ORBX_CUDA(c, cudaMemcpyAsync(sl, in_l, fs * nf, cudaMemcpyHostToDevice, s));
        ORBX_CUDA(c, cudaMemcpyAsync(sr, in_r, fs * nf, cudaMemcpyHostToDevice, s));
      }
      else
        for (int f = 0; f < nf; ++f)
        {
          ORBX_CUDA(c, cudaMemcpy2DAsync(sl + f * fs, c->in_pitch, in_l + f * frame_stride, left_stride, W, H, cudaMemcpyHostToDevice, s));
          ORBX_CUDA(c, cudaMemcpy2DAsync(sr + f * fs, c->in_pitch, in_r + f * frame_stride, right_stride, W, H, cudaMemcpyHostToDevice, s));
        }
      in_l = sl, in_r = sr, in_stride = dstride, in_fs = fs;
    }
    // a single frame on the context's stream is the latency path
    int rc = n_frames == 1 && !piped ? run_stereo_single(c, s, in_l, in_r, in_stride, in_fs) : run_stereo_range(c, s, d0, nf, in_l, in_r, in_stride, in_fs);
    if (!rc) rc = out(s, d0, f0, nf);
    if (rc) return rc;
  }
  // introspection (get_pyramid / get_grid) refers to the device slots, i.e. to the frames of the last pass over them
  const int resident = (int)std::min<int64_t>(n_frames, (int64_t)n_slots * chunk);
  set_resident(c, 2 * resident, resident, 1);
  return ORBX_OK;
}

} // namespace orbx

namespace
{

// TMA descriptors: one 3-D byte tensor {pitch, rows, images} per pyramid level over the context's pyr buffer, box = the
// level's largest FAST patch (80 bytes wide = the shared-memory patch pitch).  cuTensorMapEncodeTiled is a driver entry point.
int build_level_maps(orbx_ctx *c)
{
  typedef CUresult (*EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                               const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  void *fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  ORBX_CUDA(c, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) return fail(c, ORBX_ERR_CUDA, "cuTensorMapEncodeTiled is not available");
  // FAST: box = 80 bytes x the level's tallest patch over `pyr`; BRIEF: box = 64 bytes x 37 rows (the blurred patch a rotated
  // pattern can reach) over `blur`
  std::memset(&c->maps, 0, sizeof(c->maps));
  std::memset(&c->maps_blur, 0, sizeof(c->maps_blur));
  std::memset(&c->maps_src, 0, sizeof(c->maps_src));
  for (size_t l = 0; l < c->levels.size(); ++l)
  {
    const Level &L = c->levels[l];
    const cuuint64_t dims[3] = {(cuuint64_t)L.pitch, (cuuint64_t)L.h, (cuuint64_t)c->n_img_max};
    const cuuint64_t strides[2] = {(cuuint64_t)L.pitch, (cuuint64_t)c->p.pyr_img_stride};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    const cuuint32_t box[3] = {80u, (cuuint32_t)L.fast_box_h, 1u};
    CUresult r = ((EncodeFn)fn)(&c->maps.m[l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, c->p.pyr + L.pyr_off, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(c, ORBX_ERR_CUDA, "cuTensorMapEncodeTiled failed for level " + std::to_string(l));
    if (L.src_box_w)
    { // level-0 source rectangles of this level's tiles: the tensor is level 0 of `pyr`
      const Level &L0 = c->levels[0];
      const cuuint64_t dims0[3] = {(cuuint64_t)L0.pitch, (cuuint64_t)L0.h, (cuuint64_t)c->n_img_max};
      const cuuint64_t strides0[2] = {(cuuint64_t)L0.pitch, (cuuint64_t)c->p.pyr_img_stride};
      const cuuint32_t box_s[3] = {(cuuint32_t)L.src_box_w, (cuuint32_t)L.src_box_h, 1u};
      r = ((EncodeFn)fn)(&c->maps_src.m[l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, c->p.pyr + L0.pyr_off, dims0, strides0, box_s, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(c, ORBX_ERR_CUDA, "cuTensorMapEncodeTiled (resize source) failed for level " + std::to_string(l));
    }
    const cuuint32_t box_b[3] = {64u, 37u, 1u};
    r = ((EncodeFn)fn)(&c->maps_blur.m[l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, c->p.blur + L.pyr_off, dims, strides, box_b, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(c, ORBX_ERR_CUDA, "cuTensorMapEncodeTiled (blur) failed for level " + std::to_string(l));
  }
  c->p.img0 = 0;
  return ORBX_OK;
}

void fill_results(orbx_ctx *c, int n_images, int n_frames, orbx_device_results *out)
{
  if (!out) return;
  out->kps = c->p.kps;
  out->kps_und = c->p.kps_und;
  out->desc = c->p.desc;
  out->n_kps = c->p.n_kps;
  out->u_right = c->p.u_right;
  out->depth = c->p.depth;
  out->n_matches = c->p.n_matches;
  out->n_images = n_images;
  out->n_frames = n_frames;
  out->n_features = c->cfg.n_features;
  out->grid_start = c->p.grid_start;
  out->grid_entries = c->p.grid_entries;
  out->grid_rows = c->p.grid_rows;
  out->grid_cols = c->p.grid_cols;
}

} // namespace

extern "C"
{

  void orbx_default_config(orbx_config *cfg)
  {
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->width = 1241;
    cfg->height = 376;
    cfg->n_features = 2000;
    cfg->n_levels = 8;
    cfg->scale_factor = 1.2f;
    cfg->ini_th_fast = 20;
    cfg->min_th_fast = 7;
    cfg->fx = 718.856f;
    cfg->fy = 718.856f;
    cfg->cx = 607.1928f;
    cfg->cy = 185.2157f;
    cfg->bf = cfg->fx * 0.537166f;
    cfg->depth_scale = 1.f;
    cfg->max_batch = 1;
    cfg->device = -1;
    cfg->pattern = nullptr;
  }

  const char *orbx_status_string(int status)
  {
    switch (status)
    {
    case ORBX_OK: return "ok";
    case ORBX_ERR_INVALID_ARG: return "invalid argument";
    case ORBX_ERR_IMAGE_SIZE: return "ImageSizeError: pyramid level too small";
    case ORBX_ERR_FILE_NOT_OPEN: return "FileNotOpenError: cannot open BRIEF template";
    case ORBX_ERR_CUDA: return "CUDA error";
    case ORBX_ERR_NO_DEVICE: return "no CUDA device";
    case ORBX_ERR_CAPACITY: return "batch larger than max_batch";
    case ORBX_ERR_STATE: return "invalid state";
    case ORBX_ERR_COMM: return "communicator error (NCCL / peer memory)";
    default: return "unknown status";
    }
  }

  int orbx_load_brief_template(const char *path, float *pattern_out)
  {
    if (!path || !pattern_out) return ORBX_ERR_INVALID_ARG;
    std::ifstream ifs(path);
    if (!ifs.is_open()) return ORBX_ERR_FILE_NOT_OPEN;
    std::string line;
    bool header = true;
    int n = 0;
    while (std::getline(ifs, line))
    {
      if (header)
      { // first line is a column header (:255-259)
        header = false;
        continue;
      }
      if (n >= 256) break;
      std::istringstream iss(line);
      float v[4] = {0, 0, 0, 0};
      iss >> v[0] >> v[1] >> v[2] >> v[3];
      for (int k = 0; k < 4; ++k) pattern_out[4 * n + k] = v[k];
      ++n;
    }
    return n == 256 ? ORBX_OK : ORBX_ERR_INVALID_ARG;
  }

  int orbx_create(const orbx_config *cfg, orbx_ctx **out)
  {
    if (!cfg || !out) return ORBX_ERR_INVALID_ARG;
    *out = nullptr;
    if (cfg->width <= 0 || cfg->height <= 0 || cfg->n_features < 1 || cfg->n_levels < 1 || cfg->n_levels > kMaxLevels || !(cfg->scale_factor > 1.f) ||
        cfg->ini_th_fast < 0 || cfg->ini_th_fast > 255 || cfg->min_th_fast < 0 || cfg->min_th_fast > 255 || cfg->max_batch < 1)
      return ORBX_ERR_INVALID_ARG;
    if (cfg->n_features > 65535) return ORBX_ERR_INVALID_ARG; // keypoint indices travel as uint16 in the row index and the grid CSR
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return ORBX_ERR_NO_DEVICE; // no CPU fallback, by design
    orbx_ctx *c = new (std::nothrow) orbx_ctx();
    if (!c) return ORBX_ERR_INVALID_ARG;
    c->cfg = *cfg;
    c->cfg.pattern = cfg->pattern;
    int rc = ORBX_OK;
    do
    {
      if (cfg->device >= 0)
      {
        if (cfg->device >= ndev)
        {
          rc = ORBX_ERR_NO_DEVICE;
          break;
        }
        if (cudaSetDevice(cfg->device) != cudaSuccess)
        {
          rc = ORBX_ERR_CUDA;
          break;
        }
      }
      if (cudaGetDevice(&c->device) != cudaSuccess)
      {
        rc = ORBX_ERR_CUDA;
        break;
      }
      c->n_img_max = 2 * cfg->max_batch;
      if ((rc = build_tables(c))) break;
      c->cfg.pattern = nullptr; // not retained
      if ((rc = alloc_buffers(c))) break;
      if ((rc = build_level_maps(c))) break;
      if (fast_configure(c->p) != 0)
      {
        rc = fail(c, ORBX_ERR_CUDA, "cudaFuncSetAttribute(fast_cells_kernel, MaxDynamicSharedMemorySize)");
        break;
      }
      if (frame_index_configure(c->p) != 0)
      {
        rc = fail(c, ORBX_ERR_CUDA, "cudaFuncSetAttribute(frame_index_kernel, MaxDynamicSharedMemorySize)");
        break;
      }
      if (quadtree_configure(c->qt_smem) != 0)
      {
        rc = fail(c, ORBX_ERR_CUDA, "cudaFuncSetAttribute(quadtree_kernel, MaxDynamicSharedMemorySize)");
        break;
      }
      if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess)
      {
        rc = ORBX_ERR_CUDA;
        break;
      }
      c->stream = c->own_stream;
      if (const char *e = std::getenv("ORBX_GRAPH")) c->use_graph = std::atoi(e) != 0;
      if (const char *e = std::getenv("ORBX_PIPE")) c->kPipe = std::max(1, std::min(orbx_ctx::kPipeMax, std::atoi(e)));
      if (const char *e = std::getenv("ORBX_CHUNK")) c->kChunk = std::max(1, std::atoi(e));
      for (int i = 0; i < c->kPipe; ++i)
        if (cudaStreamCreateWithFlags(&c->pipe[i], cudaStreamNonBlocking) != cudaSuccess) rc = ORBX_ERR_CUDA;
      if (cudaEventCreateWithFlags(&c->fork_ev, cudaEventDisableTiming) != cudaSuccess) rc = ORBX_ERR_CUDA;
      for (int i = 0; i < c->kPipe; ++i)
        if (cudaEventCreateWithFlags(&c->join_ev[i], cudaEventDisableTiming) != cudaSuccess) rc = ORBX_ERR_CUDA;
    } while (0);
    if (rc != ORBX_OK)
    {
      if (!c->last_error.empty()) std::fprintf(stderr, "orbx_create: %s\n", c->last_error.c_str());
      orbx_destroy(c);
      return rc;
    }
    *out = c;
    return ORBX_OK;
  }

  void orbx_destroy(orbx_ctx *c)
  {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->own_stream)
    {
      cudaStreamSynchronize(c->own_stream);
      cudaStreamDestroy(c->own_stream);
    }
    for (auto &ps : c->pipe)
      if (ps)
      {
        cudaStreamSynchronize(ps);
        cudaStreamDestroy(ps);
      }
    if (c->fork_ev) cudaEventDestroy(c->fork_ev);
    for (auto &je : c->join_ev)
      if (je) cudaEventDestroy(je);
    for (void *q : c->allocs) cudaFree(q);
    drop_graph(c);
    destroy_self_comm(c);
    if (c->h_rec1) cudaFreeHost(c->h_rec1);
    delete c; // frees the DeviceBuffers
  }

  const char *orbx_last_error(const orbx_ctx *c) { return c ? c->last_error.c_str() : ""; }

  int orbx_set_stream(orbx_ctx *c, void *cuda_stream)
  {
    if (!c) return ORBX_ERR_INVALID_ARG;
    c->stream = cuda_stream ? (cudaStream_t)cuda_stream : c->own_stream;
    return ORBX_OK;
  }

  int orbx_set_graph(orbx_ctx *c, int enable)
  {
    if (!c) return ORBX_ERR_INVALID_ARG;
    c->use_graph = enable != 0;
    return ORBX_OK;
  }

  int orbx_set_input_format(orbx_ctx *c, int format)
  {
    if (!c) return ORBX_ERR_INVALID_ARG;
    // gray weights of bytes 0, 1, 2 of a pixel (cv::cvtColor, 8-bit: R 9798, G 19235, B 3735, 15 fractional bits)
    int bpp = 0;
    uint32_t w0 = 0, w2 = 0;
    switch (format)
    {
    case ORBX_FORMAT_GRAY8: bpp = 1; break;
    case ORBX_FORMAT_RGB8: bpp = 3, w0 = 9798, w2 = 3735; break;
    case ORBX_FORMAT_BGR8: bpp = 3, w0 = 3735, w2 = 9798; break;
    case ORBX_FORMAT_RGBA8: bpp = 4, w0 = 9798, w2 = 3735; break;
    case ORBX_FORMAT_BGRA8: bpp = 4, w0 = 3735, w2 = 9798; break;
    default: return fail(c, ORBX_ERR_INVALID_ARG, "unknown input format");
    }
    if (format == c->in_format) return ORBX_OK;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    const size_t pitch = ((size_t)c->cfg.width * bpp + 15) & ~(size_t)15;
    if (pitch > c->in_pitch)
    { // the host staging grows; work of earlier calls may still read the old buffer
      uint8_t *q = nullptr;
      ORBX_CUDA(c, cudaDeviceSynchronize());
      ORBX_CUDA(c, cudaMalloc((void **)&q, (size_t)c->n_img_max * pitch * (size_t)c->cfg.height + 256));
      std::replace(c->allocs.begin(), c->allocs.end(), (void *)c->d_in, (void *)q);
      cudaFree(c->d_in);
      c->d_in = q;
      c->in_pitch = pitch;
    }
    drop_graph(c); // the captured level-0 node is the kernel of the old format
    c->in_format = format;
    c->p.in_bpp = bpp;
    c->p.cvt_w01 = w0 | (19235u << 16);
    c->p.cvt_w2 = w2;
    return ORBX_OK;
  }

  int orbx_num_levels(const orbx_ctx *c) { return c ? c->cfg.n_levels : ORBX_ERR_INVALID_ARG; }

  int orbx_level_info(const orbx_ctx *c, int level, int32_t *width, int32_t *height, float *scale, int32_t *quota)
  {
    if (!c || level < 0 || level >= c->cfg.n_levels) return ORBX_ERR_INVALID_ARG;
    const Level &L = c->levels[level];
    if (width) *width = L.w;
    if (height) *height = L.h;
    if (scale) *scale = L.sf;
    if (quota) *quota = L.quota;
    return ORBX_OK;
  }

  int orbx_synchronize(orbx_ctx *c)
  {
    if (!c) return ORBX_ERR_INVALID_ARG;
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    return ORBX_OK;
  }

  int orbx_read_device(orbx_ctx *c, const void *device_ptr, void *host_dst, size_t bytes)
  {
    if (!c || !device_ptr || !host_dst) return ORBX_ERR_INVALID_ARG;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    ORBX_CUDA(c, cudaMemcpy(host_dst, device_ptr, bytes, cudaMemcpyDeviceToHost));
    return ORBX_OK;
  }

  int64_t orbx_launch_count(const orbx_ctx *c) { return c ? c->launches : 0; }
  uint64_t orbx_frame_epoch(const orbx_ctx *c) { return c ? c->frame_epoch : 0; }
  int64_t orbx_algorithmic_bytes(const orbx_ctx *c, int stereo)
  {
    if (!c) return 0;
    // a colour context reads bpp bytes per level-0 pixel instead of one
    const int64_t extra = (int64_t)(c->p.in_bpp - 1) * c->cfg.width * c->cfg.height * (stereo ? 2 : 1);
    return (stereo ? c->alg_bytes_stereo : c->alg_bytes_image) + extra;
  }

  // ---------------------------------------------------------------------------------------------------------------
  int orbx_extract_batch_device(orbx_ctx *c, int n_images, const uint8_t *d_images, size_t stride, size_t frame_stride, orbx_device_results *out)
  {
    if (!c || !d_images || n_images < 1) return ORBX_ERR_INVALID_ARG;
    if (n_images > c->n_img_max) return fail(c, ORBX_ERR_CAPACITY, "n_images > 2 * max_batch");
    ORBX_CUDA(c, cudaSetDevice(c->device));
    Params p = c->p;
    p.stereo = 0;
    p.in_left = d_images;
    p.in_right = nullptr;
    p.in_stride = stride;
    p.in_frame_stride = frame_stride;
    int rc = run_extract(c, p, n_images, c->stream);
    if (rc) return rc;
    set_resident(c, n_images, 0, 0); // extract-only images carry no grid / uRight / depth: frame-level consumers must fail with ORBX_ERR_STATE
    fill_results(c, n_images, 0, out);
    return ORBX_OK;
  }

  int orbx_stereo_batch_device(orbx_ctx *c, int n_frames, const uint8_t *d_left, const uint8_t *d_right, size_t stride, size_t frame_stride,
                               orbx_device_results *out)
  {
    if (!c || !d_left || !d_right || n_frames < 1) return ORBX_ERR_INVALID_ARG;
    if (n_frames > c->cfg.max_batch) return fail(c, ORBX_ERR_CAPACITY, "n_frames > max_batch");
    ORBX_CUDA(c, cudaSetDevice(c->device));
    if (n_frames == 1)
    {
      int rc = run_stereo_single(c, c->stream, d_left, d_right, stride, frame_stride);
      if (rc) return rc;
    }
    else if (n_frames <= c->kChunk)
    {
      int rc = run_stereo_range(c, c->stream, 0, n_frames, d_left, d_right, stride, frame_stride);
      if (rc) return rc;
    }
    else
    {
      // Fork the batch into chunks on the pipeline streams and join back into the caller's stream: the latency-bound
      // quadtree launches of one chunk then overlap the issue-bound FAST / pyramid launches of the others.  Every frame
      // keeps its own slot (slot = frame), so all of them stay resident.
      int rc = fork_pipes(c);
      if (rc) return rc;
      int k = 0;
      for (int f0 = 0; f0 < n_frames; f0 += c->kChunk, ++k)
      {
        rc = run_stereo_range(c, c->pipe[k % c->kPipe], f0, std::min(c->kChunk, n_frames - f0), d_left + (size_t)f0 * frame_stride,
                              d_right + (size_t)f0 * frame_stride, stride, frame_stride);
        if (rc) return rc;
      }
      for (int i = 0; i < c->kPipe; ++i)
      {
        ORBX_CUDA(c, cudaEventRecord(c->join_ev[i], c->pipe[i]));
        ORBX_CUDA(c, cudaStreamWaitEvent(c->stream, c->join_ev[i], 0));
      }
    }
    set_resident(c, 2 * n_frames, n_frames, 1);
    fill_results(c, 2 * n_frames, n_frames, out);
    return ORBX_OK;
  }

  const char *orbx_stage_name(int stage)
  {
    static const char *names[ORBX_N_STAGES] = {"pyramid_level0", "pyramid_levels", "fast_cells", "quadtree", "orient_brief", "frame_index", "stereo_match"};
    return (stage >= 0 && stage < ORBX_N_STAGES) ? names[stage] : "";
  }

  int orbx_profile_stereo_batch_device(orbx_ctx *c, int n_frames, const uint8_t *d_left, const uint8_t *d_right, size_t stride, size_t frame_stride,
                                       float *stage_ms)
  {
    if (!c || !d_left || !d_right || n_frames < 1 || !stage_ms) return ORBX_ERR_INVALID_ARG;
    if (n_frames > c->cfg.max_batch) return fail(c, ORBX_ERR_CAPACITY, "n_frames > max_batch");
    ORBX_CUDA(c, cudaSetDevice(c->device));
    cudaEvent_t ev[ORBX_N_STAGES + 1];
    for (auto &e : ev) ORBX_CUDA(c, cudaEventCreate(&e));
    // one launch per kernel over all n_frames on the context's stream (not the chunked fork of orbx_stereo_batch_device)
    int rc = run_stereo_range(c, c->stream, 0, n_frames, d_left, d_right, stride, frame_stride, ev);
    if (rc) return rc;
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < ORBX_N_STAGES; ++i) ORBX_CUDA(c, cudaEventElapsedTime(&stage_ms[i], ev[i], ev[i + 1]));
    for (auto &e : ev) cudaEventDestroy(e);
    set_resident(c, 2 * n_frames, n_frames, 1);
    return ORBX_OK;
  }

  int orbx_rgbd_batch_device(orbx_ctx *c, int n_frames, const uint8_t *d_gray, size_t gray_stride, size_t gray_frame_stride, const void *d_depth,
                             size_t depth_stride_bytes, size_t depth_frame_stride_bytes, int depth_type, orbx_device_results *out)
  {
    if (!c || !d_gray || !d_depth || n_frames < 1 || (depth_type != ORBX_DEPTH_U16 && depth_type != ORBX_DEPTH_F32)) return ORBX_ERR_INVALID_ARG;
    if (n_frames > c->n_img_max) return fail(c, ORBX_ERR_CAPACITY, "n_frames > 2 * max_batch");
    // rgbd_kernel loads whole elements at depth + f * frame_stride + y * stride: a misaligned address would fault
    const size_t esz = depth_type == ORBX_DEPTH_F32 ? 4 : 2, W = (size_t)c->cfg.width, H = (size_t)c->cfg.height;
    if ((size_t)d_depth % esz || depth_stride_bytes % esz || depth_frame_stride_bytes % esz)
      return fail(c, ORBX_ERR_INVALID_ARG, "depth pointer, stride and frame stride must be multiples of the depth element size");
    if (depth_stride_bytes < W * esz || (n_frames > 1 && depth_frame_stride_bytes < depth_stride_bytes * (H - 1) + W * esz))
      return fail(c, ORBX_ERR_INVALID_ARG, "depth stride / frame stride smaller than the depth image");
    ORBX_CUDA(c, cudaSetDevice(c->device));
    Params p = c->p;
    p.stereo = 0;
    p.in_left = d_gray;
    p.in_stride = gray_stride;
    p.in_frame_stride = gray_frame_stride;
    p.depth_img = d_depth;
    p.depth_stride = depth_stride_bytes;
    p.depth_frame_stride = depth_frame_stride_bytes;
    p.depth_type = depth_type;
    int rc = run_extract(c, p, n_frames, c->stream);
    if (rc) return rc;
    ORBX_CUDA(c, cudaMemsetAsync(p.n_matches, 0, (size_t)n_frames * sizeof(int), c->stream));
    launch_rgbd(p, n_frames, c->stream);
    launch_frame_index(p, n_frames, 1, false, c->stream);
    c->launches += 2;
    ORBX_CUDA(c, cudaGetLastError());
    set_resident(c, n_frames, n_frames, 0);
    fill_results(c, n_frames, n_frames, out);
    return ORBX_OK;
  }

  // ---------------------------------------------------------------------------------------------------------------
  // Latency path (the reference's one-frame-at-a-time call): both images staged into slot 0, ONE graph launch, the frame's
  // results packed into one record on the device and brought back in ONE copy (instead of nine), then handed out from
  // pinned memory.
  static int stereo_frame_host(orbx_ctx *c, const uint8_t *left, size_t left_stride, const uint8_t *right, size_t right_stride, size_t frame_stride,
                               orbx_keypoint *kps_left, uint8_t *desc_left, int32_t *n_left, orbx_keypoint *kps_right, uint8_t *desc_right,
                               int32_t *n_right, double *u_right, double *depth, int32_t *n_matches)
  {
    ORBX_CUDA(c, cudaSetDevice(c->device));
    orbx_record_layout lay;
    orbx_record_layout_get(c, &lay);
    const size_t rs = (size_t)lay.record_bytes;
    int rc = c->rec_staging.reserve(c, (size_t)c->cfg.max_batch * rs);
    if (rc) return rc;
    if (!c->h_rec1) ORBX_CUDA(c, cudaHostAlloc((void **)&c->h_rec1, rs, cudaHostAllocDefault));
    rc = run_stereo_chunks(c, 1, left, left_stride, right, right_stride, frame_stride, false, false, [&](cudaStream_t s, int, int64_t, int) -> int {
      const int prc = pack_frame_records(c, s, 0, 1, c->rec_staging.p, rs);
      if (prc) return prc;
      ORBX_CUDA(c, cudaMemcpyAsync(c->h_rec1, c->rec_staging.p, rs, cudaMemcpyDeviceToHost, s));
      return ORBX_OK;
    });
    if (rc) return rc;
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    const int32_t *hdr = reinterpret_cast<const int32_t *>(c->h_rec1);
    const size_t nl = (size_t)hdr[0], nr = (size_t)hdr[1];
    if (kps_left) std::memcpy(kps_left, c->h_rec1 + lay.off_kps_left, nl * sizeof(orbx_keypoint));
    if (desc_left) std::memcpy(desc_left, c->h_rec1 + lay.off_desc_left, nl * 32);
    if (n_left) *n_left = hdr[0];
    if (kps_right) std::memcpy(kps_right, c->h_rec1 + lay.off_kps_right, nr * sizeof(orbx_keypoint));
    if (desc_right) std::memcpy(desc_right, c->h_rec1 + lay.off_desc_right, nr * 32);
    if (n_right) *n_right = hdr[1];
    if (u_right) std::memcpy(u_right, c->h_rec1 + lay.off_u_right, nl * 8);
    if (depth) std::memcpy(depth, c->h_rec1 + lay.off_depth, nl * 8);
    if (n_matches) *n_matches = hdr[2];
    return ORBX_OK;
  }

  int orbx_stereo_batch(orbx_ctx *c, int n_frames, const uint8_t *left, const uint8_t *right, size_t stride, size_t frame_stride, orbx_keypoint *kps_left,
                        uint8_t *desc_left, int32_t *n_left, orbx_keypoint *kps_right, uint8_t *desc_right, int32_t *n_right, double *u_right,
                        double *depth, int32_t *n_matches)
  {
    if (!c || !left || !right || n_frames < 1) return ORBX_ERR_INVALID_ARG;
    if (n_frames == 1)
      return stereo_frame_host(c, left, stride, right, stride, frame_stride, kps_left, desc_left, n_left, kps_right, desc_right, n_right, u_right, depth,
                               n_matches);
    ORBX_CUDA(c, cudaSetDevice(c->device));
    const size_t N = (size_t)c->cfg.n_features, kb = N * sizeof(orbx_keypoint), db = N * 32;
    const Params &p = c->p;
    // a batch that fits one chunk runs on the context's stream
    const bool piped = n_frames > c->chunk();
    int rc = run_stereo_chunks(c, n_frames, left, stride, right, stride, frame_stride, false, piped, [&](cudaStream_t s, int d0, int64_t f0, int nf) -> int {
      // results: left = even images, right = odd images -> one strided 2-D copy per array
      const size_t i0 = 2 * (size_t)d0;
      if (kps_left) ORBX_CUDA(c, cudaMemcpy2DAsync(kps_left + f0 * N, kb, p.kps_und + i0 * N, 2 * kb, kb, nf, cudaMemcpyDeviceToHost, s));
      if (kps_right) ORBX_CUDA(c, cudaMemcpy2DAsync(kps_right + f0 * N, kb, p.kps + (i0 + 1) * N, 2 * kb, kb, nf, cudaMemcpyDeviceToHost, s));
      if (desc_left) ORBX_CUDA(c, cudaMemcpy2DAsync(desc_left + f0 * db, db, p.desc + i0 * db, 2 * db, db, nf, cudaMemcpyDeviceToHost, s));
      if (desc_right) ORBX_CUDA(c, cudaMemcpy2DAsync(desc_right + f0 * db, db, p.desc + (i0 + 1) * db, 2 * db, db, nf, cudaMemcpyDeviceToHost, s));
      if (n_left) ORBX_CUDA(c, cudaMemcpy2DAsync(n_left + f0, 4, p.n_kps + i0, 8, 4, nf, cudaMemcpyDeviceToHost, s));
      if (n_right) ORBX_CUDA(c, cudaMemcpy2DAsync(n_right + f0, 4, p.n_kps + i0 + 1, 8, 4, nf, cudaMemcpyDeviceToHost, s));
      if (u_right) ORBX_CUDA(c, cudaMemcpyAsync(u_right + f0 * N, p.u_right + d0 * N, N * 8 * nf, cudaMemcpyDeviceToHost, s));
      if (depth) ORBX_CUDA(c, cudaMemcpyAsync(depth + f0 * N, p.depth + d0 * N, N * 8 * nf, cudaMemcpyDeviceToHost, s));
      if (n_matches) ORBX_CUDA(c, cudaMemcpyAsync(n_matches + f0, p.n_matches + d0, 4 * (size_t)nf, cudaMemcpyDeviceToHost, s));
      return ORBX_OK;
    });
    if (rc) return rc;
    if (piped)
      for (int i = 0; i < c->kPipe; ++i) ORBX_CUDA(c, cudaStreamSynchronize(c->pipe[i]));
    else
      ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    return ORBX_OK;
  }

  int orbx_stereo_frame(orbx_ctx *c, const uint8_t *left, size_t left_stride, const uint8_t *right, size_t right_stride, orbx_keypoint *kps_left,
                        uint8_t *desc_left, int32_t *n_left, orbx_keypoint *kps_right, uint8_t *desc_right, int32_t *n_right, double *u_right, double *depth,
                        int32_t *n_matches)
  {
    if (!c || !left || !right) return ORBX_ERR_INVALID_ARG;
    return stereo_frame_host(c, left, left_stride, right, right_stride, std::max(left_stride, right_stride) * (size_t)c->cfg.height, kps_left, desc_left,
                             n_left, kps_right, desc_right, n_right, u_right, depth, n_matches);
  }

  int orbx_extract(orbx_ctx *c, const uint8_t *image, size_t stride, orbx_keypoint *kps, uint8_t *desc, int32_t *n)
  {
    if (!c || !image) return ORBX_ERR_INVALID_ARG;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    const size_t W = (size_t)c->cfg.width, H = (size_t)c->cfg.height, N = (size_t)c->cfg.n_features;
    ORBX_CUDA(c, cudaMemcpy2DAsync(c->d_in, c->in_pitch, image, stride, W * c->p.in_bpp, H, cudaMemcpyHostToDevice, c->stream));
    int rc = orbx_extract_batch_device(c, 1, c->d_in, c->in_pitch, c->in_pitch * H, nullptr);
    if (rc) return rc;
    const Params &p = c->p;
    if (kps) ORBX_CUDA(c, cudaMemcpyAsync(kps, p.kps, N * sizeof(orbx_keypoint), cudaMemcpyDeviceToHost, c->stream));
    if (desc) ORBX_CUDA(c, cudaMemcpyAsync(desc, p.desc, N * 32, cudaMemcpyDeviceToHost, c->stream));
    if (n) ORBX_CUDA(c, cudaMemcpyAsync(n, p.n_kps, 4, cudaMemcpyDeviceToHost, c->stream));
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    return ORBX_OK;
  }

  int orbx_rgbd_frame(orbx_ctx *c, const uint8_t *gray, size_t gray_stride, const void *depth_image, size_t depth_stride_bytes, int depth_type,
                      orbx_keypoint *kps_raw, orbx_keypoint *kps, uint8_t *desc, int32_t *n, double *u_right, double *depth)
  {
    if (!c || !gray || !depth_image || (depth_type != ORBX_DEPTH_U16 && depth_type != ORBX_DEPTH_F32)) return ORBX_ERR_INVALID_ARG;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    const size_t W = (size_t)c->cfg.width, H = (size_t)c->cfg.height, N = (size_t)c->cfg.n_features;
    const size_t esz = depth_type == ORBX_DEPTH_F32 ? 4 : 2;
    ORBX_CUDA(c, cudaMemcpy2DAsync(c->d_in, c->in_pitch, gray, gray_stride, W * c->p.in_bpp, H, cudaMemcpyHostToDevice, c->stream));
    ORBX_CUDA(c, cudaMemcpy2DAsync(c->d_depth_in, W * esz, depth_image, depth_stride_bytes, W * esz, H, cudaMemcpyHostToDevice, c->stream));
    int rc = orbx_rgbd_batch_device(c, 1, c->d_in, c->in_pitch, c->in_pitch * H, c->d_depth_in, W * esz, W * H * esz, depth_type, nullptr);
    if (rc) return rc;
    const Params &p = c->p;
    if (kps_raw) ORBX_CUDA(c, cudaMemcpyAsync(kps_raw, p.kps, N * sizeof(orbx_keypoint), cudaMemcpyDeviceToHost, c->stream));
    if (kps) ORBX_CUDA(c, cudaMemcpyAsync(kps, p.kps_und, N * sizeof(orbx_keypoint), cudaMemcpyDeviceToHost, c->stream));
    if (desc) ORBX_CUDA(c, cudaMemcpyAsync(desc, p.desc, N * 32, cudaMemcpyDeviceToHost, c->stream));
    if (n) ORBX_CUDA(c, cudaMemcpyAsync(n, p.n_kps, 4, cudaMemcpyDeviceToHost, c->stream));
    if (u_right) ORBX_CUDA(c, cudaMemcpyAsync(u_right, p.u_right, N * 8, cudaMemcpyDeviceToHost, c->stream));
    if (depth) ORBX_CUDA(c, cudaMemcpyAsync(depth, p.depth, N * 8, cudaMemcpyDeviceToHost, c->stream));
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    return ORBX_OK;
  }

  int orbx_get_pyramid(orbx_ctx *c, int side, int level, int blurred, uint8_t *dst, size_t dst_stride)
  {
    if (!c || !dst || level < 0 || level >= c->cfg.n_levels || side < 0) return ORBX_ERR_INVALID_ARG;
    if (int rc = require_images(c, side + 1LL)) return rc;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    const Level &L = c->levels[level];
    const uint8_t *src = (blurred ? c->p.blur : c->p.pyr) + (size_t)side * c->p.pyr_img_stride + L.pyr_off;
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    ORBX_CUDA(c, cudaMemcpy2D(dst, dst_stride, src, (size_t)L.pitch, (size_t)L.w, (size_t)L.h, cudaMemcpyDeviceToHost));
    return ORBX_OK;
  }

  int orbx_grid_info(const orbx_ctx *c, int32_t *rows, int32_t *cols, float *min_u, float *min_v, float *max_u, float *max_v)
  {
    if (!c) return ORBX_ERR_INVALID_ARG;
    if (rows) *rows = c->p.grid_rows;
    if (cols) *cols = c->p.grid_cols;
    if (min_u) *min_u = c->min_u;
    if (min_v) *min_v = c->min_v;
    if (max_u) *max_u = c->max_u;
    if (max_v) *max_v = c->max_v;
    return ORBX_OK;
  }

  int orbx_get_grid(orbx_ctx *c, int frame, int32_t *cell_start, int32_t *entries)
  {
    if (!c || frame < 0 || !cell_start || !entries) return ORBX_ERR_INVALID_ARG;
    if (int rc = require_frames(c, frame + 1LL)) return rc;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    const size_t nc = (size_t)c->p.grid_rows * c->p.grid_cols, N = (size_t)c->cfg.n_features;
    ORBX_CUDA(c, cudaMemcpy(cell_start, c->p.grid_start + (size_t)frame * (nc + 1), (nc + 1) * sizeof(int), cudaMemcpyDeviceToHost));
    std::vector<uint16_t> e16(N);
    ORBX_CUDA(c, cudaMemcpy(e16.data(), c->p.grid_entries + (size_t)frame * N, N * sizeof(uint16_t), cudaMemcpyDeviceToHost));
    const int total = cell_start[nc];
    for (int i = 0; i < total && i < (int)N; ++i) entries[i] = e16[i];
    return ORBX_OK;
  }

  // ---------------------------------------------------------------------------------------------------------------
  // tracking-side matchers (SURVEY.md section 8(f) rank 2)
  // the matcher staging grows with 50 % + 4 KiB of headroom, so that slowly rising input sizes do not reallocate every call
  static int reserve_match_scratch(orbx_ctx *c, size_t bytes)
  {
    return bytes <= c->match_scratch.bytes ? ORBX_OK : c->match_scratch.reserve(c, bytes + bytes / 2 + 4096);
  }

  static inline size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }

  // orbx_search_in_area_batch_device on the resident frames [frame0, frame0 + n_frames), on the context's stream
  static int search_in_area_device(orbx_ctx *c, int frame0, int n_frames, int query_stride, const orbx_area_query *d_queries, const uint8_t *d_query_desc,
                                   const int32_t *d_n_queries, const uint8_t *d_exclude, int32_t *d_best_idx, int32_t *d_best_dist, float *d_ratio,
                                   int32_t *d_n_candidates)
  {
    AreaArgs a{};
    a.image_stride = image_stride(c), a.max_u = c->max_u, a.max_v = c->max_v;
    a.q = d_queries, a.q_desc = d_query_desc, a.n_q = d_n_queries, a.n_q_all = query_stride, a.q_stride = query_stride;
    a.exclude = d_exclude;
    a.best_idx = d_best_idx, a.best_dist = d_best_dist, a.ratio = d_ratio, a.n_cand = d_n_candidates;
    launch_area_match(params_at(c, frame0 * a.image_stride, frame0), a, n_frames, c->stream);
    ++c->launches;
    ORBX_CUDA(c, cudaGetLastError());
    return ORBX_OK;
  }

  int orbx_search_in_area_batch_device(orbx_ctx *c, int n_frames, int query_stride, const orbx_area_query *d_queries, const uint8_t *d_query_desc,
                                       const int32_t *d_n_queries, const uint8_t *d_exclude, int32_t *d_best_idx, int32_t *d_best_dist, float *d_ratio,
                                       int32_t *d_n_candidates)
  {
    if (!c || n_frames < 1 || query_stride < 1 || !d_queries || !d_query_desc || !d_best_idx || !d_best_dist || !d_ratio || !d_n_candidates)
      return ORBX_ERR_INVALID_ARG;
    if (int rc = require_frames(c, n_frames)) return rc;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    return search_in_area_device(c, 0, n_frames, query_stride, d_queries, d_query_desc, d_n_queries, d_exclude, d_best_idx, d_best_dist, d_ratio,
                                 d_n_candidates);
  }

  int orbx_search_in_area(orbx_ctx *c, int frame, int n_queries, const orbx_area_query *queries, const uint8_t *query_desc, const uint8_t *exclude,
                          int32_t *best_idx, int32_t *best_dist, float *ratio, int32_t *n_candidates)
  {
    if (!c || frame < 0 || n_queries < 0 || (n_queries && (!queries || !query_desc))) return ORBX_ERR_INVALID_ARG;
    if (int rc = require_frames(c, frame + 1LL)) return rc;
    if (n_queries == 0) return ORBX_OK;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    const size_t n = (size_t)n_queries, N = (size_t)c->cfg.n_features;
    const size_t o_q = 0, o_d = o_q + up256(n * sizeof(orbx_area_query)), o_x = o_d + up256(n * 32), o_out = o_x + up256(N), total = o_out + up256(n * 16);
    int rc = reserve_match_scratch(c, total);
    if (rc) return rc;
    uint8_t *base = c->match_scratch.p;
    cudaStream_t s = c->stream;
    ORBX_CUDA(c, cudaMemcpyAsync(base + o_q, queries, n * sizeof(orbx_area_query), cudaMemcpyHostToDevice, s));
    ORBX_CUDA(c, cudaMemcpyAsync(base + o_d, query_desc, n * 32, cudaMemcpyHostToDevice, s));
    if (exclude) ORBX_CUDA(c, cudaMemcpyAsync(base + o_x, exclude, N, cudaMemcpyHostToDevice, s));
    int32_t *d_idx = (int32_t *)(base + o_out), *d_dist = d_idx + n, *d_nc = d_dist + n;
    float *d_ratio = (float *)(d_nc + n);
    rc = search_in_area_device(c, frame, 1, n_queries, (const orbx_area_query *)(base + o_q), base + o_d, nullptr, exclude ? base + o_x : nullptr, d_idx,
                               d_dist, d_ratio, d_nc);
    if (rc) return rc;
    if (best_idx) ORBX_CUDA(c, cudaMemcpyAsync(best_idx, d_idx, n * 4, cudaMemcpyDeviceToHost, s));
    if (best_dist) ORBX_CUDA(c, cudaMemcpyAsync(best_dist, d_dist, n * 4, cudaMemcpyDeviceToHost, s));
    if (n_candidates) ORBX_CUDA(c, cudaMemcpyAsync(n_candidates, d_nc, n * 4, cudaMemcpyDeviceToHost, s));
    if (ratio) ORBX_CUDA(c, cudaMemcpyAsync(ratio, d_ratio, n * 4, cudaMemcpyDeviceToHost, s));
    ORBX_CUDA(c, cudaStreamSynchronize(s));
    return ORBX_OK;
  }

  int orbx_verify_angle(orbx_ctx *c, int n_matches, int32_t *query_idx, int32_t *train_idx, float *distance, const orbx_keypoint *kps1, int n1,
                        const orbx_keypoint *kps2, int n2, int32_t *n_out)
  {
    if (!c || n_matches < 0 || !n_out || n1 < 0 || n2 < 0) return ORBX_ERR_INVALID_ARG;
    *n_out = 0;
    if (n_matches == 0) return ORBX_OK;
    if (!query_idx || !train_idx || !distance || !kps1 || !kps2) return ORBX_ERR_INVALID_ARG;
    for (int i = 0; i < n_matches; ++i)
      if (query_idx[i] < 0 || query_idx[i] >= n1 || train_idx[i] < 0 || train_idx[i] >= n2)
        return fail(c, ORBX_ERR_INVALID_ARG, "match index outside the keypoint arrays");
    ORBX_CUDA(c, cudaSetDevice(c->device));
    const size_t n = (size_t)n_matches;
    const size_t o_in = 0, o_k1 = o_in + up256(n * 12), o_k2 = o_k1 + up256((size_t)n1 * sizeof(orbx_keypoint)),
                 o_out = o_k2 + up256((size_t)n2 * sizeof(orbx_keypoint)), total = o_out + up256(n * 12 + 4);
    int rc = reserve_match_scratch(c, total);
    if (rc) return rc;
    uint8_t *base = c->match_scratch.p;
    cudaStream_t s = c->stream;
    int32_t *d_q = (int32_t *)(base + o_in), *d_t = d_q + n;
    float *d_d = (float *)(d_t + n);
    int32_t *d_oq = (int32_t *)(base + o_out), *d_ot = d_oq + n;
    float *d_od = (float *)(d_ot + n);
    int32_t *d_n = (int32_t *)(d_od + n);
    ORBX_CUDA(c, cudaMemcpyAsync(d_q, query_idx, n * 4, cudaMemcpyHostToDevice, s));
    ORBX_CUDA(c, cudaMemcpyAsync(d_t, train_idx, n * 4, cudaMemcpyHostToDevice, s));
    ORBX_CUDA(c, cudaMemcpyAsync(d_d, distance, n * 4, cudaMemcpyHostToDevice, s));
    ORBX_CUDA(c, cudaMemcpyAsync(base + o_k1, kps1, (size_t)n1 * sizeof(orbx_keypoint), cudaMemcpyHostToDevice, s));
    ORBX_CUDA(c, cudaMemcpyAsync(base + o_k2, kps2, (size_t)n2 * sizeof(orbx_keypoint), cudaMemcpyHostToDevice, s));
    VerifyArgs a{};
    a.n = n_matches, a.query_idx = d_q, a.train_idx = d_t, a.distance = d_d;
    a.kps1 = (const orbx_keypoint *)(base + o_k1), a.kps2 = (const orbx_keypoint *)(base + o_k2);
    a.out_query = d_oq, a.out_train = d_ot, a.out_dist = d_od, a.n_out = d_n;
    launch_verify_angle(a, s);
    ++c->launches;
    ORBX_CUDA(c, cudaGetLastError());
    ORBX_CUDA(c, cudaMemcpyAsync(n_out, d_n, 4, cudaMemcpyDeviceToHost, s));
    ORBX_CUDA(c, cudaStreamSynchronize(s));
    const size_t m = (size_t)*n_out;
    if (m)
    {
      ORBX_CUDA(c, cudaMemcpy(query_idx, d_oq, m * 4, cudaMemcpyDeviceToHost));
      ORBX_CUDA(c, cudaMemcpy(train_idx, d_ot, m * 4, cudaMemcpyDeviceToHost));
      ORBX_CUDA(c, cudaMemcpy(distance, d_od, m * 4, cudaMemcpyDeviceToHost));
    }
    return ORBX_OK;
  }

  // ---------------------------------------------------------------------------------------------------------------
  // result serialisation (SURVEY.md section 8(f) rank 4)
  int64_t orbx_serialized_capacity(const orbx_ctx *c)
  {
    if (!c) return 0;
    // head <= 31, tail 58, packed-field headers <= 16; per keypoint: entry <= 28, right_u 4, depth 4, descriptor 36, map point 10
    return (int64_t)((128 + (size_t)c->cfg.n_features * (28 + 4 + 4 + 36 + 10) + 15) & ~(size_t)15);
  }

  int64_t orbx_serialized_capacity_bow(const orbx_ctx *c)
  {
    if (!c) return 0;
    // + per keypoint at most one BowVector entry (<= 17) and one FeatureNode (<= 13 + 3 per feature id), + two field headers
    return (int64_t)((128 + 12 + (size_t)c->cfg.n_features * (28 + 4 + 4 + 36 + 10 + 17 + 13 + 3) + 15) & ~(size_t)15);
  }

  // the serialiser on the resident frames [frame0, frame0 + n_frames) into device memory, on the context's stream; with `bow`,
  // from their resident BoW
  static int serialize_device(orbx_ctx *c, int frame0, int n_frames, uint64_t id0, const float *d_pose_rt, int with_map_points, uint8_t *d_out,
                              size_t frame_stride, int64_t *d_sizes, bool bow)
  {
    const int is = image_stride(c);
    SerArgs a = ser_args(c, is, d_out, frame_stride, d_sizes, id0, d_pose_rt, with_map_points);
    if (bow) ser_bow_inputs(a, bow_at(c->bow, (size_t)frame0, (size_t)c->cfg.n_features));
    launch_serialize(params_at(c, frame0 * is, frame0), a, n_frames, c->stream);
    ++c->launches;
    ORBX_CUDA(c, cudaGetLastError());
    return ORBX_OK;
  }

  static int serialize_frames_device(orbx_ctx *c, int n_frames, uint64_t id0, const float *d_pose_rt, int with_map_points, uint8_t *d_out,
                                     size_t frame_stride, int64_t *d_sizes, bool bow)
  {
    if (!c || n_frames < 1 || !d_out || !d_sizes) return ORBX_ERR_INVALID_ARG;
    if (((size_t)d_out & 3) || (frame_stride & 3)) return fail(c, ORBX_ERR_INVALID_ARG, "output buffer and stride must be 4-byte aligned");
    if (bow && (int64_t)frame_stride < orbx_serialized_capacity_bow(c))
      return fail(c, ORBX_ERR_CAPACITY, "frame_stride is smaller than orbx_serialized_capacity_bow()");
    if ((int64_t)frame_stride < orbx_serialized_capacity(c)) return fail(c, ORBX_ERR_CAPACITY, "frame_stride is smaller than orbx_serialized_capacity()");
    if (int rc = require_frames(c, n_frames)) return rc;
    if (int rc = bow ? require_bow(c, n_frames) : ORBX_OK) return rc;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    return serialize_device(c, 0, n_frames, id0, d_pose_rt, with_map_points, d_out, frame_stride, d_sizes, bow);
  }

  int orbx_serialize_keyframes_device(orbx_ctx *c, int n_frames, uint64_t id0, const float *d_pose_rt, int with_map_points, uint8_t *d_out,
                                      size_t frame_stride, int64_t *d_sizes)
  {
    return serialize_frames_device(c, n_frames, id0, d_pose_rt, with_map_points, d_out, frame_stride, d_sizes, false);
  }

  int orbx_serialize_keyframes_bow_device(orbx_ctx *c, int n_frames, uint64_t id0, const float *d_pose_rt, int with_map_points, uint8_t *d_out,
                                          size_t frame_stride, int64_t *d_sizes)
  {
    return serialize_frames_device(c, n_frames, id0, d_pose_rt, with_map_points, d_out, frame_stride, d_sizes, true);
  }

  static int serialize_frame(orbx_ctx *c, int frame, uint64_t id, const float *pose_rt, int with_map_points, uint8_t *out, size_t cap, int64_t *n_bytes,
                             bool bow)
  {
    if (!c || frame < 0 || !out || !n_bytes) return ORBX_ERR_INVALID_ARG;
    if (int rc = require_frames(c, frame + 1LL)) return rc;
    if (int rc = bow ? require_bow(c, frame + 1LL) : ORBX_OK) return rc;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    const size_t rec = (size_t)(bow ? orbx_serialized_capacity_bow(c) : orbx_serialized_capacity(c));
    int rc = reserve_match_scratch(c, rec + 256);
    if (rc) return rc;
    uint8_t *base = c->match_scratch.p;
    cudaStream_t s = c->stream;
    float *d_pose = (float *)(base + rec);
    int64_t *d_size = (int64_t *)(base + rec + 64);
    if (pose_rt) ORBX_CUDA(c, cudaMemcpyAsync(d_pose, pose_rt, 12 * sizeof(float), cudaMemcpyHostToDevice, s));
    rc = serialize_device(c, frame, 1, id, pose_rt ? d_pose : nullptr, with_map_points, base, rec, d_size, bow);
    if (rc) return rc;
    int64_t sz = 0;
    ORBX_CUDA(c, cudaMemcpyAsync(&sz, d_size, sizeof(sz), cudaMemcpyDeviceToHost, s));
    ORBX_CUDA(c, cudaStreamSynchronize(s));
    *n_bytes = sz;
    if ((size_t)sz > cap) return fail(c, ORBX_ERR_CAPACITY, "output buffer too small for the record (see *n_bytes)");
    ORBX_CUDA(c, cudaMemcpy(out, base, (size_t)sz, cudaMemcpyDeviceToHost));
    return ORBX_OK;
  }

  int orbx_serialize_keyframe(orbx_ctx *c, int frame, uint64_t id, const float *pose_rt, int with_map_points, uint8_t *out, size_t cap, int64_t *n_bytes)
  {
    return serialize_frame(c, frame, id, pose_rt, with_map_points, out, cap, n_bytes, false);
  }

  int orbx_serialize_keyframe_bow(orbx_ctx *c, int frame, uint64_t id, const float *pose_rt, int with_map_points, uint8_t *out, size_t cap,
                                  int64_t *n_bytes)
  {
    return serialize_frame(c, frame, id, pose_rt, with_map_points, out, cap, n_bytes, true);
  }

  int orbx_keyframe_list_head(const orbx_ctx *c, uint64_t next_id, uint8_t *out, size_t cap, int64_t *n_bytes)
  {
    if (!c || !out || !n_bytes) return ORBX_ERR_INVALID_ARG;
    uint8_t buf[16 + 4 * kMaxLevels];
    size_t n = 0;
    auto varint = [&](uint64_t v) {
      while (v >= 0x80u) buf[n++] = (uint8_t)(v | 0x80u), v >>= 7;
      buf[n++] = (uint8_t)v;
    };
    if (next_id) buf[n++] = 0x08, varint(next_id); // uint64 next_id = 1 (proto3: left out when 0)
    buf[n++] = 0x12;                                // repeated float scale_factors = 2, packed
    varint(4u * (uint64_t)c->levels.size());
    for (const Level &L : c->levels) std::memcpy(buf + n, &L.sf, 4), n += 4;
    *n_bytes = (int64_t)n;
    if (n > cap) return ORBX_ERR_CAPACITY;
    std::memcpy(out, buf, n);
    return ORBX_OK;
  }

  int orbx_keyframe_list_entry_prefix(int64_t record_bytes, uint8_t *out)
  {
    if (!out || record_bytes < 0) return ORBX_ERR_INVALID_ARG;
    int n = 0;
    uint64_t v = (uint64_t)record_bytes;
    out[n++] = 0x1A; // repeated KeyFrameData keyframes = 3
    while (v >= 0x80u) out[n++] = (uint8_t)(v | 0x80u), v >>= 7;
    out[n++] = (uint8_t)v;
    return n;
  }

  int orbx_serialize_keyframe_text(orbx_ctx *c, int frame, uint64_t id, const float *pose_rt, int with_map_points, int with_scale_header, uint64_t next_id,
                                   char *out, size_t cap, int64_t *n_bytes)
  {
    if (!c || frame < 0 || !out || !n_bytes) return ORBX_ERR_INVALID_ARG;
    if (int rc = require_frames(c, frame + 1LL)) return rc;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    const int img = frame * image_stride(c);
    const size_t N = (size_t)c->cfg.n_features;
    int n = 0;
    ORBX_CUDA(c, cudaMemcpy(&n, c->p.n_kps + img, sizeof(int), cudaMemcpyDeviceToHost));
    n = std::max(0, std::min(n, (int)N));
    std::vector<orbx_keypoint> kps((size_t)n);
    std::vector<uint8_t> desc((size_t)n * 32);
    std::vector<double> ur((size_t)n), dp((size_t)n);
    if (n)
    {
      ORBX_CUDA(c, cudaMemcpy(kps.data(), c->p.kps_und + (size_t)img * N, (size_t)n * sizeof(orbx_keypoint), cudaMemcpyDeviceToHost));
      ORBX_CUDA(c, cudaMemcpy(desc.data(), c->p.desc + (size_t)img * N * 32, (size_t)n * 32, cudaMemcpyDeviceToHost));
      ORBX_CUDA(c, cudaMemcpy(ur.data(), c->p.u_right + (size_t)frame * N, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
      ORBX_CUDA(c, cudaMemcpy(dp.data(), c->p.depth + (size_t)frame * N, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
    }
    std::string t;
    t.reserve((size_t)n * 200 + 256);
    char buf[64];
    auto num = [&](double v) { append_g(t, v); };
    auto integer = [&](long long v) {
      t.append(buf, (size_t)std::snprintf(buf, sizeof(buf), "%lld", v));
      t.push_back(' ');
    };
    if (with_scale_header)
    { // :458-467
      t.append(buf, (size_t)std::snprintf(buf, sizeof(buf), "%llu ", (unsigned long long)next_id));
      for (auto &L : c->levels) num((double)L.sf);
      t.push_back('\n');
    }
    // :470  os << id << " " << maxU << " " << maxV << " " << minU << " " << minV << endl   (no blank before the line end)
    t.append(buf, (size_t)std::snprintf(buf, sizeof(buf), "%llu %g %g %g %g\n", (unsigned long long)id, (double)c->max_u, (double)c->max_v, (double)c->min_u,
                                        (double)c->min_v));
    for (int i = 0; i < n; ++i)
    { // :473-478
      num((double)kps[(size_t)i].x), num((double)kps[(size_t)i].y), integer(kps[(size_t)i].octave), num((double)kps[(size_t)i].angle);
      num(ur[(size_t)i]), num(dp[(size_t)i]);
    }
    t.push_back('\n');
    for (size_t i = 0; i < (size_t)n * 32; ++i) integer(desc[i]); // :482-487
    t.push_back('\n');
    t.push_back('\n'); // bag-of-words vector of a fresh frame: empty (:490-492)
    t.push_back('\n'); // feature vector: empty (:495-501)
    static const float eye[12] = {1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0};
    const float *pose = pose_rt ? pose_rt : eye;
    for (int i = 0; i < 12; ++i) num((double)pose[i]); // :504-509
    t.push_back('\n');
    t.push_back('\n'); // connected keyframes (:512-514)
    t.push_back('\n'); // children (:517-519)
    t.push_back('\n'); // loop edges (:522-524)
    if (with_map_points)
      for (int i = 0; i < n; ++i) t.append("-1 "); // :527-529
    t.push_back('\n');
    *n_bytes = (int64_t)t.size();
    if (t.size() > cap) return fail(c, ORBX_ERR_CAPACITY, "output buffer too small for the text record (see *n_bytes)");
    std::memcpy(out, t.data(), t.size());
    return ORBX_OK;
  }

  // ---------------------------------------------------------------------------------------------------------------
  // bag-of-words transform (SURVEY.md section 8(f) rank 3)
  void orbx_vocab_destroy(orbx_vocab *v)
  {
    if (!v) return;
    cudaSetDevice(v->device);
    cudaFree(v->child_start);
    cudaFree(v->child_ids);
    cudaFree(v->word);
    cudaFree(v->desc);
    cudaFree(v->weight);
    delete v;
  }

  int orbx_vocab_create(orbx_ctx *c, int k, int L, int n_records, const int32_t *parent, const uint8_t *is_leaf, const uint8_t *desc, const double *weight,
                        orbx_vocab **out)
  {
    if (!c || !out || k < 1 || L < 1 || n_records < 1 || !parent || !is_leaf || !desc || !weight) return ORBX_ERR_INVALID_ARG;
    *out = nullptr;
    const int n = n_records + 1;
    // record i describes node i + 1 (ids in record order, as DBoW3's text loader assigns them); children keep record order
    std::vector<int> cnt((size_t)n + 1, 0), start((size_t)n + 1, 0), ids((size_t)n_records), word((size_t)n, -1);
    for (int i = 0; i < n_records; ++i)
    {
      if (parent[i] < 0 || parent[i] > i) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary record refers to a parent that does not precede it");
      ++cnt[(size_t)parent[i]];
    }
    for (int i = 0; i < n; ++i) start[(size_t)i + 1] = start[(size_t)i] + cnt[(size_t)i];
    std::vector<int> cur(start.begin(), start.end() - 1);
    for (int i = 0; i < n_records; ++i) ids[(size_t)cur[(size_t)parent[i]]++] = i + 1;
    int n_words = 0;
    for (int i = 0; i < n_records; ++i)
    {
      const bool has_children = cnt[(size_t)i + 1] > 0;
      if ((is_leaf[i] != 0) == has_children) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary leaf flags do not match the tree structure");
      if (is_leaf[i]) word[(size_t)i + 1] = n_words++;
    }
    std::vector<uint8_t> d((size_t)n * 32, 0);
    std::memcpy(d.data() + 32, desc, (size_t)n_records * 32);
    std::vector<double> w((size_t)n, 0.0);
    std::memcpy(w.data() + 1, weight, (size_t)n_records * sizeof(double));
    ORBX_CUDA(c, cudaSetDevice(c->device));
    Building<orbx_vocab> v(new orbx_vocab(), orbx_vocab_destroy);
    v->ctx = c, v->device = c->device, v->k = k, v->L = L, v->n_nodes = n, v->n_words = n_words;
    v->rec_parent.assign(parent, parent + n_records);
    v->rec_leaf.resize((size_t)n_records);
    for (int i = 0; i < n_records; ++i) v->rec_leaf[(size_t)i] = is_leaf[i] != 0;
    v->rec_desc.assign(desc, desc + (size_t)n_records * 32);
    v->rec_weight.assign(weight, weight + n_records);
    auto up = [&](auto **dst, const auto &src) -> cudaError_t {
      cudaError_t e = cudaMalloc((void **)dst, src.size() * sizeof(src[0]) + 64);
      if (e != cudaSuccess) return e;
      return cudaMemcpy(*dst, src.data(), src.size() * sizeof(src[0]), cudaMemcpyHostToDevice);
    };
    ORBX_CUDA(c, up(&v->child_start, start));
    ORBX_CUDA(c, up(&v->child_ids, ids));
    ORBX_CUDA(c, up(&v->word, word));
    ORBX_CUDA(c, up(&v->desc, d));
    ORBX_CUDA(c, up(&v->weight, w));
    *out = v.release();
    return ORBX_OK;
  }

  int orbx_vocab_load_text(orbx_ctx *c, const char *path, orbx_vocab **out)
  {
    if (!c || !path || !out) return ORBX_ERR_INVALID_ARG;
    *out = nullptr;
    std::ifstream f(path);
    if (!f.is_open()) return fail(c, ORBX_ERR_FILE_NOT_OPEN, std::string("cannot open vocabulary ") + path);
    int k = 0, L = 0, scoring = 0, weighting = 0;
    {
      std::string line;
      std::getline(f, line);
      std::stringstream ss(line);
      if (!(ss >> k >> L >> scoring >> weighting)) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary header is not 'k L scoring weighting'");
    }
    // DBoW3: WeightingType { TF_IDF, TF, IDF, BINARY }, ScoringType { L1_NORM, L2_NORM, CHI_SQUARE, KL, BHATTACHARYYA, DOT_PRODUCT };
    // supported here: term-frequency weightings with a scoring whose mustNormalize() asks for the L1 norm
    if (weighting < 0 || weighting > 1 || !(scoring == 0 || scoring == 2 || scoring == 3 || scoring == 4))
      return fail(c, ORBX_ERR_INVALID_ARG, "only TF_IDF / TF weighting with an L1-normalising scoring is supported");
    std::vector<int32_t> parent;
    std::vector<uint8_t> leaf, desc;
    std::vector<double> weight;
    std::string line;
    while (std::getline(f, line))
    {
      if (line.find_first_not_of(" \t\r") == std::string::npos) continue;
      std::stringstream ss(line);
      int pid = 0, is_leaf = 0;
      if (!(ss >> pid >> is_leaf)) return fail(c, ORBX_ERR_INVALID_ARG, "malformed vocabulary record");
      for (int b = 0; b < 32; ++b)
      {
        int x = 0;
        if (!(ss >> x)) return fail(c, ORBX_ERR_INVALID_ARG, "malformed vocabulary record (descriptor)");
        desc.push_back((uint8_t)x);
      }
      double w = 0;
      if (!(ss >> w)) return fail(c, ORBX_ERR_INVALID_ARG, "malformed vocabulary record (weight)");
      parent.push_back(pid);
      leaf.push_back(is_leaf > 0);
      weight.push_back(w);
    }
    if (parent.empty()) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary holds no nodes");
    const int rc = orbx_vocab_create(c, k, L, (int)parent.size(), parent.data(), leaf.data(), desc.data(), weight.data(), out);
    if (rc == ORBX_OK) (*out)->scoring = scoring, (*out)->weighting = weighting;
    return rc;
  }

  int orbx_vocab_arrays(const orbx_vocab *v, int32_t *parent, uint8_t *is_leaf, uint8_t *desc, double *weight)
  {
    if (!v) return ORBX_ERR_INVALID_ARG;
    const size_t n = v->rec_parent.size();
    if (parent) std::memcpy(parent, v->rec_parent.data(), n * sizeof(int32_t));
    if (is_leaf) std::memcpy(is_leaf, v->rec_leaf.data(), n);
    if (desc) std::memcpy(desc, v->rec_desc.data(), n * 32);
    if (weight) std::memcpy(weight, v->rec_weight.data(), n * sizeof(double));
    return ORBX_OK;
  }

  int orbx_vocab_save_text(const orbx_vocab *v, const char *path)
  {
    if (!v || !path) return ORBX_ERR_INVALID_ARG;
    // TemplatedVocabulary::saveToTextFile of ORB-SLAM2: "k L  scoring weighting", then per node
    // "parent isLeaf " + FORB::toString (every byte followed by a blank) + " " + weight
    std::string t;
    t.reserve(v->rec_parent.size() * 140 + 32);
    t += std::to_string(v->k) + " " + std::to_string(v->L) + "  " + std::to_string(v->scoring) + " " + std::to_string(v->weighting) + "\n";
    for (size_t i = 0; i < v->rec_parent.size(); ++i)
    {
      t += std::to_string(v->rec_parent[i]);
      t += v->rec_leaf[i] ? " 1 " : " 0 ";
      for (int b = 0; b < 32; ++b)
      {
        t += std::to_string((int)v->rec_desc[i * 32 + (size_t)b]);
        t.push_back(' ');
      }
      t.push_back(' ');
      append_g(t, v->rec_weight[i]);
      t.back() = '\n';
    }
    FILE *f = std::fopen(path, "wb");
    if (!f) return ORBX_ERR_FILE_NOT_OPEN;
    const bool ok = std::fwrite(t.data(), 1, t.size(), f) == t.size();
    return (std::fclose(f) == 0 && ok) ? ORBX_OK : ORBX_ERR_FILE_NOT_OPEN;
  }

  int orbx_vocab_info(const orbx_vocab *v, int32_t *k, int32_t *L, int32_t *n_nodes, int32_t *n_words)
  {
    if (!v) return ORBX_ERR_INVALID_ARG;
    if (k) *k = v->k;
    if (L) *L = v->L;
    if (n_nodes) *n_nodes = v->n_nodes;
    if (n_words) *n_words = v->n_words;
    return ORBX_OK;
  }

  int orbx_bow_transform_batch_device(orbx_ctx *c, const orbx_vocab *v, int n_frames, int levelsup, orbx_device_bow *out)
  {
    if (!c || !v || n_frames < 1 || !out) return ORBX_ERR_INVALID_ARG;
    if (v->device != c->device) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary lives on another device");
    if (int rc = require_frames(c, n_frames)) return rc;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    int rc = bow_buffers(c);
    if (rc) return rc;
    const BowArgs a = bow_args(v, levelsup, image_stride(c), c->bow);
    launch_bow_transform(c, c->p, a, n_frames, c->stream);
    c->bow_epoch = c->frame_epoch;
    c->bow_frames = n_frames;
    c->bow_vocab = v;
    ORBX_CUDA(c, cudaGetLastError());
    out->bow_ids = a.bow_ids, out->bow_vals = a.bow_vals, out->n_bow = a.n_bow;
    out->fv_nodes = a.fv_nodes, out->fv_start = a.fv_start, out->fv_feats = a.fv_feats, out->n_fv_nodes = a.n_fv;
    out->stride = c->cfg.n_features;
    return ORBX_OK;
  }

  int orbx_bow_transform(orbx_ctx *c, const orbx_vocab *v, int frame, int levelsup, int32_t *bow_ids, double *bow_vals, int32_t *n_bow, int32_t *fv_nodes,
                         int32_t *fv_start, int32_t *fv_feats, int32_t *n_fv_nodes)
  {
    if (!c || !v || frame < 0 || !n_bow || !n_fv_nodes) return ORBX_ERR_INVALID_ARG;
    if (int rc = require_frames(c, frame + 1LL)) return rc;
    orbx_device_bow d{};
    const int rc = orbx_bow_transform_batch_device(c, v, frame + 1, levelsup, &d); // frames 0..frame (single-frame calls: frame == 0)
    if (rc) return rc;
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    const BowArgs b = bow_at(c->bow, (size_t)frame, (size_t)c->cfg.n_features);
    ORBX_CUDA(c, cudaMemcpy(n_bow, b.n_bow, 4, cudaMemcpyDeviceToHost));
    ORBX_CUDA(c, cudaMemcpy(n_fv_nodes, b.n_fv, 4, cudaMemcpyDeviceToHost));
    if (bow_ids) ORBX_CUDA(c, cudaMemcpy(bow_ids, b.bow_ids, (size_t)*n_bow * 4, cudaMemcpyDeviceToHost));
    if (bow_vals) ORBX_CUDA(c, cudaMemcpy(bow_vals, b.bow_vals, (size_t)*n_bow * 8, cudaMemcpyDeviceToHost));
    if (fv_nodes) ORBX_CUDA(c, cudaMemcpy(fv_nodes, b.fv_nodes, (size_t)*n_fv_nodes * 4, cudaMemcpyDeviceToHost));
    if (fv_start) ORBX_CUDA(c, cudaMemcpy(fv_start, b.fv_start, ((size_t)*n_fv_nodes + 1) * 4, cudaMemcpyDeviceToHost));
    if (fv_feats)
    {
      int32_t n_listed = 0; // == fv_start[n_fv_nodes]: only that many entries were written
      ORBX_CUDA(c, cudaMemcpy(&n_listed, b.fv_start + *n_fv_nodes, 4, cudaMemcpyDeviceToHost));
      if (n_listed > 0) ORBX_CUDA(c, cudaMemcpy(fv_feats, b.fv_feats, (size_t)n_listed * 4, cudaMemcpyDeviceToHost));
    }
    return ORBX_OK;
  }

  int orbx_search_by_bow(orbx_ctx *c, int frame, int n_kf_nodes, const int32_t *kf_fv_nodes, const int32_t *kf_fv_start, const int32_t *kf_fv_feats,
                         const uint8_t *kf_desc, int n_kf, const uint8_t *kf_query_ok, const uint8_t *frame_cand_ok, int32_t *best_idx, int32_t *best_dist,
                         float *ratio, int32_t *n_candidates)
  {
    if (!c || frame < 0 || n_kf_nodes < 0 || n_kf < 0) return ORBX_ERR_INVALID_ARG;
    if (n_kf_nodes == 0) return ORBX_OK;
    if (!kf_fv_nodes || !kf_fv_start || !kf_fv_feats || !kf_desc) return ORBX_ERR_INVALID_ARG;
    if (int rc = require_bow(c, frame + 1LL)) return rc;
    const int n_listed = kf_fv_start[n_kf_nodes];
    if (n_listed <= 0) return ORBX_OK;
    for (int i = 0; i < n_listed; ++i)
      if (kf_fv_feats[i] < 0 || kf_fv_feats[i] >= n_kf) return fail(c, ORBX_ERR_INVALID_ARG, "keyframe FeatureVector refers to a feature outside kf_desc");
    ORBX_CUDA(c, cudaSetDevice(c->device));
    const size_t N = (size_t)c->cfg.n_features, nl = (size_t)n_listed, nn = (size_t)n_kf_nodes;
    const size_t o_nodes = 0, o_start = o_nodes + up256(nn * 4), o_feats = o_start + up256((nn + 1) * 4), o_desc = o_feats + up256(nl * 4),
                 o_qok = o_desc + up256((size_t)n_kf * 32), o_cok = o_qok + up256((size_t)n_kf), o_out = o_cok + up256(N), total = o_out + up256(nl * 16);
    int rc = reserve_match_scratch(c, total);
    if (rc) return rc;
    uint8_t *base = c->match_scratch.p;
    cudaStream_t s = c->stream;
    ORBX_CUDA(c, cudaMemcpyAsync(base + o_nodes, kf_fv_nodes, nn * 4, cudaMemcpyHostToDevice, s));
    ORBX_CUDA(c, cudaMemcpyAsync(base + o_start, kf_fv_start, (nn + 1) * 4, cudaMemcpyHostToDevice, s));
    ORBX_CUDA(c, cudaMemcpyAsync(base + o_feats, kf_fv_feats, nl * 4, cudaMemcpyHostToDevice, s));
    ORBX_CUDA(c, cudaMemcpyAsync(base + o_desc, kf_desc, (size_t)n_kf * 32, cudaMemcpyHostToDevice, s));
    if (kf_query_ok) ORBX_CUDA(c, cudaMemcpyAsync(base + o_qok, kf_query_ok, (size_t)n_kf, cudaMemcpyHostToDevice, s));
    if (frame_cand_ok) ORBX_CUDA(c, cudaMemcpyAsync(base + o_cok, frame_cand_ok, N, cudaMemcpyHostToDevice, s));
    const BowArgs b = bow_at(c->bow, (size_t)frame, N);
    BowMatchArgs a{};
    a.f_nodes = b.fv_nodes, a.f_start = b.fv_start, a.f_feats = b.fv_feats, a.f_n_nodes = b.n_fv;
    a.f_desc = c->p.desc + (size_t)frame * image_stride(c) * N * 32, a.frame_cand_ok = frame_cand_ok ? base + o_cok : nullptr;
    a.k_nodes = (const int *)(base + o_nodes), a.k_start = (const int *)(base + o_start), a.k_feats = (const int *)(base + o_feats);
    a.k_n_nodes = n_kf_nodes, a.k_n_listed = n_listed;
    a.k_desc = base + o_desc, a.kf_query_ok = kf_query_ok ? base + o_qok : nullptr;
    int32_t *d_idx = (int32_t *)(base + o_out), *d_dist = d_idx + nl, *d_nc = d_dist + nl;
    float *d_ratio = (float *)(d_nc + nl);
    a.best_idx = d_idx, a.best_dist = d_dist, a.n_cand = d_nc, a.ratio = d_ratio;
    launch_bow_match(a, s);
    ++c->launches;
    ORBX_CUDA(c, cudaGetLastError());
    if (best_idx) ORBX_CUDA(c, cudaMemcpyAsync(best_idx, d_idx, nl * 4, cudaMemcpyDeviceToHost, s));
    if (best_dist) ORBX_CUDA(c, cudaMemcpyAsync(best_dist, d_dist, nl * 4, cudaMemcpyDeviceToHost, s));
    if (n_candidates) ORBX_CUDA(c, cudaMemcpyAsync(n_candidates, d_nc, nl * 4, cudaMemcpyDeviceToHost, s));
    if (ratio) ORBX_CUDA(c, cudaMemcpyAsync(ratio, d_ratio, nl * 4, cudaMemcpyDeviceToHost, s));
    ORBX_CUDA(c, cudaStreamSynchronize(s));
    return ORBX_OK;
  }

  int orbx_debug_level_corners(orbx_ctx *c, int image, int level, int32_t *xs, int32_t *ys, int32_t *scores, int cap, int32_t *n)
  {
    if (!c || !n || level < 0 || level >= c->cfg.n_levels || image < 0) return ORBX_ERR_INVALID_ARG;
    if (int rc = require_images(c, image + 1LL)) return rc;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    const Level &L = c->levels[level];
    std::vector<int> cnt(L.n_level_cells);
    ORBX_CUDA(c, cudaMemcpy(cnt.data(), c->p.cell_cnt + (size_t)image * c->p.n_cells + L.cell_base, cnt.size() * sizeof(int), cudaMemcpyDeviceToHost));
    int k = 0;
    std::vector<uint32_t> buf;
    for (int ci = 0; ci < L.n_level_cells; ++ci)
    {
      const Cell &ce = c->cells[L.cell_base + ci];
      buf.resize(cnt[ci]);
      if (cnt[ci])
        ORBX_CUDA(c, cudaMemcpy(buf.data(), c->p.cell_list + (size_t)image * c->p.cell_entries + ce.slot, cnt[ci] * sizeof(uint32_t),
                                cudaMemcpyDeviceToHost));
      for (int j = 0; j < cnt[ci]; ++j, ++k)
        if (k < cap)
        {
          if (xs) xs[k] = (int)(buf[j] & 0xfffu);
          if (ys) ys[k] = (int)((buf[j] >> 12) & 0xfffu);
          if (scores) scores[k] = (int)(buf[j] >> 24);
        }
    }
    *n = k;
    return ORBX_OK;
  }

  int orbx_debug_level_selected(orbx_ctx *c, int image, int level, int32_t *xs, int32_t *ys, int32_t *scores, int cap, int32_t *n)
  {
    if (!c || !n || level < 0 || level >= c->cfg.n_levels || image < 0) return ORBX_ERR_INVALID_ARG;
    if (int rc = require_images(c, image + 1LL)) return rc;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    const Level &L = c->levels[level];
    int cnt = 0;
    ORBX_CUDA(c, cudaMemcpy(&cnt, c->p.sel_cnt + (size_t)image * c->p.n_levels + level, sizeof(int), cudaMemcpyDeviceToHost));
    std::vector<uint32_t> buf(cnt > 0 ? cnt : 1);
    if (cnt) ORBX_CUDA(c, cudaMemcpy(buf.data(), c->p.sel + (size_t)image * c->p.sel_entries + L.sel_off, cnt * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    for (int k = 0; k < cnt && k < cap; ++k)
    {
      if (xs) xs[k] = (int)(buf[k] & 0xfffu);
      if (ys) ys[k] = (int)((buf[k] >> 12) & 0xfffu);
      if (scores) scores[k] = (int)(buf[k] >> 24);
    }
    *n = cnt;
    return ORBX_OK;
  }

  int orbx_debug_quadtree_stats(orbx_ctx *c, int64_t *fast, int64_t *sequential, int64_t *phase_cycles)
  {
    if (!c) return ORBX_ERR_INVALID_ARG;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    ORBX_CUDA(c, cudaDeviceSynchronize());
    unsigned long long h[16] = {};
    ORBX_CUDA(c, cudaMemcpy(h, c->p.qt_stats, sizeof(h), cudaMemcpyDeviceToHost));
    if (fast) *fast = (int64_t)h[0];
    if (sequential) *sequential = (int64_t)h[1];
    if (phase_cycles)
      for (int i = 0; i < 8; ++i) phase_cycles[i] = (int64_t)h[2 + i];
    return ORBX_OK;
  }

  int orbx_debug_run_quadtree(orbx_ctx *c, int level, const int32_t *xs, const int32_t *ys, const int32_t *scores, int n)
  {
    if (!c || level < 0 || level >= c->cfg.n_levels || n < 0 || (n > 0 && (!xs || !ys || !scores))) return ORBX_ERR_INVALID_ARG;
    const Level &L = c->levels[level];
    if (n > L.list_cap) return fail(c, ORBX_ERR_CAPACITY, "more corners than the level's cell slots can hold");
    ORBX_CUDA(c, cudaSetDevice(c->device));
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    // spread the list over the level's cell slots in order: the kernel concatenates them back in the same order
    std::vector<int> cnt(c->p.n_cells, 0);
    ORBX_CUDA(c, cudaMemcpy(c->p.cell_cnt, cnt.data(), cnt.size() * sizeof(int), cudaMemcpyHostToDevice));
    int k = 0;
    for (int ci = 0; ci < L.n_level_cells && k < n; ++ci)
    {
      const Cell &ce = c->cells[L.cell_base + ci];
      const int m = std::min(ce.cap, n - k);
      std::vector<uint32_t> buf(m);
      for (int j = 0; j < m; ++j, ++k)
      {
        if (xs[k] < 0 || xs[k] > 4095 || ys[k] < 0 || ys[k] > 4095 || scores[k] < 0 || scores[k] > 255) return ORBX_ERR_INVALID_ARG;
        buf[j] = (uint32_t)xs[k] | ((uint32_t)ys[k] << 12) | ((uint32_t)scores[k] << 24);
      }
      cnt[L.cell_base + ci] = m;
      ORBX_CUDA(c, cudaMemcpy(c->p.cell_list + ce.slot, buf.data(), (size_t)m * sizeof(uint32_t), cudaMemcpyHostToDevice));
    }
    ORBX_CUDA(c, cudaMemcpy(c->p.cell_cnt, cnt.data(), cnt.size() * sizeof(int), cudaMemcpyHostToDevice));
    launch_quadtree(c->p, 1, c->qt_smem, c->stream);
    c->launches += 1;
    ORBX_CUDA(c, cudaGetLastError());
    ORBX_CUDA(c, cudaStreamSynchronize(c->stream));
    // image 0 was overwritten: the frame-level results of an earlier call no longer match it
    set_resident(c, std::max(c->last_images, 1), 0, c->last_stereo);
    return ORBX_OK;
  }

} // extern "C"
