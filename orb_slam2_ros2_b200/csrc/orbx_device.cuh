// orbx_device.cuh -- device-side data layout shared by the kernels (orbx_kernels.cu) and the host layer (orbx_api.cu).
//
// HBM layout (all buffers are per context, sized for n_img_max = 2 * max_batch images):
//   pyr / blur     [image][pyr_img_stride]   every level stored with a 16-byte aligned pitch at Level::pyr_off
//   cell_list      [image][cell_entries]     one fixed-capacity slot per FAST cell, entries packed x:12 | y:12 | score:8
//   cell_cnt       [image][n_cells]
//   sel / sel_cnt  [image][sel_entries] / [image][n_levels]   quadtree survivors per level (ascending detection index)
//   kps, kps_und   [image][n_features]       cv::KeyPoint layout (28 B)
//   desc           [image][n_features][32]
//   rtab           [image][n_features]       {x, minRow, maxRow} row-band table for the stereo search
//   row_start/row_entries [frame][H+1] / [frame][row_cap]   CSR row index of the right keypoints (createRowIndexDB)
//   u_right, depth [frame][n_features]       doubles, -1 = no match
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

#include "../../include/orbx.h"

namespace orbx
{

constexpr int kMaxLevels = 16;  // one TMA descriptor per level travels as a kernel parameter (LevelMaps)
constexpr int kEdge = 16;       // FAST ROI margin: mnBorderSize - 3 (src/ORBExtractor.cc:334-337)
constexpr int kTileW = 64;      // pyramid/blur output tile
constexpr int kTileH = 64;
constexpr int kHalo = 3;        // 7x7 Gaussian
constexpr int kPyrThreads = 256;
constexpr int kFastThreads = 32;  // one warp = one FAST cell per CTA
constexpr int kQtThreads = 256;
constexpr int kMaxPatch = 65;   // largest FAST cell patch edge: a cell is at most 59 px wide, + 6 px apron
constexpr int kMaxStrips = 255; // root split fan-out: round(w/h) vertical strips
constexpr uint32_t kNil = 0xFFFFu;

struct Level
{
  int w, h, pitch;  // level image size and row pitch (bytes)
  int pyr_off;      // byte offset of the level inside one image's pyramid buffer
  float sf;         // mvfScaledFactors[level]
  int quota;        // mvnFeatures[level]
  int tab_x, tab_y; // offsets into the resize tables (unused for level 0)
  int area2x;       // exact 2x2 decimation: cv::resize re-routes INTER_LINEAR to INTER_AREA
  int tab_pair;     // offset into Params::tab_pair (one entry per pair of adjacent columns of the tile grid, incl. halo)
  int src_box_w, src_box_h; // TMA box that holds the level-0 source rectangle of any tile of this level (0: taps gathered from global memory)
  int pair_window;  // resize: the taps of two adjacent columns always lie inside one aligned 8-byte window of a level-0 row
  // FAST cell grid (src/ORBExtractor.cc:334-343)
  int n_cols, n_rows, w_cell, h_cell;
  int fast_box_h;   // rows of the TMA box that fetches one FAST patch of this level (its tallest patch)
  int cell_base;    // index of this level's first cell in the cell table
  int n_level_cells;
  // quadtree (src/ORBExtractor.cc:81-96,144-173)
  int roi_w, roi_h, n_ini;
  int strip_off;    // offset into Params::strips (n_ini + 1 column bounds)
  int list_cap;     // worst-case number of corners on this level
  int scratch_off;  // entry offset of this level inside one image's quadtree scratch (global-memory path)
  int sel_off;      // entry offset of this level inside one image's sel buffer
};

struct Tile
{
  int level, x0, y0;
  int src; // pyramid_levels_kernel: origin of the tile's level-0 source rectangle (TMA box), x | y << 16
};

struct Cell
{
  int level;
  int x0, y0;   // patch origin in level coordinates (iniX, iniY)
  int pw, ph;   // patch size (maxX - iniX, maxY - iniY)
  int slot;     // entry offset of the cell's slot inside one image's cell_list
  int cap;      // slot capacity
  int box_h;    // = Level::fast_box_h of its level (rows of the TMA box)
};

struct RTab
{
  float x;
  short min_row, max_row;
};

// TMA descriptors of the pyramid levels: 3-D {pitch, rows, images} byte tensors over `pyr`; box = 80 bytes x the level's
// tallest FAST patch.  Passed to the kernel by value (__grid_constant__).
struct LevelMaps
{
  CUtensorMap m[kMaxLevels];
};

struct Params
{
  int n_levels, n_features, ini_th, min_th;
  int n_tiles, n_cells;
  int n_tiles0; // tiles of level 0 (first in the tile table): pyramid_level0_kernel; the rest: pyramid_levels_kernel
  int width, height;
  int stereo; // images are interleaved left/right pairs
  // per-warp shared-memory slice of the FAST kernel (one warp per cell): patch at 0, then these offsets
  int fast_off_bar, fast_off_map, fast_off_cand, fast_off_mask, fast_off_lut, fast_map_pitch, fast_warp_bytes;
  const Level *levels;
  const Tile *tiles;
  const Cell *cells;
  const int *tab_ofs;     // resize source index per destination index
  const short2 *tab_coef; // resize 11-bit coefficients
  const uint4 *tab_pair;  // resize, two adjacent columns: {window_a | sel_a << 16, window_b | sel_b << 16, coef_a, coef_b}
  const long long *strips_fx; // root strip column bounds, 24.40 fixed point (exact: they are float-rounded values)
  const char4 *pattern;   // 256 x (x1, y1, x2, y2)
  // inputs
  const uint8_t *in_left, *in_right;
  size_t in_stride, in_frame_stride;
  const void *depth_img;
  size_t depth_stride, depth_frame_stride;
  int depth_type;
  int img0; // index of this launch's first image inside the context buffers (the TMA descriptors address whole buffers)
  // per-image buffers
  uint8_t *pyr, *blur;
  size_t pyr_img_stride;
  uint32_t *cell_list;
  size_t cell_entries;
  int *cell_cnt;
  uint32_t *sel;
  int sel_entries;
  int *sel_cnt;
  // quadtree scratch (global-memory path for levels whose corner count exceeds the shared-memory capacity)
  uint32_t *qt_scratch;
  size_t qt_scratch_img_stride; // in uint32 entries
  int qt_smem_cap;              // corners that fit the shared-memory path
  int qt_node_cap;              // node pool capacity (max quota + max root fan-out + 8)
  int qt_big_cap;               // capacity of the list of nodes holding >= 256 corners
  int qt_cell_cap;              // largest number of FAST cells on one level (+1): per-cell offsets in shared memory
  unsigned long long *qt_stats; // [2] CTAs that took the loop-free path / the sequential loop (introspection)
  int qt_fast;                  // take the loop-free formulation of Quadtree::split() where the keys decide (default; ORBX_QT_FAST=0 disables)
  // results
  orbx_keypoint *kps, *kps_und;
  uint8_t *desc;
  int *n_kps;
  RTab *rtab;
  int *row_start;            // [frame][height + 1]  CSR over image rows of the right keypoints whose band covers the row
  uint16_t *row_entries;     // [frame][row_cap]     right keypoint indices
  int row_cap;
  double *u_right, *depth;
  int *n_matches;
  // VirtualFrame::initGrid (src/Frame.cc:53-69): CSR over the 64x48-px grid cells of the (undistorted) left keypoints
  int *grid_start;        // [frame][grid_rows * grid_cols + 1]
  uint16_t *grid_entries; // [frame][n_features], ascending keypoint index inside a cell
  int grid_rows, grid_cols;
  // camera
  float fx, fy, cx, cy, bf, depth_scale_inv;
  float dist[5];
  int undistort;
};

// tracking-side matchers (orbx_match.cu)
struct AreaArgs
{
  const orbx_area_query *q; // [frame][q_stride]
  const uint8_t *q_desc;    // [frame][q_stride][32]
  const int *n_q;           // [frame] or null (then n_q_all queries for every frame)
  int n_q_all, q_stride;
  const uint8_t *exclude;   // [frame][n_features] or null
  int *best_idx, *best_dist, *n_cand; // [frame][q_stride]
  float *ratio;
  int image_stride;         // frame f's (left) image is image f * image_stride
  float max_u, max_v;       // mfMaxU / mfMaxV
};

struct BowMatchArgs
{
  // the frame's FeatureVector (device results of the last bag-of-words call) and descriptors
  const int *f_nodes, *f_start, *f_feats, *f_n_nodes;
  const uint8_t *f_desc, *frame_cand_ok;
  // the keyframe's FeatureVector, descriptors and mask (uploaded by the caller)
  const int *k_nodes, *k_start, *k_feats;
  int k_n_nodes, k_n_listed;
  const uint8_t *k_desc, *kf_query_ok;
  int *best_idx, *best_dist, *n_cand; // [k_n_listed]
  float *ratio;
};

struct VerifyArgs
{
  int n;
  const int *query_idx, *train_idx;
  const float *distance;
  const orbx_keypoint *kps1, *kps2;
  int *out_query, *out_train;
  float *out_dist;
  int *n_out;
};

// result serialisation (orbx_serialize.cu)
struct SerArgs
{
  uint8_t *out;          // [frame][stride], 4-byte aligned
  size_t stride;
  long long *sizes;      // [frame] bytes written
  unsigned long long id0; // record of frame f carries id0 + f
  const float *pose;     // [frame][12] R (row-major) | t, or null = identity
  int with_map_points;
  int image_stride;
  float max_u, max_v, min_u, min_v;
  // optional BowVector / FeatureVector of the launch's frames in the layout of BowArgs (per frame: n_features entries,
  // fv_start n_features + 1); null = fields 10 / 11 present but empty
  const int *bow_ids, *n_bow, *fv_nodes, *fv_start, *fv_feats, *n_fv;
  const double *bow_vals;
};

// bag-of-words transform (orbx_bow.cu)
struct BowArgs
{
  // vocabulary tree: node 0 = root; children of node i = child_ids[child_start[i] .. child_start[i + 1]) in id order
  const int *child_start, *child_ids;
  const uint8_t *v_desc;  // [n_nodes][32]
  const double *v_weight; // [n_nodes]
  const int *v_word;      // [n_nodes] word id of a leaf
  int L, levelsup, image_stride;
  // per feature: [frame][n_features]
  int *f_word, *f_nid;
  double *f_weight;
  // per frame results: BowVector [frame][n_features] + count, FeatureVector CSR
  int *bow_ids, *n_bow;
  double *bow_vals;
  int *fv_nodes, *fv_start /* [frame][n_features + 1] */, *fv_feats, *n_fv;
};

// the BoW results of b's frames as serialiser inputs (frame f of the launch = frame f of b)
inline void ser_bow_inputs(SerArgs &s, const BowArgs &b)
{
  s.bow_ids = b.bow_ids, s.bow_vals = b.bow_vals, s.n_bow = b.n_bow;
  s.fv_nodes = b.fv_nodes, s.fv_start = b.fv_start, s.fv_feats = b.fv_feats, s.n_fv = b.n_fv;
}

// launchers (orbx_kernels.cu / orbx_match.cu / orbx_serialize.cu / orbx_bow.cu); every call enqueues exactly one kernel on `s`
constexpr int kPyrBoxBytesHost = 18 * 1024; // = kPyrBoxBytes of orbx_kernels.cu: shared-memory bytes a level's source box may take
void launch_pyramid_level0(const Params &p, int n_images, cudaStream_t s);
void launch_pyramid_levels(const Params &p, const LevelMaps &src_maps, int n_images, cudaStream_t s);
const void *pyramid_kernel_symbol(); // host handle of the level-0 pyramid kernel, the only reader of the caller's images (to find its node in a captured graph)
void launch_fast(const Params &p, const LevelMaps &maps, int n_images, cudaStream_t s);
int fast_configure(const Params &p); // opt in to the dynamic shared memory of the FAST kernel
void launch_quadtree(const Params &p, int n_images, size_t smem_bytes, cudaStream_t s);
void launch_orient_brief(const Params &p, const LevelMaps &blur_maps, int n_images, cudaStream_t s);
void launch_stereo(const Params &p, int n_frames, cudaStream_t s);
void launch_rgbd(const Params &p, int n_frames, cudaStream_t s);
void launch_frame_index(const Params &p, int n_frames, int image_stride, bool with_rowindex, cudaStream_t s); // row index (stereo) + initGrid
int frame_index_configure(const Params &p); // opt in to large dynamic shared memory when the configuration needs it
void launch_area_match(const Params &p, const AreaArgs &a, int n_frames, cudaStream_t s);
void launch_verify_angle(const VerifyArgs &a, cudaStream_t s);
void launch_bow_match(const BowMatchArgs &a, cudaStream_t s);
void launch_serialize(const Params &p, const SerArgs &a, int n_frames, cudaStream_t s);
void launch_bow_descend(const Params &p, const BowArgs &a, int n_frames, cudaStream_t s);
void launch_bow_assemble(const Params &p, const BowArgs &a, int n_frames, cudaStream_t s);
void launch_bow_word_frames(const Params &p, const BowArgs &a, int n_frames, int *n_frames_of_word, cudaStream_t s);
size_t quadtree_smem_bytes(int list_cap, int node_cap, int big_cap, int max_level_cells);
int quadtree_configure(size_t smem_bytes); // opt in to large dynamic shared memory

// the counter-based generator of orbx_vocab_build and orbx_loopver_verify (include/orbx.h)
constexpr unsigned long long kGolden = 0x9E3779B97F4A7C15ull;
__host__ __device__ __forceinline__ unsigned long long splitmix64(unsigned long long x)
{
  unsigned long long z = x + kGolden;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the kernel (per device), not to a context: it is only ever RAISED, so a
// second context with a smaller configuration cannot shrink the limit under a live one (launches of the larger context would
// fail with "invalid argument").  `state` = the caller's per-kernel high-water marks, one per device.  A refused size is
// cleared from the runtime's last error, so that it is not reported again by an unrelated call's cudaGetLastError.
struct SmemOptIn
{
  std::mutex mu;
  int high[64] = {};
};
template <class Kernel> int raise_dynamic_smem(Kernel kernel, SmemOptIn &state, size_t bytes)
{
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return -1;
  std::lock_guard<std::mutex> lock(state.mu);
  if ((size_t)state.high[dev] >= bytes) return 0;
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
  {
    cudaGetLastError();
    return -1;
  }
  state.high[dev] = (int)bytes;
  return 0;
}

} // namespace orbx
