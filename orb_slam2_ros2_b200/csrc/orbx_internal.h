// orbx_internal.h -- host-side state shared by the translation units behind the C ABI (orbx_api.cu, orbx_sequence.cu).
#pragma once

#include <functional>
#include <string>
#include <vector>

#include "orbx_device.cuh"

namespace orbx
{
// Device memory that grows on demand and is freed with its context.  reserve(c, want) makes `p` hold at least `want` bytes;
// a buffer that has to grow is freed after a device synchronisation (work on any of the context's streams may still use it).
struct DeviceBuffer
{
  uint8_t *p = nullptr;
  size_t bytes = 0;
  DeviceBuffer() = default;
  DeviceBuffer(const DeviceBuffer &) = delete;
  DeviceBuffer &operator=(const DeviceBuffer &) = delete;
  ~DeviceBuffer() { if (p) cudaFree(p); }
  int reserve(orbx_ctx *c, size_t want);
};
} // namespace orbx

struct orbx_ctx
{
  orbx_config cfg;
  int device = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  int n_img_max = 0;
  std::vector<orbx::Level> levels;
  std::vector<orbx::Tile> tiles;
  int n_tiles0 = 0; // level-0 tiles (first in `tiles`)
  std::vector<orbx::Cell> cells;
  orbx::Params p;            // template: geometry + base pointers
  size_t qt_smem = 0;
  std::string last_error;
  int64_t launches = 0;
  int64_t alg_bytes_image = 0, alg_bytes_stereo = 0;
  // device allocations
  std::vector<void *> allocs;
  uint8_t *d_in = nullptr;      // staging for host-side calls: [n_img_max][H][in_pitch]
  size_t in_pitch = 0;
  uint8_t *d_depth_in = nullptr; // [max_batch][H][W] float/uint16 (sized for float)
  int last_images = 0;          // images processed by the most recent call (for orbx_get_pyramid)
  int last_stereo = 0;
  int last_frames = 0;
  orbx::LevelMaps maps;      // TMA descriptors of the pyramid levels, FAST patch boxes (kernel parameter, __grid_constant__)
  orbx::LevelMaps maps_blur; // TMA descriptors of the blurred levels, BRIEF patch boxes
  orbx::LevelMaps maps_src;  // TMA descriptors over level 0 of `pyr`, one box size per resized level (its tiles' source rectangles)
  float min_u = 0, min_v = 0, max_u = 0, max_v = 0; // undistorted image bounds (VirtualFrame ctor, Frame.h:33-43)
  // host-batch pipeline: chunks of frames round-robin over kPipe streams so that H2D, kernels and D2H overlap
  static constexpr int kPipeMax = 8;
  int kPipe = 8;  // streams (tunable for experiments: ORBX_PIPE); 8 x 8 frames measured best on B200
  int kChunk = 8; // frames per chunk (ORBX_CHUNK)
  int chunk() const { return kChunk < cfg.max_batch ? kChunk : cfg.max_batch; } // frames per chunk of this context's slots
  cudaStream_t pipe[kPipeMax] = {};
  cudaEvent_t fork_ev = nullptr;
  cudaEvent_t join_ev[kPipeMax] = {};
  // staging for the host-side matcher and serialiser calls (orbx_search_in_area, orbx_serialize_keyframe, ...)
  orbx::DeviceBuffer match_scratch;
  // bag-of-words transform: per-feature and per-frame result buffers, allocated on first use
  orbx::BowArgs bow{};
  bool bow_ready = false;
  // sequences (orbx_sequence.cu): per-slot record staging for host outputs, gathered arrays of single-rank calls
  orbx::DeviceBuffer rec_staging;
  struct orbx_comm *self_comm = nullptr;
  uint8_t *h_rec1 = nullptr; // pinned host record of the single-frame calls (one D2H copy instead of nine)
  // single-pair latency path: the launch sequence of one stereo frame captured once as a CUDA graph (orbx_set_graph)
  int use_graph = 1;
  cudaGraph_t graph1 = nullptr;
  cudaGraphExec_t graph1_exec = nullptr;
  cudaGraphNode_t graph1_pyr = nullptr; // the only node whose parameters carry the caller's input pointers
  const uint8_t *graph1_left = nullptr, *graph1_right = nullptr;
  size_t graph1_stride = 0, graph1_fs = 0;
  int graph1_kernels = 0;
  uint64_t frame_epoch = 0;   // bumped by every call that produces frames
  uint64_t bow_epoch = ~0ull; // frame_epoch at the last bag-of-words call
  int bow_frames = 0;         // frames covered by that call
  // keyframe records of sequences (orbx_sequence_stereo_keyframes): per-slot staging of records + poses for host outputs,
  // and the int64 sizes of a whole block (copied to the host once at the end)
  orbx::DeviceBuffer kf_staging, kf_sizes;
};

// DBoW3 vocabulary tree resident on one device
struct orbx_vocab
{
  const orbx_ctx *ctx = nullptr; // the context that created it
  int device = 0;
  int k = 0, L = 0, n_nodes = 0, n_words = 0;
  int *child_start = nullptr, *child_ids = nullptr, *word = nullptr;
  uint8_t *desc = nullptr;
  double *weight = nullptr;
};

namespace orbx
{

// records `msg` as the context's last error and returns `code`
int fail(orbx_ctx *c, int code, const std::string &msg);
// Params whose per-image buffers start at image `img0` (and per-frame buffers at frame `frame0`)
Params params_at(const orbx_ctx *c, int img0, int frame0);
// the same BowArgs with every per-frame buffer starting at frame `frame0` (N = n_features)
BowArgs bow_at(const BowArgs &b, size_t frame0, size_t N);
// SerArgs of a serialiser launch over device slots whose frame f reads image f * image_stride; no BoW inputs (ser_bow_inputs)
SerArgs ser_args(const orbx_ctx *c, int image_stride, uint8_t *out, size_t stride, int64_t *sizes, uint64_t id0, const float *pose, int with_map_points);
// Stereo input of n_frames frames (host memory, or device memory with `on_device`) streamed through the device slots in
// chunks of c->chunk() frames.  Chunk k lives in slot k % n_slots and, with `piped`, runs on stream pipe[slot % kPipe]
// after a fork from the context's stream; otherwise everything runs on the context's stream.  Per chunk: host frames are
// staged into the slot, the kernels are enqueued, then out(s, d0, f0, nf) enqueues the caller's outputs of frames
// [f0, f0 + nf) = device slots [d0, d0 + nf) on the chunk's stream s.  The right image may have its own row stride; frame
// f starts at f * frame_stride on both sides.  Leaves the last pass over the slots resident; the caller synchronises.
using ChunkOut = std::function<int(cudaStream_t s, int d0, int64_t f0, int nf)>;
int run_stereo_chunks(orbx_ctx *c, int64_t n_frames, const uint8_t *left, size_t left_stride, const uint8_t *right, size_t right_stride, size_t frame_stride,
                      bool on_device, bool piped, const ChunkOut &out);
// per-frame records (orbx_record_layout) of device slots [d0, d0 + nf) assembled at d_rec
int pack_frame_records(orbx_ctx *c, cudaStream_t s, int d0, int nf, uint8_t *d_rec, size_t rec_stride);
// frees the gathered arrays a context keeps for single-rank sequence calls
void destroy_self_comm(orbx_ctx *c);
// allocates the context's bag-of-words result buffers (n_img_max frames, as many as an RGB-D batch holds) on first use
int bow_buffers(orbx_ctx *c);
// c->bow with the vocabulary's tree, ready for launch_bow_descend / launch_bow_assemble over device slots whose frame f
// reads image f * image_stride
BowArgs bow_args(const orbx_ctx *c, const orbx_vocab *v, int levelsup, int image_stride);

} // namespace orbx

#define ORBX_CUDA(ctx, expr)                                                                                               \
  do                                                                                                                       \
  {                                                                                                                        \
    cudaError_t e__ = (expr);                                                                                              \
    if (e__ != cudaSuccess) return orbx::fail((ctx), ORBX_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
  } while (0)
