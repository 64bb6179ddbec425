// orbx_internal.h -- host-side state shared by the translation units behind the C ABI (orbx_api.cu, orbx_sequence.cu).
#pragma once

#include <functional>
#include <memory>
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

// the next multiple of 16 bytes: offsets of arrays laid out one after another in one device buffer
inline size_t up16(size_t v) { return (v + 15) & ~(size_t)15; }

// an object a builder is making, freed by its public *_destroy on every error path; release() hands it to the caller
template <class T> using Building = std::unique_ptr<T, void (*)(T *)>;
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
  size_t in_pitch = 0;          // 16-byte multiple >= width * p.in_bpp (grows with orbx_set_input_format)
  int in_format = ORBX_FORMAT_GRAY8;
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
  const orbx_vocab *bow_vocab = nullptr; // the vocabulary of that call
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
  int scoring = 0, weighting = 0; // DBoW3 ScoringType / WeightingType of the text header (0 = L1_NORM / TF_IDF)
  int *child_start = nullptr, *child_ids = nullptr, *word = nullptr;
  uint8_t *desc = nullptr;
  double *weight = nullptr;
  // the text format's records (record i = node i + 1), kept on the host for orbx_vocab_save_text / orbx_vocab_arrays
  std::vector<int32_t> rec_parent;
  std::vector<uint8_t> rec_leaf, rec_desc;
  std::vector<double> rec_weight;
};

namespace orbx
{

// records `msg` as the context's last error and returns `code`
int fail(orbx_ctx *c, int code, const std::string &msg);
// ORBX_OK when an object that context `owner_ctx` made on device `owner_device` belongs to `c`, else ORBX_ERR_INVALID_ARG
// with a message that names `what` as another context's
int require_owner(orbx_ctx *c, const orbx_ctx *owner_ctx, int owner_device, const char *what);
// resident CTAs of a grid-stride kernel on the context's device (CTAs per SM x SMs) in *n; ORBX_ERR_CUDA ("<what> does not
// fit an SM") when not one CTA fits
int resident_ctas(orbx_ctx *c, const void *kernel, int threads, size_t smem, const char *what, int *n);
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
// ORBX_OK when the bag of words of frames [0, end) is resident from the orbx_bow_transform* call on the most recent call's
// frames, ORBX_ERR_STATE otherwise
int require_bow(orbx_ctx *c, int64_t end);
// allocates the context's bag-of-words result buffers (n_img_max frames, as many as an RGB-D batch holds) on first use
int bow_buffers(orbx_ctx *c);
// every bag-of-words entry point's check before it enqueues anything: `too_large` (the caller's error code) for more than
// ORBX_BOW_MAX_STRIDE features per frame, else opts the assemble and word-frame kernels in to the sort's shared memory
// (ORBX_ERR_CUDA if that fails).  Needs the context's device current.
int bow_configure(orbx_ctx *c, int n_features, int too_large);
// `b` with the vocabulary's tree, ready for launch_bow_descend / launch_bow_assemble over frames whose frame f reads image
// f * image_stride (the context's slots: b = c->bow)
BowArgs bow_args(const orbx_vocab *v, int levelsup, int image_stride, BowArgs b = {});
// the transform of n_frames frames on `s`: launch_bow_descend, then launch_bow_assemble; counts both launches
void launch_bow_transform(orbx_ctx *c, const Params &p, const BowArgs &a, int n_frames, cudaStream_t s);
// A training set desc[F][stride][32] + n_kps[F] (host memory, or device memory with `on_device`) as the builders read it:
// the counts on the host, each checked to lie in 0..stride (else ORBX_ERR_INVALID_ARG, "<what>: a count lies outside
// 0..stride"), and device pointers to both arrays -- the caller's, or copies of host arrays staged on the context's stream
// that live as long as the TrainingSet.
struct TrainingSet
{
  std::vector<int32_t> n;
  const uint8_t *desc = nullptr;
  const int32_t *d_n = nullptr;
  DeviceBuffer staged;
};
int read_training_set(orbx_ctx *c, const uint8_t *desc, const int32_t *n_kps, int F, int stride, bool on_device, const char *what, TrainingSet &ts);
// BowVectors and FeatureVectors (orbx_bow_transform's, at `levelsup`) of F frames of device descriptors d_desc[f][stride][32],
// d_n[f] each, in chunks of frames: frame f's results go to out.bow_ids / bow_vals / fv_nodes / fv_feats + f * stride,
// out.fv_start + f * (stride + 1), out.n_bow / n_fv + f; the arrays left null in `out` get per-chunk scratch.  Synchronises.
int bow_frames(orbx_ctx *c, const orbx_vocab *v, int levelsup, const uint8_t *d_desc, const int *d_n, int F, int stride, const BowArgs &out);
// appends `v` as std::ostream << double prints it by default ("%g": 6 significant digits) and a blank
void append_g(std::string &t, double v);

// The arrays of one call of a query entry point whose io lives on the host or on the device, each stated once with the
// kernel argument it sets:
//   out(arg, user, bytes)      the caller's array (device io), a slice of `buf` that finish() copies back to `user` (host io,
//                              array wanted) or null (not wanted)
//   scratch(arg, bytes, host)  a slice of `buf` in either case, filled from `host` by place() when that is given
// place() sizes `buf`, points every staged argument at its slice and enqueues the copies in; after the launch, finish()
// enqueues the copies back and synchronises (host io only).  Everything runs on the context's stream.
struct IoStaging
{
  struct Slice
  {
    std::function<void(uint8_t *)> set;
    const void *from;
    void *to;
    size_t off, bytes;
  };
  orbx_ctx *c;
  DeviceBuffer &buf;
  bool on_device;
  size_t total = 0;
  std::vector<Slice> slices;
  template <class T> void out(T *&arg, T *user, size_t bytes)
  {
    if (on_device || !user) arg = user;
    else stage(arg, nullptr, user, bytes);
  }
  template <class T> void scratch(T *&arg, size_t bytes, const void *host = nullptr) { stage(arg, host, nullptr, bytes); }
  template <class T> void stage(T *&arg, const void *from, void *to, size_t bytes)
  {
    slices.push_back({[&arg](uint8_t *p) { arg = reinterpret_cast<T *>(p); }, from, to, total, bytes});
    total += up16(bytes);
  }
  int place();
  int finish();
};

} // namespace orbx

#define ORBX_CUDA(ctx, expr)                                                                                               \
  do                                                                                                                       \
  {                                                                                                                        \
    cudaError_t e__ = (expr);                                                                                              \
    if (e__ != cudaSuccess) return orbx::fail((ctx), ORBX_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
  } while (0)
