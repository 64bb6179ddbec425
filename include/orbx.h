/*
 * orbx.h -- C ABI of the B200-native ORB front-end (liborbx.so).
 *
 * Drop-in boundary for the per-frame feature path of sunshanlu/ORB_SLAM2_ROS2.  Every entry point names the
 * reference interface it replaces (paths relative to /root/reference/src/ORB_SLAM2/).  Plain pointers and sizes
 * only; the library owns all device memory and runs hand-written sm_100a kernels.  There is NO CPU fallback:
 * orbx_create() fails with ORBX_ERR_NO_DEVICE / ORBX_ERR_CUDA when no usable CUDA device exists.
 *
 * Threading: a context is not re-entrant; independent contexts may be used from different host threads
 * (the reference runs two ORBExtractor::extract() calls on two std::threads, src/Frame.cc:100-105 -- here the left
 * and right images of a pair are processed by the same launches, so one call covers both).
 */
#ifndef ORBX_H
#define ORBX_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORBX_VERSION 100

/* status codes (0 = success).  The C++ shim (include/orbx/orb_slam2_shim.hpp) rethrows them as the reference's
 * exception types from include/ORB_SLAM2/Error.h. */
#define ORBX_OK 0
#define ORBX_ERR_INVALID_ARG (-1)
#define ORBX_ERR_IMAGE_SIZE (-2)    /* ImageSizeError: a pyramid level is smaller than 2*19 px (src/ORBExtractor.cc:310-314),
                                       or too small for one 30-px FAST cell (the reference divides by zero, :340-343) */
#define ORBX_ERR_FILE_NOT_OPEN (-3) /* FileNotOpenError: BRIEF template file (src/ORBExtractor.cc:247-250) */
#define ORBX_ERR_CUDA (-4)
#define ORBX_ERR_NO_DEVICE (-5)
#define ORBX_ERR_CAPACITY (-6)      /* more frames than orbx_config.max_batch */
#define ORBX_ERR_STATE (-7)         /* e.g. orbx_get_pyramid before any frame was processed */
#define ORBX_ERR_COMM (-8)          /* NCCL missing / failed, or peers cannot reach each other's memory */

/* memory layout of cv::KeyPoint (28 bytes) so that results can be memcpy'd into std::vector<cv::KeyPoint> */
typedef struct orbx_keypoint {
  float x, y;      /* pt, level coordinates multiplied by the level scale factor (src/ORBExtractor.cc:408-409) */
  float size;      /* 7 (cv::FAST) */
  float angle;     /* degrees in (-180, 180]  (src/ORBExtractor.cc:407) */
  float response;  /* FAST score */
  int32_t octave;  /* pyramid level */
  int32_t class_id;/* -1 */
} orbx_keypoint;

#define ORBX_DESC_BYTES 32
#define ORBX_DEPTH_U16 0
#define ORBX_DEPTH_F32 1

/* Everything the reference reads from its YAML for this path (src/System.cc:27-73): ORBExtractor.* and Camera.* */
typedef struct orbx_config {
  int32_t width, height;   /* input image size (8-bit, single channel) */
  int32_t n_features;      /* ORBExtractor.nFeatures (1..65535: keypoint indices travel as uint16 in the row index / grid) */
  int32_t n_levels;        /* ORBExtractor.nLevels (1..16) */
  float scale_factor;      /* ORBExtractor.scaleFactor (> 1) */
  int32_t ini_th_fast;     /* ORBExtractor.iniThFAST */
  int32_t min_th_fast;     /* ORBExtractor.minThFAST */
  float fx, fy, cx, cy;    /* Camera.fx .. Camera.cy */
  float bf;                /* Camera::mfBf = fx * Camera.bl (src/System.cc:60) */
  float dist[5];           /* k1 k2 p1 p2 k3; undistortion is skipped when k1 == 0 (src/Camera.cc:31) */
  float depth_scale;       /* Camera.DepthScale (RGB-D) */
  int32_t max_batch;       /* frames one batch call may carry (>= 1) */
  int32_t device;          /* CUDA device ordinal, -1 = current device */
  const float *pattern;    /* 256 x (x1,y1,x2,y2) BRIEF test pairs, or NULL for the built-in bit_pattern_31_ */
} orbx_config;

typedef struct orbx_ctx orbx_ctx;

/* ---- life cycle ---------------------------------------------------------------------------------------- */
/* fills *cfg with the KITTI defaults of config/kitti_config_00.yaml */
void orbx_default_config(orbx_config *cfg);
/* replaces: ORBExtractor::ORBExtractor's table setup (initPyramid :283-317, initBriefTemplate, initMaxU) -- done once
 * per context instead of once per process/frame */
int orbx_create(const orbx_config *cfg, orbx_ctx **out);
void orbx_destroy(orbx_ctx *ctx);
const char *orbx_status_string(int status);
/* text of the last CUDA / argument error seen by this context ("" if none) */
const char *orbx_last_error(const orbx_ctx *ctx);
/* replaces: ORBExtractor::initBriefTemplate (src/ORBExtractor.cc:242-267): header line + 256 rows "x1 y1 x2 y2" */
int orbx_load_brief_template(const char *path, float *pattern_out /* [1024] */);
/* launch on this CUDA stream (cudaStream_t) instead of the context's own non-blocking stream; NULL restores the
 * context's own stream (pass cudaStreamLegacy / cudaStreamPerThread explicitly to use a default stream) */
int orbx_set_stream(orbx_ctx *ctx, void *cuda_stream);

/* Single-pair calls (orbx_stereo_frame, orbx_stereo_batch* with one frame) replay their launch sequence as ONE CUDA graph
 * captured at the first call (on by default; the legacy default stream cannot be captured and always takes plain launches).
 * enable = 0 restores plain stream launches (bench.py reports the p50 latency both ways).  Environment: ORBX_GRAPH=0. */
int orbx_set_graph(orbx_ctx *ctx, int enable);

/* ---- per-config tables ---------------------------------------------------------------------------------- */
/* replaces: ORBExtractor::getScaledFactors() (include/ORB_SLAM2/ORBExtractor.h:116), ORBExtractor::mnLevels,
 * mvnFeatures (:155) and the level sizes of getPyramid() */
int orbx_num_levels(const orbx_ctx *ctx);
int orbx_level_info(const orbx_ctx *ctx, int level, int32_t *width, int32_t *height, float *scale, int32_t *quota);

/* ---- single frame, host buffers (the reference's call surface) ---------------------------------------- */
/* replaces: ORBExtractor(image, ...) + ORBExtractor::extract(keyPoints, descriptors)
 * (include/ORB_SLAM2/ORBExtractor.h:107,110; src/ORBExtractor.cc:205-214,499-508).
 * kps: capacity n_features; desc: n_features x 32 bytes (row i is the reference's descriptors[i], a 1x32 CV_8U Mat). */
int orbx_extract(orbx_ctx *ctx, const uint8_t *image, size_t stride, orbx_keypoint *kps, uint8_t *desc, int32_t *n);

/* replaces: ORBExtractor::getPyramid() (include/ORB_SLAM2/ORBExtractor.h:113), Frame::getLeftPyramid/getRightPyramid
 * (include/ORB_SLAM2/Frame.h:346-347) for the most recent single-frame call.  side: 0 = left / mono, 1 = right.
 * blurred != 0 returns the Gaussian-blurred level (the private mvBriefMat, :152). */
int orbx_get_pyramid(orbx_ctx *ctx, int side, int level, int blurred, uint8_t *dst, size_t dst_stride);

/* replaces: Frame::createStereo (include/ORB_SLAM2/Frame.h:313-322) = Frame::Frame stereo ctor (src/Frame.cc:85-111:
 * two extractors, Camera::undistortPoints on the left keypoints) + ORBMatcher::searchByStereo (src/ORBMatcher.cc:18-81).
 * kps_left are the undistorted left keypoints (mvFeatsLeft), u_right / depth = mvFeatsRightU / mvDepths (-1 = none),
 * *n_matches = Frame::mnN.  Any output pointer may be NULL. */
int orbx_stereo_frame(orbx_ctx *ctx, const uint8_t *left, size_t left_stride, const uint8_t *right, size_t right_stride,
                      orbx_keypoint *kps_left, uint8_t *desc_left, int32_t *n_left, orbx_keypoint *kps_right,
                      uint8_t *desc_right, int32_t *n_right, double *u_right, double *depth, int32_t *n_matches);

/* replaces: Frame::createRGBD (include/ORB_SLAM2/Frame.h:325-331) = RGB-D ctor (src/Frame.cc:125-159).
 * depth_image: raw sensor depth (uint16 or float32, row stride in BYTES), divided by depth_scale on the fly.
 * kps_raw (optional) are the keypoints before undistortion (used for the lookup), kps the undistorted ones. */
int orbx_rgbd_frame(orbx_ctx *ctx, const uint8_t *gray, size_t gray_stride, const void *depth_image,
                    size_t depth_stride_bytes, int depth_type, orbx_keypoint *kps_raw, orbx_keypoint *kps,
                    uint8_t *desc, int32_t *n, double *u_right, double *depth);

/* replaces: VirtualFrame::initGrid (src/Frame.cc:53-69, called by both Frame ctors) for frame `frame` of the most recent
 * call: the 64x48-px bucket grid over the (undistorted) left keypoints, as a CSR.  rows/cols and the undistorted image
 * bounds mfMinU/mfMinV/mfMaxU/mfMaxV (include/ORB_SLAM2/Frame.h:33-43) come from orbx_grid_info.  cell_start has
 * rows*cols+1 entries; cell (r, c) lists entries[cell_start[r*cols+c] .. cell_start[r*cols+c+1]) in ascending order. */
int orbx_grid_info(const orbx_ctx *ctx, int32_t *rows, int32_t *cols, float *min_u, float *min_v, float *max_u, float *max_v);
int orbx_get_grid(orbx_ctx *ctx, int frame, int32_t *cell_start, int32_t *entries /* [n_features] */);

/* ---- batches (offline map / vocabulary building: frames are independent) -------------------------------- */
/* A sequence of n_frames stereo pairs (ANY length) from HOST memory; pinned memory makes the copies asynchronous.  The
 * frames stream through the context's max_batch device slots in chunks, so that the H2D copy of one chunk, the kernels of
 * another and the D2H copy of a third overlap.
 * left/right: frame f at base + f * frame_stride bytes, rows `stride` bytes apart (stride >= width and frame_stride >=
 * stride * (height - 1) + width, else ORBX_ERR_INVALID_ARG).  Outputs are fixed-stride arrays:
 * kps_*[f * n_features + i], desc_*[(f * n_features + i) * 32], u_right/depth[f * n_features + i], n_*[f].
 * Returns after all results have landed in the output arrays. */
int orbx_stereo_batch(orbx_ctx *ctx, int n_frames, const uint8_t *left, const uint8_t *right, size_t stride,
                      size_t frame_stride, orbx_keypoint *kps_left, uint8_t *desc_left, int32_t *n_left,
                      orbx_keypoint *kps_right, uint8_t *desc_right, int32_t *n_right, double *u_right, double *depth,
                      int32_t *n_matches);

/* device-resident results of the last *_device call; pointers stay valid until the next call on the context.
 * Image index: stereo frame f -> left image 2f, right image 2f+1; mono / RGB-D frame f -> image f. */
typedef struct orbx_device_results {
  const orbx_keypoint *kps;     /* [n_images][n_features] raw keypoints */
  const orbx_keypoint *kps_und; /* [n_images][n_features] undistorted keypoints (== kps when k1 == 0) */
  const uint8_t *desc;          /* [n_images][n_features][32] */
  const int32_t *n_kps;         /* [n_images] */
  const double *u_right;        /* [n_frames][n_features] */
  const double *depth;          /* [n_frames][n_features] */
  const int32_t *n_matches;     /* [n_frames] */
  int32_t n_images, n_frames, n_features;
  const int32_t *grid_start;    /* [n_frames][grid_rows * grid_cols + 1]  CSR of VirtualFrame::mGrids (src/Frame.cc:53-69) */
  const uint16_t *grid_entries; /* [n_frames][n_features] keypoint indices, ascending inside a cell */
  int32_t grid_rows, grid_cols;
} orbx_device_results;

/* same work as orbx_stereo_batch with inputs already in DEVICE memory; asynchronous on the context's stream
 * (orbx_set_stream); no host synchronisation. */
int orbx_stereo_batch_device(orbx_ctx *ctx, int n_frames, const uint8_t *d_left, const uint8_t *d_right, size_t stride,
                             size_t frame_stride, orbx_device_results *out);
/* mono extraction of n_images device-resident images (ORBExtractor only) */
int orbx_extract_batch_device(orbx_ctx *ctx, int n_images, const uint8_t *d_images, size_t stride, size_t frame_stride,
                              orbx_device_results *out);
/* RGB-D frames with device-resident gray + depth images (up to 2 * max_batch frames).  Depth frame f, row y starts at
 * d_depth + f * depth_frame_stride_bytes + y * depth_stride_bytes.  d_depth and both strides must be multiples of the
 * element size (2 for ORBX_DEPTH_U16, 4 for ORBX_DEPTH_F32), depth_stride_bytes >= width * element size and, for more
 * than one frame, depth_frame_stride_bytes >= depth_stride_bytes * (height - 1) + width * element size; otherwise
 * ORBX_ERR_INVALID_ARG before anything is enqueued. */
int orbx_rgbd_batch_device(orbx_ctx *ctx, int n_frames, const uint8_t *d_gray, size_t gray_stride,
                           size_t gray_frame_stride, const void *d_depth, size_t depth_stride_bytes,
                           size_t depth_frame_stride_bytes, int depth_type, orbx_device_results *out);
/* Every call that produces frames (extract / stereo / RGB-D / batch / sequence) bumps the context's epoch.  Frame-level
 * queries (orbx_get_grid, orbx_get_pyramid, orbx_search_in_area, orbx_serialize_keyframe, orbx_bow_transform ...) refer to
 * the most recent call: a caller that keeps several frames alive stores the epoch at creation and compares it before
 * querying (the C++ shim does, include/orbx/orb_slam2_shim.hpp). */
uint64_t orbx_frame_epoch(const orbx_ctx *ctx);
/* block until the context's stream is idle */
int orbx_synchronize(orbx_ctx *ctx);
/* synchronous device-to-host copy of `bytes` bytes of a device result array (after draining the context's stream) */
int orbx_read_device(orbx_ctx *ctx, const void *device_ptr, void *host_dst, size_t bytes);

/* ---- whole sequences sharded by frame over GPUs (BASELINE config 3; SURVEY.md section 8e) -------------------------- */
/* replaces: the dataset loop of the reference's examples (example/Stereo/KittiStereo.cc:28-37 -> Frame::createStereo,
 * include/ORB_SLAM2/Frame.h:313-322) for offline map / vocabulary building.  Frames are independent on this path: rank r
 * of R processes the contiguous block [r * ceil(F/R), min(F, (r + 1) * ceil(F/R))) of an F-frame sequence; the only
 * exchange is the gather of the left descriptors (+ counts), issued by the library itself.  One process (or host thread)
 * and one context per GPU. */
typedef struct orbx_comm orbx_comm;
#define ORBX_COMM_ID_BYTES 128  /* == NCCL_UNIQUE_ID_BYTES */
#define ORBX_IPC_HANDLE_BYTES 64 /* == sizeof(cudaIpcMemHandle_t) */
#define ORBX_TRANSPORT_NONE 0   /* single rank */
#define ORBX_TRANSPORT_NCCL 1   /* ncclSend/ncclRecv pieces on a side stream, overlapping the kernels of later chunks */
#define ORBX_TRANSPORT_PEER 2   /* descriptors are stored straight into every rank's gathered array (NVLink peer memory) by the
                                   kernel that assembles the records: gather fused into the producer, no separate collective */

/* the block of rank `rank` (lo inclusive, hi exclusive) */
void orbx_frame_range(int64_t n_frames_total, int rank, int world, int64_t *lo, int64_t *hi);
/* multi-process (one rank per process, e.g. under torchrun / mpirun): rank 0 calls orbx_comm_unique_id (ncclGetUniqueId) and
 * ships the bytes to the other ranks by any means; then EVERY rank calls orbx_comm_create (ncclCommInitRank: collective).
 * max_frames_total = longest sequence the communicator will carry (sizes the gathered arrays; all ranks must agree).
 * libnccl.so.2 is resolved with dlopen at the first call: ORBX_ERR_COMM if it is missing. */
int orbx_comm_unique_id(uint8_t *id /* [ORBX_COMM_ID_BYTES] */);
int orbx_comm_create(orbx_ctx *ctx, int rank, int world, const uint8_t *id, int64_t max_frames_total, orbx_comm **out);
/* optional, after orbx_comm_create: switch the data path to ORBX_TRANSPORT_PEER.  Every rank exports its gathered array
 * (orbx_comm_ipc_handle, a cudaIpcMemHandle_t), the caller all-gathers the handles, every rank maps them
 * (orbx_comm_open_peers: handles[r * ORBX_IPC_HANDLE_BYTES ..] = rank r's).  NCCL then only carries the closing barrier. */
int orbx_comm_ipc_handle(orbx_comm *comm, uint8_t *handle /* [ORBX_IPC_HANDLE_BYTES] */);
int orbx_comm_open_peers(orbx_comm *comm, const uint8_t *handles /* [world][ORBX_IPC_HANDLE_BYTES] */);
/* single process driving `world` contexts (same or different devices; one host thread each, or one thread calling the ranks
 * one after the other): ORBX_TRANSPORT_PEER without NCCL.  out[r] is rank r's communicator.  The gathered arrays are
 * complete on every rank once every rank's orbx_sequence_stereo call has returned. */
int orbx_comm_create_local(orbx_ctx *const *ctxs, int world, int64_t max_frames_total, orbx_comm **out /* [world] */);
void orbx_comm_destroy(orbx_comm *comm);
int orbx_comm_info(const orbx_comm *comm, int32_t *rank, int32_t *world, int32_t *transport);

/* One frame's results as ONE fixed-stride record, so that a chunk of frames leaves the device in a single copy:
 *   int32 n_left, n_right, n_matches (Frame::mnN), 0 at offset 0, then the arrays below (capacity n_features each; entries
 *   beyond the counts are zero).  kps_left are the undistorted left keypoints (mvFeatsLeft), kps_right the right ones. */
typedef struct orbx_record_layout {
  int64_t record_bytes;   /* multiple of 16 */
  int64_t off_kps_left;   /* orbx_keypoint[n_features] */
  int64_t off_desc_left;  /* uint8[n_features][32] */
  int64_t off_kps_right;
  int64_t off_desc_right;
  int64_t off_u_right;    /* double[n_features]  mvFeatsRightU */
  int64_t off_depth;      /* double[n_features]  mvDepths */
  int32_t n_features, reserved;
} orbx_record_layout;
int orbx_record_layout_get(const orbx_ctx *ctx, orbx_record_layout *out);

typedef struct orbx_sequence_io {
  const uint8_t *left, *right; /* THIS RANK'S block: local frame i (global lo + i) at base + i * frame_stride, rows `stride` apart */
  size_t stride, frame_stride;
  int32_t input_on_device;     /* 0: host memory (pinned makes the copies asynchronous); 1: device memory, read in place */
  int32_t records_on_device;   /* where `records` lives */
  void *records;               /* [n_local][record_stride] or NULL; 16-byte aligned */
  size_t record_stride;        /* >= orbx_record_layout.record_bytes, multiple of 16 */
  uint8_t *gathered_desc_host; /* optional host copies of the gathered arrays: [n_frames_total][n_features][32] / [n_frames_total] */
  int32_t *gathered_n_host;
} orbx_sequence_io;

typedef struct orbx_sequence_result {
  int64_t frame_lo, frame_hi;   /* this rank's block */
  int64_t block;                /* ceil(F / world) */
  const uint8_t *gathered_desc; /* DEVICE [world * block][n_features][32]: row f = left descriptors of global frame f (zero beyond its count) */
  const int32_t *gathered_n;    /* DEVICE [world * block]: left keypoints of global frame f (0 for the padding rows f >= F) */
  int32_t n_features, world;
} orbx_sequence_result;

/* Collective over the communicator (comm == NULL: a single rank).  Blocks until this rank's records have landed and -- NCCL /
 * multi-process transports -- the gathered arrays are complete on this rank.  The frames stream through the context's
 * max_batch device slots in chunks on the pipeline streams (H2D of one chunk, kernels of another, D2H of a third overlap). */
int orbx_sequence_stereo(orbx_ctx *ctx, orbx_comm *comm, int64_t n_frames_total, const orbx_sequence_io *io, orbx_sequence_result *out);

/* Offline map export: the same call, and in addition every frame of this rank's block as the orbslam2.KeyFrameData record
 * of a keyframe made from it (orbx_serialize_keyframe_bow, src/KeyFrame.cc:553-647,585-599).  After a chunk's records are
 * packed, three kernels run on its stream: the bag-of-words descent and assembly (VirtualFrame::computeBow,
 * include/ORB_SLAM2/Frame.h:224-231) and the serialiser.  Keyframe records stay on their rank; the descriptor gather is
 * unchanged.  Host outputs leave the device in one copy per chunk (and one copy of `sizes` at the end).  The BoW results
 * are not kept resident: orbx_search_by_bow still returns ORBX_ERR_STATE afterwards.  Write a KeyFrameList with
 * orbx_keyframe_list_head (rank 0 only, next_id = id0 + n_frames_total) and orbx_keyframe_list_entry_prefix. */
typedef struct orbx_keyframe_io {
  const struct orbx_vocab *vocab; /* NULL: fields 10 / 11 present but empty, as orbx_serialize_keyframe (must belong to this context) */
  int32_t levelsup;        /* 4 = VirtualFrame::computeBow (include/ORB_SLAM2/Frame.h:224-231) */
  int32_t with_map_points;
  uint64_t id0;            /* the record of GLOBAL frame f carries id id0 + f */
  const float *pose_rt;    /* [n_local][12] Tcw (R row-major, t) in the same memory as `out`, or NULL = identity */
  int32_t on_device;       /* where out / sizes / pose_rt live */
  uint8_t *out;            /* [n_local][stride], this rank's block; 16-byte aligned */
  size_t stride;           /* >= orbx_serialized_capacity_bow (vocab) / orbx_serialized_capacity (no vocab), multiple of 16 */
  int64_t *sizes;          /* [n_local] bytes of each record */
} orbx_keyframe_io;
int orbx_sequence_stereo_keyframes(orbx_ctx *ctx, orbx_comm *comm, int64_t n_frames_total, const orbx_sequence_io *io,
                                   const orbx_keyframe_io *kf, orbx_sequence_result *out);

/* ---- tracking-side Hamming matchers (SURVEY.md section 8(f) rank 2) -------------------------------------- */
/* One query of VirtualFrame::findFeaturesInArea (src/Frame.cc:286-311): the keypoint `kp` (position in undistorted
 * image coordinates + octave), the radius BEFORE its multiplication by getScaledFactor2(kp.octave), and the inclusive
 * octave range of the candidates. */
typedef struct orbx_area_query {
  float x, y;
  float radius;
  int32_t octave;
  int32_t min_level, max_level;
} orbx_area_query; /* 24 bytes */

/* replaces the inner step of both ORBMatcher::searchByProjection overloads (src/ORBMatcher.cc:296-343 constant-velocity /
 * fuse, :575-591 local map), against frame `frame` of the most recent stereo / RGB-D call (its keypoints, descriptors and
 * grid are resident on the device): for query i, candidates = findFeaturesInArea(kp, radius, min_level, max_level) in
 * the reference's order, minus those with exclude[idx] != 0 (the "already has a map point" filter, :322-331; NULL = keep
 * all), then ORBMatcher::getBestMatch (src/ORBMatcher.cc:967-990) with query_desc[i*32 .. +32).
 * Outputs (any may be NULL): best_idx[i] = index of the best candidate among the frame's left keypoints or -1 when no
 * candidate is left (the reference `continue`s), best_dist[i] = its Hamming distance (INT_MAX if none), ratio[i] =
 * float(best) / float(second) exactly as the reference computes it (its "second" ignores displaced minima),
 * n_candidates[i].  The caller applies `ratio < mfRatio && dist < mnMinThreshold`.
 * Windows that leave the grid are clipped (the reference indexes mGrids out of range there). */
int orbx_search_in_area(orbx_ctx *ctx, int frame, int n_queries, const orbx_area_query *queries,
                        const uint8_t *query_desc, const uint8_t *exclude /* [n_features] */, int32_t *best_idx,
                        int32_t *best_dist, float *ratio, int32_t *n_candidates);
/* same, for frames 0..n_frames-1 of the most recent *_device call, everything in DEVICE memory, asynchronous on the
 * context's stream: frame f uses d_queries[f * query_stride + i], i < d_n_queries[f] (NULL: query_stride queries each),
 * d_exclude[f * n_features + idx] (or NULL); outputs are [n_frames][query_stride]. */
int orbx_search_in_area_batch_device(orbx_ctx *ctx, int n_frames, int query_stride, const orbx_area_query *d_queries,
                                     const uint8_t *d_query_desc, const int32_t *d_n_queries, const uint8_t *d_exclude,
                                     int32_t *d_best_idx, int32_t *d_best_dist, float *d_ratio, int32_t *d_n_candidates);
/* replaces: ORBMatcher::verifyAngle (src/ORBMatcher.cc:1013-1051): keeps the matches that fall into the three fullest
 * of the 30 bins of angle(kps1[queryIdx]) - angle(kps2[trainIdx]); survivors are written back in place in the
 * reference's order (ascending bin, original order inside a bin); *n_out = their number. */
int orbx_verify_angle(orbx_ctx *ctx, int n_matches, int32_t *query_idx, int32_t *train_idx, float *distance,
                      const orbx_keypoint *kps1, int n1, const orbx_keypoint *kps2, int n2, int32_t *n_out);

/* ---- result serialisation (SURVEY.md section 8(f) rank 4) ------------------------------------------------- */
/* replaces: KeyFrame::serializeToProtobuf (src/KeyFrame.cc:553-647) for a keyframe made from frame `frame` of the most
 * recent stereo / RGB-D call: the orbslam2.KeyFrameData record (proto3 wire format, proto/Keyframe.proto:45-64) with
 * id, the undistorted image bounds, keypoints (x, y, octave, angle), right_u / depths narrowed to float, descriptors,
 * present-but-empty bow_vector / feature_vector, pose Tcw = pose_rt (R row-major [9] then t [3]; NULL = identity as in
 * the VirtualFrame ctor, include/ORB_SLAM2/Frame.h:44-45) and, if with_map_points, -1 for every keypoint's map point.
 * The record is assembled on the device; only its bytes are copied out.  *n_bytes is set even when cap is too small
 * (ORBX_ERR_CAPACITY).  A KeyFrameList (proto/Keyframe.proto:66-70) is these records as length-delimited field 3. */
int64_t orbx_serialized_capacity(const orbx_ctx *ctx); /* upper bound of one record for this context (multiple of 16) */
int orbx_serialize_keyframe(orbx_ctx *ctx, int frame, uint64_t id, const float *pose_rt /* [12] or NULL */,
                            int with_map_points, uint8_t *out, size_t cap, int64_t *n_bytes);
/* replaces: the TEXT variant of the same record, std::ostream &operator<<(std::ostream &, KeyFrame &) (src/KeyFrame.cc:423-533),
 * for a keyframe made from frame `frame`: optionally the one-off header line "nextId scale_0 .. scale_{L-1} " (:458-467), then
 * "id maxU maxV minU minV", the keypoints "x y octave angle rightU depth " each, the descriptors as decimal bytes, the empty
 * BoW / FeatureVector lines, the pose (R row-major then t), the empty connection / child / loop-edge lines and the map-point
 * ids (-1 each), every line closed by '\n' -- numbers exactly as the reference's stream prints them (operator<< of float /
 * double = "%g" with 6 significant digits).  This format is host-side glue in the reference and here: the arrays come back in
 * one copy per array and are formatted by the calling thread.  *n_bytes is set even when cap is too small (ORBX_ERR_CAPACITY). */
int orbx_serialize_keyframe_text(orbx_ctx *ctx, int frame, uint64_t id, const float *pose_rt /* [12] or NULL */, int with_map_points,
                                 int with_scale_header, uint64_t next_id, char *out, size_t cap, int64_t *n_bytes);
/* frames 0..n_frames-1 of the most recent *_device call into DEVICE memory, asynchronous on the context's stream: record f
 * (id = id0 + f, pose d_pose_rt[f * 12 ..] or identity) at d_out + f * frame_stride (>= orbx_serialized_capacity, both
 * 4-byte aligned), its size in d_sizes[f]. */
int orbx_serialize_keyframes_device(orbx_ctx *ctx, int n_frames, uint64_t id0, const float *d_pose_rt,
                                    int with_map_points, uint8_t *d_out, size_t frame_stride, int64_t *d_sizes);

/* The same record for a keyframe whose bag of words has been computed (src/KeyFrame.cc:553-647, fields 10 / 11 filled from
 * mBowVec / mFeatVec at :585-599): bow_vector = 10 { map<uint32, double> words = 1 } with one entry per word in ascending
 * word id (std::map order), key and value always written; feature_vector = 11 { repeated FeatureNode nodes = 1 } with the
 * nodes in ascending id, each { node_id = 1 (left out when 0), packed feature_ids = 2 in ascending feature index }.
 * The BoW of the frame(s) must be resident from orbx_bow_transform* on the same call's frames (as for orbx_search_by_bow):
 * ORBX_ERR_STATE otherwise.  Everything else is as orbx_serialize_keyframe / orbx_serialize_keyframes_device, with the
 * larger bound orbx_serialized_capacity_bow (multiple of 16). */
int64_t orbx_serialized_capacity_bow(const orbx_ctx *ctx);
int orbx_serialize_keyframe_bow(orbx_ctx *ctx, int frame, uint64_t id, const float *pose_rt /* [12] or NULL */,
                                int with_map_points, uint8_t *out, size_t cap, int64_t *n_bytes);
int orbx_serialize_keyframes_bow_device(orbx_ctx *ctx, int n_frames, uint64_t id0, const float *d_pose_rt,
                                        int with_map_points, uint8_t *d_out, size_t frame_stride, int64_t *d_sizes);

/* KeyFrameList { uint64 next_id = 1; repeated float scale_factors = 2; repeated KeyFrameData keyframes = 3 }
 * (proto/Keyframe.proto:66-70, writer src/Map.cc:205-224), written piecewise: the head (next_id, left out when 0, and the
 * context's level scale factors, packed), then for every record the prefix 0x1A varint(record_bytes) and the record.
 * A sharded export stays ONE list: rank 0 writes head + entries, every other rank entries only; the per-rank outputs
 * concatenated in rank order parse as a single KeyFrameList.  *n_bytes is set even when cap is too small. */
int orbx_keyframe_list_head(const orbx_ctx *ctx, uint64_t next_id, uint8_t *out, size_t cap, int64_t *n_bytes);
/* writes the entry prefix of a record of record_bytes bytes; returns its length (<= 11) or ORBX_ERR_INVALID_ARG */
int orbx_keyframe_list_entry_prefix(int64_t record_bytes, uint8_t *out /* [11] */);

/* ---- bag-of-words transform (SURVEY.md section 8(f) rank 3) ----------------------------------------------- */
/* A DBoW3::Vocabulary (the reference loads one in src/System.cc:93) resident on the context's device.  Records follow
 * the ORB-SLAM2 / DBoW3 text format the reference's README prescribes: record i describes node i + 1 (node 0 is the
 * root), `parent` precedes its children, word ids are assigned to the leaf records in order.
 * PARITY NOTE: DBoW3 is an un-vendored dependency of the reference and no vocabulary ships with it; these entry points
 * follow DBoW3's published algorithm (oracle/orb_oracle.c restates it) -- TF_IDF / TF weighting, L1-normalising scoring. */
typedef struct orbx_vocab orbx_vocab;
int orbx_vocab_create(orbx_ctx *ctx, int k, int L, int n_records, const int32_t *parent, const uint8_t *is_leaf,
                      const uint8_t *desc /* [n_records][32] */, const double *weight, orbx_vocab **out);
/* text file: "k L scoring weighting" then one "parent isLeaf d0 .. d31 weight" line per node (ORBvoc.txt) */
int orbx_vocab_load_text(orbx_ctx *ctx, const char *path, orbx_vocab **out);
void orbx_vocab_destroy(orbx_vocab *vocab);
int orbx_vocab_info(const orbx_vocab *vocab, int32_t *k, int32_t *L, int32_t *n_nodes, int32_t *n_words);

/* replaces: VirtualFrame::computeBow (include/ORB_SLAM2/Frame.h:224-231) = DBoW3::Vocabulary::transform(mvLeftDescriptor,
 * mBowVec, mFeatVec, levelsup = 4) for frame `frame` of the most recent stereo / RGB-D call.
 * BowVector (std::map<WordId, WordValue>): bow_ids ascending with their L1-normalised weights, *n_bow entries.
 * FeatureVector (std::map<NodeId, std::vector<unsigned>>): fv_nodes ascending, *n_fv_nodes of them; the features of node
 * j are fv_feats[fv_start[j] .. fv_start[j + 1]) in ascending feature index.  Arrays have n_features (+1 for fv_start)
 * entries; any array may be NULL. */
int orbx_bow_transform(orbx_ctx *ctx, const orbx_vocab *vocab, int frame, int levelsup, int32_t *bow_ids,
                       double *bow_vals, int32_t *n_bow, int32_t *fv_nodes, int32_t *fv_start, int32_t *fv_feats,
                       int32_t *n_fv_nodes);
/* device-resident results for frames 0..n_frames-1 of the most recent *_device call (asynchronous on the context's stream) */
typedef struct orbx_device_bow {
  const int32_t *bow_ids;   /* [n_frames][stride] */
  const double *bow_vals;   /* [n_frames][stride] */
  const int32_t *n_bow;     /* [n_frames] */
  const int32_t *fv_nodes;  /* [n_frames][stride] */
  const int32_t *fv_start;  /* [n_frames][stride + 1] */
  const int32_t *fv_feats;  /* [n_frames][stride] */
  const int32_t *n_fv_nodes; /* [n_frames] */
  int32_t stride;           /* n_features */
} orbx_device_bow;
int orbx_bow_transform_batch_device(orbx_ctx *ctx, const orbx_vocab *vocab, int n_frames, int levelsup, orbx_device_bow *out);

/* replaces the matching loop of ORBMatcher::searchByBow (src/ORBMatcher.cc:170-255) between frame `frame` of the most recent
 * call (whose FeatureVector must be resident: call orbx_bow_transform* for it first) and a keyframe given by its
 * FeatureVector (CSR: kf_fv_nodes ascending, kf_fv_start[n_kf_nodes + 1], kf_fv_feats) and descriptors kf_desc[n_kf][32].
 * kf_query_ok[pkId] != 0: this keyframe feature takes part (the MapPoint conditions of :195-212; NULL = all);
 * frame_cand_ok[pId] != 0: this frame feature may be matched (:216-233; NULL = all; n_features entries).
 * Outputs have one entry per kf_fv_feats entry e (the reference's visiting order): candidates = the frame's features under
 * the same vocabulary node that pass the mask, then ORBMatcher::getBestMatch (:238).  n_candidates[e] == 0 (best_idx -1)
 * when the node is not shared, the feature is masked or no candidate is left (the reference `continue`s).  The caller keeps
 * the rows with dist <= mnMinThreshold && !(ratio > mfRatio) (:240) and runs orbx_verify_angle (:248-249). */
int orbx_search_by_bow(orbx_ctx *ctx, int frame, int n_kf_nodes, const int32_t *kf_fv_nodes, const int32_t *kf_fv_start,
                       const int32_t *kf_fv_feats, const uint8_t *kf_desc, int n_kf, const uint8_t *kf_query_ok,
                       const uint8_t *frame_cand_ok, int32_t *best_idx, int32_t *best_dist, float *ratio,
                       int32_t *n_candidates);

/* ---- introspection for benchmarks / profiles ----------------------------------------------------------- */
#define ORBX_N_STAGES 7
/* Same work as orbx_stereo_batch_device, with a CUDA event recorded on the stream after every kernel; blocks until
 * done and returns the device time of each stage in milliseconds:
 * [0] pyramid level 0 (+blur)  [1] pyramid levels >= 1 (+blur)  [2] FAST cells  [3] quadtree  [4] orientation+BRIEF
 * [5] frame index (row index of the right keypoints + grid of the left ones)  [6] stereo match */
int orbx_profile_stereo_batch_device(orbx_ctx *ctx, int n_frames, const uint8_t *d_left, const uint8_t *d_right,
                                     size_t stride, size_t frame_stride, float *stage_ms /* [ORBX_N_STAGES] */);
/* name of stage i of the list above */
const char *orbx_stage_name(int stage);
/* number of kernels this library launched on the context since creation (bench.py's gpu_launches) */
int64_t orbx_launch_count(const orbx_ctx *ctx);
/* algorithmic bytes of one stereo frame / one mono image at this configuration (SURVEY.md section 8d) */
int64_t orbx_algorithmic_bytes(const orbx_ctx *ctx, int stereo);

/* ---- stage-level read-back for parity tests (results of the most recent call; synchronises the stream) ---- */
/* FAST corners of one level in the reference's detection order (cell-row-major, row-major inside a cell), in ROI
 * coordinates as in src/ORBExtractor.cc:368-372, i.e. the `levelKps` handed to the Quadtree (:376) */
int orbx_debug_level_corners(orbx_ctx *ctx, int image, int level, int32_t *xs, int32_t *ys, int32_t *scores, int cap,
                             int32_t *n);
/* quadtree survivors of one level (level coordinates, ascending detection index): Quadtree::getFeatIdxs (:378-386) */
int orbx_debug_level_selected(orbx_ctx *ctx, int image, int level, int32_t *xs, int32_t *ys, int32_t *scores, int cap,
                              int32_t *n);
/* How many (image, level) quadtree problems this context solved with the loop-free formulation of Quadtree::split() and how
 * many needed the sequential loop (corners that must be split below the key depth, nodes whose corners all sit on split
 * lines, more than 8 root strips, quota < 2, levels denser than the shared-memory list).  ORBX_QT_FAST=0 forces the loop.
 * phase_cycles (optional, [8]): SM clock cycles the loop-free problems spent per phase, summed over problems (table nodes |
 * level-by-level descent | stop bucket | responses + pop ranks | leaves | surplus + flags | unused | unused). */
int orbx_debug_quadtree_stats(orbx_ctx *ctx, int64_t *fast, int64_t *sequential, int64_t *phase_cycles);
/* Runs ONLY the quadtree kernel (Quadtree::split + nodes2kpoints, src/ORBExtractor.cc:126-192) of image 0 on a caller-
 * supplied corner list for `level` (ROI coordinates, detection order; the other levels get no corners), so that the
 * kernel can be checked against the reference on arbitrary inputs: corners on split lines, starved levels, deep nodes.
 * Read the result with orbx_debug_level_selected(ctx, 0, level, ...). */
int orbx_debug_run_quadtree(orbx_ctx *ctx, int level, const int32_t *xs, const int32_t *ys, const int32_t *scores, int n);

#ifdef __cplusplus
}
#endif
#endif /* ORBX_H */
