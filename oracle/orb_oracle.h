/*
 * orb_oracle.h -- CPU restatement of the ORB_SLAM2_ROS2 per-frame feature front-end.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it,
 * and only as the checker (or the timed CPU baseline), never as a fallback for the CUDA path.
 *
 * Pinning status: the reference ships no golden vectors for this path (SURVEY.md section 4), so the
 * oracle is pinned by (i) cv2 4.13.0 for the OpenCV primitives (resize / GaussianBlur / FAST /
 * undistortPoints; tests/test_oracle_cv2.py) and (ii) the reference's own ORBExtractor.cc and the
 * searchByStereo line ranges of ORBMatcher.cc compiled unmodified against oracle/stub
 * (oracle/_ref, tests/test_oracle_vs_ref.py), plus committed fixtures under tests/golden/.
 *
 * All citations are relative to /root/reference/src/ORB_SLAM2/.
 */
#ifndef ORB_ORACLE_H
#define ORB_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* cv::KeyPoint memory layout (28 bytes). */
typedef struct oracle_keypoint {
  float x, y, size, angle, response;
  int32_t octave, class_id;
} oracle_keypoint;

#define ORACLE_MAX_LEVELS 32

/* ---- per-config tables: src/ORBExtractor.cc:283-317 ---- */
void oracle_scale_factors(float scale_factor, int n_levels, float *sf);
void oracle_level_quotas(int n_features, float scale_factor, int n_levels, int *quota);
/* returns 0, or -1 when a level is smaller than 2*19 px (ImageSizeError, :310-314) */
int oracle_level_sizes(int width, int height, const float *sf, int n_levels, int *lw, int *lh);
/* src/ORBExtractor.cc:217-236 */
void oracle_umax(int *umax /*[16]*/);

/* ---- OpenCV primitives (bit-exact restatements, checked against cv2 4.13.0) ---- */
/* cv::resize(src, dst, Size(dw,dh), 0, 0, INTER_LINEAR) for 8UC1 */
void oracle_resize_linear_u8(const uint8_t *src, int sw, int sh, size_t sstride, uint8_t *dst, int dw, int dh,
                             size_t dstride);
/* cv::GaussianBlur(src, dst, Size(7,7), 2, 2, BORDER_REFLECT_101) for 8UC1 */
void oracle_gaussian_blur7_u8(const uint8_t *src, int w, int h, size_t sstride, uint8_t *dst, size_t dstride);
/* cv::FAST(patch, kps, threshold, true): TYPE_9_16 + non-max suppression.  Output row-major.
 * Returns the number of keypoints (at most cap are written). */
int oracle_fast9_nms(const uint8_t *img, int w, int h, size_t stride, int threshold, int *xs, int *ys, int *scores,
                     int cap);
/* the per-pixel FAST-9 arc value m (corner at threshold t iff m > t; cv score = m - 1) */
int oracle_fast9_arc_value(const uint8_t *p, size_t stride);
/* cv::undistortPoints(pts, pts, K, D, noArray(), K): 5 fixed-point iterations in double */
void oracle_undistort_points(float *xy, int n, float fx, float fy, float cx, float cy, const float *dist, int n_dist);

/* ---- extractor stages ---- */
/* src/ORBExtractor.cc:331-375: per-cell FAST with threshold fallback over one level image.
 * Writes ROI coordinates (level coords minus 16) in detection order. Returns count (<= cap written). */
int oracle_fast_cells(const uint8_t *img, int w, int h, size_t stride, int ini_th, int min_th, int *xs, int *ys,
                      int *scores, int cap, int *n_fallback_cells);
/* src/ORBExtractor.cc:19-192: priority quadtree. xs/ys are ROI coords, returns the number of selected indices
 * (ascending) written to out_idx (capacity need). n_pops (optional) receives the number of loop iterations. */
int oracle_quadtree_select(int roi_w, int roi_h, int n, const float *xs, const float *ys, const float *resp, int need,
                           int *out_idx, long *n_pops);
/* src/ORBExtractor.cc:465-487 */
double oracle_ic_angle(const uint8_t *img, size_t stride, int x, int y);
/* src/ORBExtractor.cc:427-456,534-540; pattern = 256 x (x1,y1,x2,y2) floats */
void oracle_brief(const uint8_t *blurred, size_t stride, float px, float py, double theta, const float *pattern,
                  uint8_t *desc /*[32]*/);

typedef struct oracle_pyramid {
  int n_levels;
  int w[ORACLE_MAX_LEVELS], h[ORACLE_MAX_LEVELS];
  float sf[ORACLE_MAX_LEVELS];
  int quota[ORACLE_MAX_LEVELS];
  uint8_t *img[ORACLE_MAX_LEVELS];  /* dense rows (stride == w) */
  uint8_t *blur[ORACLE_MAX_LEVELS]; /* dense rows */
} oracle_pyramid;

/* ORBExtractor ctor (:205-214 -> initPyramid :278-320). Returns 0 / -1 (ImageSizeError). */
int oracle_pyramid_build(oracle_pyramid *p, const uint8_t *img, int w, int h, size_t stride, int n_features,
                         int n_levels, float scale_factor);
void oracle_pyramid_free(oracle_pyramid *p);

/* ORBExtractor::extract (:499-508): kps (cap n_features), desc (n x 32), angles_rad optional (double theta). */
int oracle_extract(const oracle_pyramid *p, int ini_th, int min_th, const float *pattern, oracle_keypoint *kps,
                   uint8_t *desc, double *angles_rad, int *level_counts /*[n_levels] optional*/);

/* ---- stereo / RGB-D association ---- */
/* src/ORBMatcher.cc:18-81 (+ :841-1011). kps_left are the (undistorted) left keypoints. Returns nMatches.  A match whose
 * SAD window leaves its level image is dropped, where the reference throws (DESIGN section 2). */
int oracle_search_by_stereo(const oracle_pyramid *left, const oracle_pyramid *right, const oracle_keypoint *kl,
                            const uint8_t *dl, int nl, const oracle_keypoint *kr, const uint8_t *dr, int nr, float fx,
                            float bf, double *u_right, double *depth, int *match_idx /*optional [nl]*/);
/* src/Frame.cc:125-159. depth_raw: u16 (is_float=0) or f32 (is_float=1) H x W image, dense stride in elements. */
void oracle_rgbd_lookup(const void *depth_raw, int is_float, int w, int h, size_t stride_elems, float depth_scale,
                        const oracle_keypoint *kps_raw, const oracle_keypoint *kps_undist, int n, float bf,
                        double *u_right, double *depth);

/* ---- tracking-side area matchers (SURVEY section 8(f) rank 2) ---- */
typedef struct oracle_area_query {
  float x, y;     /* kp.pt */
  float radius;   /* before the sf[octave]^2 scaling of findFeaturesInArea */
  int32_t octave; /* kp.octave */
  int32_t min_level, max_level;
} oracle_area_query;

/* VirtualFrame::initGrid, src/Frame.cc:53-69 -> CSR (start[rows*cols+1], entries[n]) */
void oracle_init_grid(const oracle_keypoint *kps, int n, float min_u, float min_v, float max_u, float max_v, int *rows_out,
                      int *cols_out, int *start, int cap_cells, int *entries);
/* VirtualFrame::findFeaturesInArea, src/Frame.cc:286-311 */
int oracle_find_features_in_area(const oracle_keypoint *kps, const int *start, const int *entries, int rows, int cols,
                                 const float *sf, float max_u, float max_v, float x, float y, float radius, int octave,
                                 int min_level, int max_level, int *out);
/* ORBMatcher::getBestMatch, src/ORBMatcher.cc:967-990; returns the best candidate's index */
int oracle_best_match(const uint8_t *desc, const uint8_t *cand_desc, const int *cand_idx, int n, int *best_dist,
                      float *ratio);
/* inner step of ORBMatcher::searchByProjection, src/ORBMatcher.cc:296-343 / :575-591 */
void oracle_search_in_area(const oracle_keypoint *kps, const uint8_t *desc, int n_kps, const int *start,
                           const int *entries, int rows, int cols, const float *sf, float max_u, float max_v,
                           const oracle_area_query *q, const uint8_t *q_desc, int n_q, const uint8_t *exclude,
                           int *best_idx, int *best_dist, float *ratio, int *n_cand);
/* ORBMatcher::verifyAngle, src/ORBMatcher.cc:1013-1051 (in place; returns the new count) */
int oracle_verify_angle(int n, int *query_idx, int *train_idx, float *distance, const oracle_keypoint *kps1,
                        const oracle_keypoint *kps2);

/* ---- result serialisation (SURVEY section 8(f) rank 4) ---- */
/* orbslam2.KeyFrameData bytes (proto/Keyframe.proto:45-64) as written by KeyFrame::serializeToProtobuf
 * (src/KeyFrame.cc:553-647) for a keyframe made from a fresh frame.  Returns the size, 0 if cap is too small. */
size_t oracle_serialize_keyframe(const oracle_keypoint *kps, const uint8_t *desc, const double *u_right,
                                 const double *depth, int n, uint64_t id, float max_u, float max_v, float min_u,
                                 float min_v, const float *pose_rt, int with_map_points, uint8_t *out, size_t cap);

/* ---- bag-of-words transform (SURVEY section 8(f) rank 3; PARITY UNPINNED, see orb_oracle.c) ---- */
/* A DBoW3 vocabulary tree: node 0 is the root; the children of node i are child_ids[child_start[i] .. child_start[i+1])
 * in id order; leaves carry a word id (internal nodes -1) and a weight. */
typedef struct oracle_vocab {
  int32_t k, L, n_nodes;
  const int32_t *child_start; /* [n_nodes + 1] */
  const int32_t *child_ids;   /* [n_nodes - 1] */
  const uint8_t *desc;        /* [n_nodes][32] */
  const double *weight;       /* [n_nodes] */
  const int32_t *word_id;     /* [n_nodes] */
} oracle_vocab;

void oracle_bow_descend(const oracle_vocab *v, const uint8_t *desc, int levelsup, int32_t *word_id, double *weight,
                        int32_t *nid);
int oracle_bow_transform(const oracle_vocab *v, const uint8_t *desc, int n, int levelsup, int32_t *bow_ids,
                         double *bow_vals, int32_t *fv_nodes, int32_t *fv_start, int32_t *fv_feats, int *fv_count);

/* matching loop of ORBMatcher::searchByBow, src/ORBMatcher.cc:170-255 (masks instead of MapPoint objects); FeatureVectors
 * as CSRs (nodes ascending, start[n+1], feature indices).  Returns the number of output rows. */
int oracle_search_by_bow(const int32_t *f_nodes, const int32_t *f_start, const int32_t *f_feats, int f_n_nodes,
                         const uint8_t *f_desc, const uint8_t *frame_cand_ok, const int32_t *k_nodes,
                         const int32_t *k_start, const int32_t *k_feats, int k_n_nodes, const uint8_t *k_desc,
                         const uint8_t *kf_query_ok, int32_t *kf_idx, int32_t *best_idx, int32_t *best_dist,
                         float *ratio, int32_t *n_cand);

#ifdef __cplusplus
}
#endif
#endif
