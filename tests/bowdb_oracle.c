/* bowdb_oracle.c -- plain-C restatement of the keyframe database (orbx_bowdb_*, include/orbx.h): the first stage of ORB-SLAM2's
 * KeyFrameDatabase::DetectLoopCandidates with DBoW3's L1Scoring::score, sequentially, over BowVectors the caller computed with
 * oracle_bow_transform (oracle/orb_oracle.c).  Compiled with -ffp-contract=off so that every double operation rounds once.
 *
 *   oracle_bowdb_query(ids, vals, n, stride, n_frames, n_words,     the database: frame f's BowVector = ids / vals + f * stride, n[f]
 *                      q_ids, q_vals, q_n, q_stride, n_queries,    the queries: query i's BowVector = q_ids / q_vals + i * q_stride
 *                      q_frame0, window,                           query i is frame q_frame0 + i; window < 0: nothing excluded
 *                      min_score, top_k,
 *                      cand_frame, cand_score, cand_common,        [n_queries][top_k]
 *                      counts)                                     [n_queries][4]: n_sharing, max_common, n_scored, n_kept
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

typedef struct
{
  float score;
  int32_t frame;
} kept_t;

/* score descending, then frame ascending */
static int cmp_kept(const void *a, const void *b)
{
  const kept_t *x = (const kept_t *)a, *y = (const kept_t *)b;
  if (x->score != y->score) return x->score > y->score ? -1 : 1;
  return (x->frame > y->frame) - (x->frame < y->frame);
}

/* the first position in ids[lo .. hi) whose id is >= w (std::map::lower_bound) */
static int64_t lower_bound(const int32_t *ids, int64_t lo, int64_t hi, int32_t w)
{
  while (lo < hi)
  {
    const int64_t mid = lo + (hi - lo) / 2;
    if (ids[mid] < w) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

/* DBoW3 L1Scoring::score(v1, v2) */
static double l1_score(const int32_t *i1, const double *v1, int64_t n1, const int32_t *i2, const double *v2, int64_t n2)
{
  int64_t a = 0, b = 0;
  double score = 0;
  while (a < n1 && b < n2)
  {
    const double vi = v1[a], wi = v2[b];
    if (i1[a] == i2[b])
    {
      score += fabs(vi - wi) - fabs(vi) - fabs(wi);
      ++a;
      ++b;
    }
    else if (i1[a] < i2[b])
      a = lower_bound(i1, a, n1, i2[b]);
    else
      b = lower_bound(i2, b, n2, i1[a]);
  }
  score = -score / 2.0;
  return score;
}

int oracle_bowdb_query(const int32_t *ids, const double *vals, const int32_t *n, int64_t stride, int32_t n_frames, int32_t n_words,
                       const int32_t *q_ids, const double *q_vals, const int32_t *q_n, int64_t q_stride, int32_t n_queries, int64_t q_frame0,
                       int32_t window, float min_score, int32_t top_k, int32_t *cand_frame, float *cand_score, int32_t *cand_common,
                       int32_t *counts)
{
  /* the inverted file: per word, the frames that hold it, in frame order (KeyFrameDatabase::add) */
  int64_t *start = calloc((size_t)n_words + 1, sizeof(int64_t));
  int64_t total = 0;
  for (int32_t f = 0; f < n_frames; ++f) total += n[f];
  int32_t *post = malloc((size_t)(total > 0 ? total : 1) * sizeof(int32_t));
  int64_t *cur = malloc(((size_t)n_words + 1) * sizeof(int64_t));
  int32_t *loop_query = malloc((size_t)n_frames * sizeof(int32_t)), *loop_words = calloc((size_t)n_frames, sizeof(int32_t));
  int32_t *sharing = malloc((size_t)n_frames * sizeof(int32_t));
  kept_t *kept = malloc((size_t)n_frames * sizeof(kept_t));
  if (!start || !post || !cur || !loop_query || !loop_words || !sharing || !kept) return -1;
  for (int32_t f = 0; f < n_frames; ++f)
    for (int32_t j = 0; j < n[f]; ++j)
    {
      if (ids[f * stride + j] < 0 || ids[f * stride + j] >= n_words) return -1;
      ++start[ids[f * stride + j] + 1];
    }
  for (int32_t w = 0; w < n_words; ++w) start[w + 1] += start[w];
  for (int32_t w = 0; w <= n_words; ++w) cur[w] = start[w];
  for (int32_t f = 0; f < n_frames; ++f)
    for (int32_t j = 0; j < n[f]; ++j) post[cur[ids[f * stride + j]]++] = f;
  for (int32_t f = 0; f < n_frames; ++f) loop_query[f] = -1;

  for (int32_t qi = 0; qi < n_queries; ++qi)
  {
    const int32_t *qd = q_ids + qi * q_stride;
    const double *qv = q_vals + qi * q_stride;
    const int64_t qf = q_frame0 + qi;
    int32_t n_sharing = 0, max_common = 0, n_scored = 0, n_kept = 0;
    /* mnLoopQuery / mnLoopWords as in DetectLoopCandidates */
    for (int32_t j = 0; j < q_n[qi]; ++j)
    {
      const int32_t w = qd[j];
      for (int64_t p = start[w]; p < start[w + 1]; ++p)
      {
        const int32_t f = post[p];
        if (loop_query[f] != qi)
        {
          loop_words[f] = 0;
          const int connected = window >= 0 && llabs((long long)f - (long long)qf) <= window;
          if (!connected)
          {
            loop_query[f] = qi;
            sharing[n_sharing++] = f;
          }
        }
        ++loop_words[f];
      }
    }
    if (n_sharing > 0)
    {
      for (int32_t i = 0; i < n_sharing; ++i)
        if (loop_words[sharing[i]] > max_common) max_common = loop_words[sharing[i]];
      const int min_common = max_common * 0.8f;
      for (int32_t i = 0; i < n_sharing; ++i)
      {
        const int32_t f = sharing[i];
        if (loop_words[f] > min_common)
        {
          ++n_scored;
          const float si = (float)l1_score(qd, qv, q_n[qi], ids + f * stride, vals + f * stride, n[f]);
          if (si >= min_score)
          {
            kept[n_kept].score = si;
            kept[n_kept].frame = f;
            ++n_kept;
          }
        }
      }
      qsort(kept, (size_t)n_kept, sizeof(kept_t), cmp_kept);
    }
    for (int32_t t = 0; t < top_k; ++t)
    {
      cand_frame[(int64_t)qi * top_k + t] = t < n_kept ? kept[t].frame : -1;
      cand_score[(int64_t)qi * top_k + t] = t < n_kept ? kept[t].score : 0.f;
      cand_common[(int64_t)qi * top_k + t] = t < n_kept ? loop_words[kept[t].frame] : 0;
    }
    counts[4 * qi] = n_sharing, counts[4 * qi + 1] = max_common, counts[4 * qi + 2] = n_scored, counts[4 * qi + 3] = n_kept;
  }
  free(start);
  free(post);
  free(cur);
  free(loop_query);
  free(loop_words);
  free(sharing);
  free(kept);
  return 0;
}
