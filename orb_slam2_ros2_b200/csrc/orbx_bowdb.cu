// orbx_bowdb.cu -- keyframe database: BoW inverted file and loop / relocalisation candidates (orbx_bowdb_*), sm_100a.
//
// Restates the first stage of ORB-SLAM2's KeyFrameDatabase::DetectLoopCandidates / DetectRelocalizationCandidates with
// DBoW3's L1Scoring::score under the rules of include/orbx.h; tests/bowdb_oracle.c is the sequential restatement the kernels
// are tested against bit for bit.
//   build: the BowVectors of every frame come from bow_descend_kernel + bow_assemble_kernel (orbx_bow.cu) in chunks of
//   frames; the inverted file is a CSR by word:
//     bowdb_word_count_kernel   postings per word (one integer atomic per BowVector entry)
//     bowdb_scan_kernel         exclusive scan over the words (one CTA: a serial run per thread + a block scan)
//     bowdb_fill_kernel         frame ids into the postings (order inside a word is not observable: counts are integers)
//   query: bowdb_query_kernel, one CTA per query (a grid-stride loop over the queries):
//     counting   per query word, its postings add 1 to a 16-bit shared-word counter of the frame; two counters share one
//                32-bit shared-memory word (a count never exceeds the query's n_bow <= 65535: no carry crosses over)
//     selection  connected frames masked; n_sharing / max_common by block reduction; the frames with common > min_common
//                compacted in ascending frame order into a list (shared memory when it fits beside the counters, else a
//                per-CTA slice of global scratch)
//     scoring    a warp per candidate: lanes look the candidate's words up in the query's (both ascending), compute their
//                term, and lane 0 adds the terms as one serial chain in ascending word id (__dadd_rn) -- DBoW's loop
//     output     (score desc, frame asc) packed into 64-bit keys, bitonic sort of the kept ones, the first top_k written
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "orbx_internal.h"
#include "orbx_match.cuh"

struct orbx_bowdb
{
  const orbx_ctx *ctx = nullptr;
  const orbx_vocab *vocab = nullptr;
  int device = 0;
  int F = 0, stride = 0, n_words = 0;
  long long n_postings = 0;
  int *ids = nullptr;       // [F][stride] BowVector word ids, ascending
  double *vals = nullptr;   // [F][stride] their L1-normalised weights
  int *n = nullptr;         // [F]
  long long *word_start = nullptr; // [n_words + 1]
  int *post = nullptr;      // [n_postings] frame ids, grouped by word
  // query launch shape, fixed at build time
  int P = 0;                // power of two >= F: capacity of one candidate list
  size_t smem = 0;          // dynamic shared memory of the query kernel
  int list_in_smem = 0;
  int grid_max = 0;         // resident CTAs of the query kernel on the device
  unsigned long long *g_list = nullptr; // [grid_max][P] when the list does not fit beside the counters
  orbx::DeviceBuffer staging; // outputs of host-output queries
};

namespace orbx
{

namespace
{

constexpr int kQT = 256; // threads of the query CTA
constexpr unsigned kFull = 0xffffffffu;
constexpr unsigned long long kNone = ~0ull; // a list slot holding no kept candidate (sorts last)
constexpr size_t kSmemOptIn = 227 * 1024;  // shared memory one CTA may opt in to on sm_100
constexpr size_t kCounterBytes = (size_t)(ORBX_BOWDB_MAX_FRAMES + 1) / 2 * 4;
static_assert(kCounterBytes + 2048 <= kSmemOptIn, "ORBX_BOWDB_MAX_FRAMES counters must fit the query kernel's shared memory");

__global__ void __launch_bounds__(256) bowdb_word_count_kernel(const int *ids, const int *n, int stride, long long total, long long *cnt)
{
  const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
  if (e >= total) return;
  const long long f = e / stride;
  if ((int)(e - f * stride) < n[f]) atomicAdd((unsigned long long *)&cnt[ids[e]], 1ull);
}

// exclusive scan of cnt[0 .. n) in place (cnt[n] = total), one CTA of 1024 threads
__global__ void __launch_bounds__(1024) bowdb_scan_kernel(long long *cnt, int n)
{
  __shared__ long long s_warp[32];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int per = (n + 1023) / 1024, j0 = min(tid * per, n), j1 = min(j0 + per, n);
  long long mine = 0;
  for (int j = j0; j < j1; ++j) mine += cnt[j];
  long long inc = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1)
  {
    const long long t = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_warp[wid] = inc;
  __syncthreads();
  long long base = 0, tot = 0;
  for (int w = 0; w < 32; ++w)
  {
    if (w < wid) base += s_warp[w];
    tot += s_warp[w];
  }
  long long run = base + inc - mine;
  for (int j = j0; j < j1; ++j)
  {
    const long long c = cnt[j];
    cnt[j] = run;
    run += c;
  }
  if (tid == 0) cnt[n] = tot;
}

__global__ void __launch_bounds__(256) bowdb_fill_kernel(const int *ids, const int *n, int stride, long long total, const long long *start,
                                                         unsigned long long *cursor, int *post)
{
  const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
  if (e >= total) return;
  const long long f = e / stride;
  if ((int)(e - f * stride) >= n[f]) return;
  const int w = ids[e];
  post[start[w] + (long long)atomicAdd(&cursor[w], 1ull)] = (int)f;
}

struct QueryArgs
{
  // database
  const int *ids, *n;
  const double *vals;
  long long stride;
  const long long *word_start;
  const int *post;
  int F, P, list_in_smem;
  unsigned long long *g_list;
  // queries: query i has the BowVector q_ids / q_vals + i * q_stride, q_n[i] entries, and is frame q_frame0 + i
  const int *q_ids, *q_n;
  const double *q_vals;
  long long q_stride, q_frame0;
  int window; // < 0: nothing excluded
  int n_queries, top_k;
  float min_score;
  int *cand_frame, *cand_common, *n_sharing, *max_common, *n_scored, *n_kept;
  float *cand_score;
};

// float -> unsigned whose ascending order is the float's ascending order (and back)
__device__ __forceinline__ unsigned float_key(float x)
{
  const unsigned u = __float_as_uint(x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_float(unsigned k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

__device__ __forceinline__ int counter_of(const unsigned *cnt, int f) { return (int)((cnt[f >> 1] >> (16 * (f & 1))) & 0xffffu); }

__global__ void __launch_bounds__(kQT) bowdb_query_kernel(const QueryArgs a)
{
  extern __shared__ __align__(16) unsigned char smem[];
  unsigned *cnt = reinterpret_cast<unsigned *>(smem); // [(F + 1) / 2]: 16-bit counters
  const size_t cnt_bytes = (((size_t)(a.F + 1) / 2 * 4) + 15) & ~(size_t)15;
  unsigned long long *list = a.list_in_smem ? reinterpret_cast<unsigned long long *>(smem + cnt_bytes) : a.g_list + (size_t)blockIdx.x * a.P;
  __shared__ int s_warp[kQT / 32], s_red[2][kQT / 32];
  __shared__ int s_kept;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int n_cnt = (a.F + 1) / 2;
  for (int qi = blockIdx.x; qi < a.n_queries; qi += gridDim.x)
  {
    const int *q_ids = a.q_ids + (size_t)qi * a.q_stride;
    const double *q_vals = a.q_vals + (size_t)qi * a.q_stride;
    const int nq = a.q_n[qi];
    const long long qf = a.q_frame0 + qi;
    for (int i = tid; i < n_cnt; i += kQT) cnt[i] = 0;
    if (tid == 0) s_kept = 0;
    __syncthreads();
    // counting: a warp per query word, lanes over its postings
    for (int j = wid; j < nq; j += kQT / 32)
    {
      const int w = q_ids[j];
      const long long p1 = a.word_start[w + 1];
      for (long long p = a.word_start[w] + lane; p < p1; p += 32)
      {
        const int f = a.post[p];
        atomicAdd(&cnt[f >> 1], 1u << (16 * (f & 1)));
      }
    }
    __syncthreads();
    // selection: connected frames masked, then n_sharing / max_common over each thread's contiguous run of frames
    const int per = (a.F + kQT - 1) / kQT, f0 = min(tid * per, a.F), f1 = min(f0 + per, a.F);
    auto common_of = [&](int f) -> int {
      if (a.window >= 0 && llabs((long long)f - qf) <= a.window) return 0;
      return counter_of(cnt, f);
    };
    int sharing = 0, mx = 0;
    for (int f = f0; f < f1; ++f)
    {
      const int c = common_of(f);
      sharing += c > 0;
      mx = max(mx, c);
    }
    for (int o = 16; o > 0; o >>= 1)
    {
      sharing += __shfl_xor_sync(kFull, sharing, o);
      mx = max(mx, __shfl_xor_sync(kFull, mx, o));
    }
    if (lane == 0) s_red[0][wid] = sharing, s_red[1][wid] = mx;
    __syncthreads();
    sharing = 0, mx = 0;
    for (int w = 0; w < kQT / 32; ++w) sharing += s_red[0][w], mx = max(mx, s_red[1][w]);
    // int minCommonWords = maxCommonWords * 0.8f  (KeyFrameDatabase.cc)
    const int min_common = (int)((float)mx * 0.8f);
    int mine = 0;
    if (sharing > 0)
      for (int f = f0; f < f1; ++f) mine += common_of(f) > min_common;
    int n_sc;
    int pos = block_exscan<kQT>(mine, &n_sc, s_warp);
    if (sharing > 0)
      for (int f = f0; f < f1; ++f)
        if (common_of(f) > min_common) list[pos++] = (unsigned long long)f;
    __syncthreads();
    // scoring: a warp per candidate
    for (int ci = wid; ci < n_sc; ci += kQT / 32)
    {
      const int g = (int)list[ci];
      const int *g_ids = a.ids + (size_t)g * a.stride;
      const double *g_vals = a.vals + (size_t)g * a.stride;
      const int m = a.n[g];
      double score = 0.0; // lane 0's chain
      for (int base = 0; base < m; base += 32)
      {
        const int j = base + lane;
        bool hit = false;
        double t = 0.0;
        if (j < m)
        {
          const int w = g_ids[j];
          int lo = 0, hi = nq; // lower_bound of w in the query's ids
          while (lo < hi)
          {
            const int mid = (lo + hi) >> 1;
            if (q_ids[mid] < w) lo = mid + 1;
            else hi = mid;
          }
          if (lo < nq && q_ids[lo] == w)
          {
            hit = true;
            const double vi = q_vals[lo], wi = g_vals[j];
            t = __dsub_rn(__dsub_rn(fabs(__dsub_rn(vi, wi)), fabs(vi)), fabs(wi));
          }
        }
        unsigned b = __ballot_sync(kFull, hit);
        while (b)
        {
          const int src = __ffs(b) - 1;
          b &= b - 1;
          const double x = __shfl_sync(kFull, t, src);
          score = __dadd_rn(score, x);
        }
      }
      if (lane == 0)
      {
        const float si = __double2float_rn(__ddiv_rn(-score, 2.0));
        unsigned long long key = kNone;
        if (si >= a.min_score)
        {
          key = ((unsigned long long)(~float_key(si)) << 32) | (unsigned)g;
          atomicAdd(&s_kept, 1);
        }
        list[ci] = key;
      }
    }
    __syncthreads();
    const int n_kp = s_kept;
    // (score desc, frame asc): ascending bitonic sort of the keys, padded to a power of two with kNone
    int P2 = 1;
    while (P2 < n_sc) P2 <<= 1;
    if (n_sc > 1)
    {
      for (int i = n_sc + tid; i < P2; i += kQT) list[i] = kNone;
      __syncthreads();
      for (int k = 2; k <= P2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1)
        {
          for (int i = tid; i < P2; i += kQT)
          {
            const int x = i ^ j;
            if (x > i)
            {
              const unsigned long long u = list[i], v = list[x];
              if ((u > v) == ((i & k) == 0))
              {
                list[i] = v;
                list[x] = u;
              }
            }
          }
          __syncthreads();
        }
    }
    const size_t o = (size_t)qi * a.top_k;
    for (int t = tid; t < a.top_k; t += kQT)
    {
      int fr = -1, cm = 0;
      float sc = 0.f;
      if (t < n_kp)
      {
        const unsigned long long key = list[t];
        fr = (int)(key & 0xffffffffu);
        sc = key_float(~(unsigned)(key >> 32));
        cm = counter_of(cnt, fr);
      }
      if (a.cand_frame) a.cand_frame[o + t] = fr;
      if (a.cand_score) a.cand_score[o + t] = sc;
      if (a.cand_common) a.cand_common[o + t] = cm;
    }
    if (tid == 0)
    {
      const bool any = sharing > 0;
      if (a.n_sharing) a.n_sharing[qi] = sharing;
      if (a.max_common) a.max_common[qi] = any ? mx : 0;
      if (a.n_scored) a.n_scored[qi] = any ? n_sc : 0;
      if (a.n_kept) a.n_kept[qi] = any ? n_kp : 0;
    }
    __syncthreads(); // the counters and the list are reused by the next query
  }
}

size_t up16(size_t v) { return (v + 15) & ~(size_t)15; }

} // namespace

int bow_frames(orbx_ctx *c, const orbx_vocab *v, int levelsup, const uint8_t *d_desc, const int *d_n, int F, int stride, const BowArgs &out)
{
  constexpr int kChunk = 1024; // frames per transform launch: bounds the per-feature scratch at 28 B x stride x 1024
  cudaStream_t s = c->stream;
  const size_t ch = (size_t)std::min(F, kChunk) * stride;
  auto sc = [](const void *mine, size_t bytes) { return mine ? 0 : up16(bytes); }; // scratch only for the outputs left null
  const size_t o_word = 0, o_nid = o_word + up16(ch * 4), o_w = o_nid + up16(ch * 4), o_ids = o_w + up16(ch * 8), o_vals = o_ids + sc(out.bow_ids, ch * 4),
               o_nb = o_vals + sc(out.bow_vals, ch * 8), o_fvn = o_nb + sc(out.n_bow, (size_t)kChunk * 4), o_fvs = o_fvn + sc(out.fv_nodes, ch * 4),
               o_fvf = o_fvs + sc(out.fv_start, ch * 4 + (size_t)kChunk * 4), o_nfv = o_fvf + sc(out.fv_feats, ch * 4),
               sc_total = o_nfv + sc(out.n_fv, (size_t)kChunk * 4);
  DeviceBuffer scratch;
  if (int rc = scratch.reserve(c, sc_total)) return rc;
  BowArgs b{};
  b.child_start = v->child_start, b.child_ids = v->child_ids, b.v_desc = v->desc, b.v_weight = v->weight, b.v_word = v->word;
  b.L = v->L, b.levelsup = levelsup, b.image_stride = 1;
  b.f_word = (int *)(scratch.p + o_word), b.f_nid = (int *)(scratch.p + o_nid), b.f_weight = (double *)(scratch.p + o_w);
  for (int f0 = 0; f0 < F; f0 += kChunk)
  {
    const int nf = std::min(kChunk, F - f0);
    const size_t e0 = (size_t)f0 * stride;
    auto at = [&](auto *mine, size_t off, size_t per_frame) { return mine ? mine + (size_t)f0 * per_frame : (decltype(mine))(scratch.p + off); };
    Params p{};
    p.n_features = stride;
    p.desc = const_cast<uint8_t *>(d_desc) + e0 * 32;
    p.n_kps = const_cast<int *>(d_n) + f0;
    BowArgs bb = b;
    bb.bow_ids = at(out.bow_ids, o_ids, stride), bb.bow_vals = at(out.bow_vals, o_vals, stride), bb.n_bow = at(out.n_bow, o_nb, 1);
    bb.fv_nodes = at(out.fv_nodes, o_fvn, stride), bb.fv_start = at(out.fv_start, o_fvs, (size_t)stride + 1), bb.fv_feats = at(out.fv_feats, o_fvf, stride);
    bb.n_fv = at(out.n_fv, o_nfv, 1);
    launch_bow_descend(p, bb, nf, s);
    launch_bow_assemble(p, bb, nf, s);
    c->launches += 2;
  }
  ORBX_CUDA(c, cudaGetLastError());
  // the scratch is freed on return: the work that reads it has to finish first
  ORBX_CUDA(c, cudaStreamSynchronize(s));
  return ORBX_OK;
}

} // namespace orbx

using namespace orbx;

namespace
{

// frees a partly built database on the error paths of orbx_bowdb_build
struct DbGuard
{
  orbx_bowdb *db;
  ~DbGuard()
  {
    if (db) orbx_bowdb_destroy(db);
  }
};

int run_query(orbx_ctx *c, const orbx_bowdb *db, QueryArgs a, const orbx_bowdb_io *io)
{
  const size_t nq = (size_t)a.n_queries, nk = nq * (size_t)a.top_k;
  cudaStream_t s = c->stream;
  uint8_t *st = nullptr;
  const size_t o_f = 0, o_s = o_f + up16(nk * 4), o_c = o_s + up16(nk * 4), o_n = o_c + up16(nk * 4), total = o_n + 4 * up16(nq * 4);
  if (io->on_device)
  {
    a.cand_frame = io->cand_frame, a.cand_score = io->cand_score, a.cand_common = io->cand_common;
    a.n_sharing = io->n_sharing, a.max_common = io->max_common, a.n_scored = io->n_scored, a.n_kept = io->n_kept;
  }
  else
  {
    if (int rc = const_cast<orbx_bowdb *>(db)->staging.reserve(c, total)) return rc;
    st = db->staging.p;
    a.cand_frame = io->cand_frame ? (int *)(st + o_f) : nullptr;
    a.cand_score = io->cand_score ? (float *)(st + o_s) : nullptr;
    a.cand_common = io->cand_common ? (int *)(st + o_c) : nullptr;
    int *cnts = (int *)(st + o_n);
    const size_t q4 = up16(nq * 4) / 4;
    a.n_sharing = io->n_sharing ? cnts : nullptr;
    a.max_common = io->max_common ? cnts + q4 : nullptr;
    a.n_scored = io->n_scored ? cnts + 2 * q4 : nullptr;
    a.n_kept = io->n_kept ? cnts + 3 * q4 : nullptr;
  }
  a.ids = db->ids, a.n = db->n, a.vals = db->vals, a.stride = db->stride, a.word_start = db->word_start, a.post = db->post;
  a.F = db->F, a.P = db->P, a.list_in_smem = db->list_in_smem, a.g_list = db->g_list;
  const int grid = (int)std::min<size_t>(nq, (size_t)db->grid_max);
  bowdb_query_kernel<<<grid, kQT, db->smem, s>>>(a);
  ++c->launches;
  ORBX_CUDA(c, cudaGetLastError());
  if (io->on_device) return ORBX_OK;
  auto back = [&](void *dst, const void *src, size_t bytes) -> cudaError_t {
    return dst ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s) : cudaSuccess;
  };
  ORBX_CUDA(c, back(io->cand_frame, a.cand_frame, nk * 4));
  ORBX_CUDA(c, back(io->cand_score, a.cand_score, nk * 4));
  ORBX_CUDA(c, back(io->cand_common, a.cand_common, nk * 4));
  ORBX_CUDA(c, back(io->n_sharing, a.n_sharing, nq * 4));
  ORBX_CUDA(c, back(io->max_common, a.max_common, nq * 4));
  ORBX_CUDA(c, back(io->n_scored, a.n_scored, nq * 4));
  ORBX_CUDA(c, back(io->n_kept, a.n_kept, nq * 4));
  ORBX_CUDA(c, cudaStreamSynchronize(s));
  return ORBX_OK;
}

int check_io(orbx_ctx *c, const orbx_bowdb *db, const orbx_bowdb_io *io, bool range)
{
  if (!io) return ORBX_ERR_INVALID_ARG;
  if (db->ctx != c || db->device != c->device) return fail(c, ORBX_ERR_INVALID_ARG, "the database belongs to another context");
  if (io->top_k < 1 || io->top_k > db->F) return fail(c, ORBX_ERR_INVALID_ARG, "top_k must be 1..n_frames");
  if (range ? io->exclude_window < 0 : io->exclude_window != -1)
    return fail(c, ORBX_ERR_INVALID_ARG, "exclude_window must be >= 0 for range queries and -1 for the resident-frame query");
  if (std::isnan(io->min_score)) return fail(c, ORBX_ERR_INVALID_ARG, "min_score is NaN");
  return ORBX_OK;
}

} // namespace

extern "C"
{

  void orbx_bowdb_destroy(orbx_bowdb *db)
  {
    if (!db) return;
    cudaSetDevice(db->device);
    cudaFree(db->ids);
    cudaFree(db->vals);
    cudaFree(db->n);
    cudaFree(db->word_start);
    cudaFree(db->post);
    cudaFree(db->g_list);
    delete db;
  }

  int orbx_bowdb_info(const orbx_bowdb *db, int32_t *n_frames, int32_t *n_words, int64_t *n_postings)
  {
    if (!db) return ORBX_ERR_INVALID_ARG;
    if (n_frames) *n_frames = db->F;
    if (n_words) *n_words = db->n_words;
    if (n_postings) *n_postings = db->n_postings;
    return ORBX_OK;
  }

  int orbx_bowdb_build(orbx_ctx *c, const orbx_vocab *v, const uint8_t *desc, const int32_t *n_kps, int32_t F, int32_t stride, int32_t on_device,
                       orbx_bowdb **out)
  {
    if (!c || !v || !desc || !n_kps || !out) return ORBX_ERR_INVALID_ARG;
    *out = nullptr;
    if (v->ctx != c || v->device != c->device) return fail(c, ORBX_ERR_INVALID_ARG, "the vocabulary belongs to another context");
    if (F < 1) return fail(c, ORBX_ERR_INVALID_ARG, "keyframe database: n_frames < 1");
    if (F > ORBX_BOWDB_MAX_FRAMES) return fail(c, ORBX_ERR_CAPACITY, "keyframe database: more than ORBX_BOWDB_MAX_FRAMES frames");
    if (stride < 1) return fail(c, ORBX_ERR_INVALID_ARG, "keyframe database: stride < 1");
    cudaStream_t s = c->stream;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    if (int rc = bow_configure(c, stride, ORBX_ERR_INVALID_ARG)) return rc;
    std::vector<int32_t> h_n((size_t)F);
    if (on_device)
    {
      ORBX_CUDA(c, cudaMemcpyAsync(h_n.data(), n_kps, (size_t)F * 4, cudaMemcpyDeviceToHost, s));
      ORBX_CUDA(c, cudaStreamSynchronize(s));
    }
    else
      std::memcpy(h_n.data(), n_kps, (size_t)F * 4);
    for (int f = 0; f < F; ++f)
      if (h_n[(size_t)f] < 0 || h_n[(size_t)f] > stride) return fail(c, ORBX_ERR_INVALID_ARG, "keyframe database: a count lies outside 0..stride");

    orbx_bowdb *db = new orbx_bowdb();
    DbGuard guard{db};
    db->ctx = c, db->vocab = v, db->device = c->device, db->F = F, db->stride = stride, db->n_words = v->n_words;
    const size_t rows = (size_t)F * stride;
    ORBX_CUDA(c, cudaMalloc((void **)&db->ids, rows * 4));
    ORBX_CUDA(c, cudaMalloc((void **)&db->vals, rows * 8));
    ORBX_CUDA(c, cudaMalloc((void **)&db->n, (size_t)F * 4));
    ORBX_CUDA(c, cudaMalloc((void **)&db->word_start, ((size_t)v->n_words + 1) * 8));
    // inputs in device memory; the transform's per-feature and FeatureVector outputs in chunk scratch
    DeviceBuffer in_desc, in_n, cursor;
    const uint8_t *d_desc = desc;
    const int *d_n = n_kps;
    if (!on_device)
    {
      if (int rc = in_desc.reserve(c, rows * 32)) return rc;
      if (int rc = in_n.reserve(c, (size_t)F * 4)) return rc;
      ORBX_CUDA(c, cudaMemcpyAsync(in_desc.p, desc, rows * 32, cudaMemcpyHostToDevice, s));
      ORBX_CUDA(c, cudaMemcpyAsync(in_n.p, n_kps, (size_t)F * 4, cudaMemcpyHostToDevice, s));
      d_desc = in_desc.p, d_n = (const int *)in_n.p;
    }
    BowArgs bow{};
    bow.bow_ids = db->ids, bow.bow_vals = db->vals, bow.n_bow = db->n;
    if (int rc = bow_frames(c, v, 0, d_desc, d_n, F, stride, bow)) return rc;
    ORBX_CUDA(c, cudaGetLastError());
    // inverted file: postings per word, exclusive scan, fill
    const unsigned blocks = (unsigned)((rows + 255) / 256);
    ORBX_CUDA(c, cudaMemsetAsync(db->word_start, 0, ((size_t)v->n_words + 1) * 8, s));
    bowdb_word_count_kernel<<<blocks, 256, 0, s>>>(db->ids, db->n, stride, (long long)rows, db->word_start);
    bowdb_scan_kernel<<<1, 1024, 0, s>>>(db->word_start, v->n_words);
    c->launches += 2;
    ORBX_CUDA(c, cudaGetLastError());
    ORBX_CUDA(c, cudaMemcpyAsync(&db->n_postings, db->word_start + v->n_words, 8, cudaMemcpyDeviceToHost, s));
    ORBX_CUDA(c, cudaStreamSynchronize(s));
    ORBX_CUDA(c, cudaMalloc((void **)&db->post, (size_t)std::max(db->n_postings, 1LL) * 4));
    if (int rc = cursor.reserve(c, (size_t)v->n_words * 8)) return rc;
    ORBX_CUDA(c, cudaMemsetAsync(cursor.p, 0, (size_t)v->n_words * 8, s));
    bowdb_fill_kernel<<<blocks, 256, 0, s>>>(db->ids, db->n, stride, (long long)rows, db->word_start, (unsigned long long *)cursor.p, db->post);
    ++c->launches;
    ORBX_CUDA(c, cudaGetLastError());
    // query launch shape: the counters always live in shared memory; the candidate list joins them when it fits
    db->P = 1;
    while (db->P < F) db->P <<= 1;
    const size_t cnt_bytes = up16((size_t)(F + 1) / 2 * 4), list_bytes = (size_t)db->P * 8;
    db->list_in_smem = cnt_bytes + list_bytes + 2048 <= kSmemOptIn;
    db->smem = cnt_bytes + (db->list_in_smem ? list_bytes : 0);
    if (db->smem > 48 * 1024)
    {
      static SmemOptIn state;
      if (raise_dynamic_smem(bowdb_query_kernel, state, db->smem)) return fail(c, ORBX_ERR_CUDA, "cannot reserve shared memory for the keyframe database query");
    }
    int per_sm = 0, n_sm = 0;
    ORBX_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bowdb_query_kernel, kQT, db->smem));
    ORBX_CUDA(c, cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, c->device));
    if (per_sm < 1) return fail(c, ORBX_ERR_CUDA, "the keyframe database query kernel does not fit an SM");
    db->grid_max = per_sm * n_sm;
    if (!db->list_in_smem) ORBX_CUDA(c, cudaMalloc((void **)&db->g_list, (size_t)db->grid_max * list_bytes));
    // the scratch buffers are freed on return: the work that reads them has to finish first
    ORBX_CUDA(c, cudaStreamSynchronize(s));
    guard.db = nullptr;
    *out = db;
    return ORBX_OK;
  }

  int orbx_bowdb_query_range(orbx_ctx *c, const orbx_bowdb *db, int64_t q_lo, int64_t q_hi, const orbx_bowdb_io *io)
  {
    if (!c || !db) return ORBX_ERR_INVALID_ARG;
    if (int rc = check_io(c, db, io, true)) return rc;
    if (q_lo < 0 || q_hi < q_lo || q_hi > db->F) return fail(c, ORBX_ERR_INVALID_ARG, "query range outside [0, n_frames)");
    if (q_lo == q_hi) return ORBX_OK;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    QueryArgs a{};
    a.q_ids = db->ids + (size_t)q_lo * db->stride, a.q_vals = db->vals + (size_t)q_lo * db->stride, a.q_n = db->n + q_lo;
    a.q_stride = db->stride, a.q_frame0 = q_lo, a.window = io->exclude_window;
    a.n_queries = (int)(q_hi - q_lo), a.top_k = io->top_k, a.min_score = io->min_score;
    return run_query(c, db, a, io);
  }

  int orbx_bowdb_query_frame(orbx_ctx *c, const orbx_bowdb *db, int frame, const orbx_bowdb_io *io)
  {
    if (!c || !db || frame < 0) return ORBX_ERR_INVALID_ARG;
    if (int rc = check_io(c, db, io, false)) return rc;
    if (int rc = require_bow(c, frame + 1LL)) return rc;
    if (c->bow_vocab != db->vocab) return fail(c, ORBX_ERR_STATE, "the resident bag of words was computed with another vocabulary than the database's");
    ORBX_CUDA(c, cudaSetDevice(c->device));
    const BowArgs b = bow_at(c->bow, (size_t)frame, (size_t)c->cfg.n_features);
    QueryArgs a{};
    a.q_ids = b.bow_ids, a.q_vals = b.bow_vals, a.q_n = b.n_bow, a.q_stride = c->cfg.n_features, a.q_frame0 = 0, a.window = -1;
    a.n_queries = 1, a.top_k = io->top_k, a.min_score = io->min_score;
    return run_query(c, db, a, io);
  }

} // extern "C"
