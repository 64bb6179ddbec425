// orbx_vocab.cu -- bag-of-words vocabulary construction on the device (orbx_vocab_build), sm_100a.
//
// Restates DBoW2 / DBoW3 TemplatedVocabulary::create (hierarchical k-means, HKmeansStep) under the rules of include/orbx.h;
// tests/vocab_build_oracle.c (oracle_vocab_build) is the sequential restatement the kernels are tested against bit for bit.
// The tree is built level by level: every node of a level that runs k-means moves through seeding, assignment and mean in
// lockstep, as one set of segmented problems.  A segment (the descriptors of one node, contiguous) is cut into tiles of at
// most kTile descriptors and every kernel that touches descriptors runs one CTA per tile, so a level-1 node of millions
// of descriptors spreads over the whole GPU while a node of a hundred descriptors is one CTA; the per-node steps
// (k-means++ pick, mean) run one CTA per node.
//   vocab_gather_kernel      training rows [frame][stride] -> the root's contiguous segment
//   vocab_kpp_dist_kernel    k-means++ round: min_dist update against the newest centre, one sum per tile
//   vocab_kpp_pick_kernel    k-means++ round: S over the node's tiles, cut = 1 + r_j % S, first descriptor whose running sum
//                            reaches it (two block scans: tiles, then descriptors of one tile)
//   vocab_assign_kernel      nearest centre per descriptor (first among equals), changed flag, and the 256 bit counters
//                            of every (node, cluster) (32x32 bit transposes through ballots, shared then global integer atomics)
//   vocab_update_kernel      per node: converged / capped, or the majority mean as the next centres
//   vocab_tile_count_kernel / vocab_scatter_kernel   order-preserving partition of the members into the child segments
//   vocab_trivial_copy_kernel  descriptors of the nodes with n <= k (one child each) for the host's node table
// The IDF counts reuse bow_descend_kernel and bow_word_frames_kernel (orbx_bow.cu).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "orbx_internal.h"

namespace orbx
{

namespace
{

constexpr int kVT = 256;     // threads per CTA
constexpr int kTile = 4096;  // descriptors per tile
constexpr unsigned kFull = 0xffffffffu;

struct VbArgs
{
  const uint4 *D; // [n][2] descriptors of the level, segment by segment
  uint4 *Dn;      // next level
  uint16_t *md;   // k-means++ min_dist
  uint8_t *asg;   // cluster of every descriptor
  int k;
  // tiles of the k-means segments
  const int *tile_seg, *tile_start, *tile_len;
  unsigned long long *tile_sum;
  int *tile_cnt;       // [T][k]
  const int *tile_dst; // [T][k] first destination in Dn of the tile's members of cluster c, -1 = not split again
  // k-means segments
  const int *seg_start, *seg_n, *seg_tile0, *seg_ntiles;
  const unsigned long long *seg_key;
  uint4 *cent;        // [S][k][2]
  int *kk;            // [S] centres
  unsigned *cnt;      // [S][k][256] bit counters
  unsigned *members;  // [S][k]
  int *changed, *active, *iters, *capped; // [S]
  int *n_active;
};

__device__ __forceinline__ int hamming(uint4 a0, uint4 a1, uint4 b0, uint4 b1)
{
  return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) + __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) +
         __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

// exclusive block scan of one 64-bit value per thread; *total = the block's sum
__device__ unsigned long long block_exscan(unsigned long long v, unsigned long long *total, unsigned long long *s_warp)
{
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned long long inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1)
  {
    const unsigned long long t = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_warp[wid] = inc;
  __syncthreads();
  unsigned long long base = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < kVT / 32; ++w)
  {
    const unsigned long long t = s_warp[w];
    if (w < wid) base += t;
    tot += t;
  }
  __syncthreads();
  *total = tot;
  return base + inc - v;
}

__global__ void __launch_bounds__(kVT) vocab_gather_kernel(const uint4 *src, const int *n_kps, const long long *row_off, int stride, long long n_rows_x_stride,
                                                            uint4 *D)
{
  const long long e = (long long)blockIdx.x * kVT + threadIdx.x;
  if (e >= n_rows_x_stride) return;
  const long long f = e / stride;
  const int i = (int)(e - f * stride);
  if (i >= n_kps[f]) return;
  const long long o = row_off[f] + i;
  D[2 * o] = __ldg(src + 2 * e);
  D[2 * o + 1] = __ldg(src + 2 * e + 1);
}

// round r >= 1: min_dist against centre r - 1 (round 1 sets it); tile_sum = the tile's part of S
__global__ void __launch_bounds__(kVT) vocab_kpp_dist_kernel(const VbArgs a, int round)
{
  __shared__ unsigned long long s_warp[kVT / 32];
  const int t = blockIdx.x, seg = a.tile_seg[t];
  if (a.kk[seg] != round) // seeding of this node stopped (S == 0)
  {
    if (threadIdx.x == 0) a.tile_sum[t] = 0;
    return;
  }
  const uint4 c0 = a.cent[2 * ((size_t)seg * a.k + round - 1)], c1 = a.cent[2 * ((size_t)seg * a.k + round - 1) + 1];
  const int base = a.tile_start[t], len = a.tile_len[t];
  unsigned long long sum = 0;
  for (int e = threadIdx.x; e < len; e += kVT)
  {
    const size_t g = (size_t)base + e;
    int d = hamming(a.D[2 * g], a.D[2 * g + 1], c0, c1);
    if (round > 1) d = min(d, (int)a.md[g]);
    a.md[g] = (uint16_t)d;
    sum += (unsigned long long)d;
  }
  unsigned long long total;
  block_exscan(sum, &total, s_warp);
  if (threadIdx.x == 0) a.tile_sum[t] = total;
}

// round 0: centre 0 = descriptor r_0 % n.  round r >= 1: S = sum over the node's tiles; S == 0 stops the seeding, else
// centre r = the first descriptor whose running min_dist sum reaches cut = 1 + r_r % S
__global__ void __launch_bounds__(kVT) vocab_kpp_pick_kernel(const VbArgs a, int round)
{
  __shared__ unsigned long long s_warp[kVT / 32];
  __shared__ int s_tile, s_pick;
  __shared__ unsigned long long s_rem;
  const int seg = blockIdx.x, tid = threadIdx.x;
  const unsigned long long K = a.seg_key[seg];
  if (round == 0)
  {
    if (tid == 0)
    {
      const size_t g = (size_t)a.seg_start[seg] + (size_t)(splitmix64(K) % (unsigned long long)a.seg_n[seg]);
      a.cent[2 * (size_t)seg * a.k] = a.D[2 * g];
      a.cent[2 * (size_t)seg * a.k + 1] = a.D[2 * g + 1];
      a.kk[seg] = 1;
    }
    return;
  }
  if (a.kk[seg] != round) return;
  const int t0 = a.seg_tile0[seg], nt = a.seg_ntiles[seg];
  const int per = (nt + kVT - 1) / kVT, j0 = min(tid * per, nt), j1 = min(j0 + per, nt);
  unsigned long long mine = 0;
  for (int j = j0; j < j1; ++j) mine += a.tile_sum[t0 + j];
  unsigned long long S;
  const unsigned long long ex = block_exscan(mine, &S, s_warp);
  if (S == 0) return; // every descriptor equals a centre: fewer than k clusters
  const unsigned long long cut = 1 + splitmix64(K ^ ((unsigned long long)round * kGolden)) % S;
  if (ex < cut && cut <= ex + mine)
  {
    unsigned long long run = ex;
    for (int j = j0; j < j1; ++j)
    {
      const unsigned long long ts = a.tile_sum[t0 + j];
      if (run + ts >= cut)
      {
        s_tile = t0 + j;
        s_rem = cut - run;
        break;
      }
      run += ts;
    }
  }
  __syncthreads();
  const int t = s_tile;
  const unsigned long long rem = s_rem;
  const int base = a.tile_start[t], len = a.tile_len[t];
  const int per2 = (len + kVT - 1) / kVT, e0 = min(tid * per2, len), e1 = min(e0 + per2, len);
  unsigned long long mine2 = 0;
  for (int e = e0; e < e1; ++e) mine2 += a.md[(size_t)base + e];
  unsigned long long tot2;
  const unsigned long long ex2 = block_exscan(mine2, &tot2, s_warp);
  if (ex2 < rem && rem <= ex2 + mine2)
  {
    unsigned long long run = ex2;
    for (int e = e0; e < e1; ++e)
    {
      run += a.md[(size_t)base + e];
      if (run >= rem)
      {
        s_pick = e;
        break;
      }
    }
  }
  __syncthreads();
  if (tid == 0)
  {
    const size_t g = (size_t)base + s_pick;
    a.cent[2 * ((size_t)seg * a.k + round)] = a.D[2 * g];
    a.cent[2 * ((size_t)seg * a.k + round) + 1] = a.D[2 * g + 1];
    a.kk[seg] = round + 1;
  }
}

// pass p: nearest centre of every descriptor of the tile; members and the 256 bit counters per cluster
__global__ void __launch_bounds__(kVT) vocab_assign_kernel(const VbArgs a, int pass)
{
  __shared__ uint4 s_c[ORBX_VOCAB_MAX_K][2];
  __shared__ unsigned s_cnt[ORBX_VOCAB_MAX_K * 256];
  __shared__ unsigned s_mem[ORBX_VOCAB_MAX_K];
  __shared__ int s_changed;
  const int t = blockIdx.x, seg = a.tile_seg[t], tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (!a.active[seg]) return;
  const int nk = a.kk[seg];
  for (int i = tid; i < nk * 2; i += kVT) s_c[i >> 1][i & 1] = a.cent[2 * (size_t)seg * a.k + i];
  for (int i = tid; i < nk * 256; i += kVT) s_cnt[i] = 0;
  if (tid < nk) s_mem[tid] = 0;
  if (tid == 0) s_changed = 0;
  __syncthreads();
  const int base = a.tile_start[t], len = a.tile_len[t];
  bool changed = false;
  for (int chunk = wid * 32; chunk < len; chunk += kVT) // warp-uniform trip count
  {
    const int e = chunk + lane;
    const bool valid = e < len;
    uint4 x0 = make_uint4(0, 0, 0, 0), x1 = x0;
    int bc = -1;
    if (valid)
    {
      const size_t g = (size_t)base + e;
      x0 = a.D[2 * g], x1 = a.D[2 * g + 1];
      int best = hamming(x0, x1, s_c[0][0], s_c[0][1]);
      bc = 0;
      for (int c = 1; c < nk; ++c)
      {
        const int d = hamming(x0, x1, s_c[c][0], s_c[c][1]);
        if (d < best) best = d, bc = c;
      }
      if (pass > 1 && a.asg[g] != bc) changed = true;
      a.asg[g] = (uint8_t)bc;
    }
    // lane b of the transpose of word q holds the lanes whose descriptor has bit 32q + b
    const unsigned xw[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
    unsigned col[8];
#pragma unroll
    for (int q = 0; q < 8; ++q)
    {
      unsigned mine = 0;
#pragma unroll
      for (int b = 0; b < 32; ++b)
      {
        const unsigned m = __ballot_sync(kFull, (xw[q] >> b) & 1u);
        if (lane == b) mine = m;
      }
      col[q] = mine;
    }
    for (int c = 0; c < nk; ++c)
    {
      const unsigned in_c = __ballot_sync(kFull, bc == c);
      if (!in_c) continue;
      if (lane == 0) atomicAdd(&s_mem[c], (unsigned)__popc(in_c));
#pragma unroll
      for (int q = 0; q < 8; ++q)
      {
        const unsigned n = __popc(col[q] & in_c);
        if (n) atomicAdd(&s_cnt[c * 256 + q * 32 + lane], n);
      }
    }
  }
  if (changed) s_changed = 1;
  __syncthreads();
  unsigned *g_cnt = a.cnt + (size_t)seg * a.k * 256;
  for (int i = tid; i < nk * 256; i += kVT)
    if (s_cnt[i]) atomicAdd(&g_cnt[i], s_cnt[i]);
  if (tid < nk && s_mem[tid]) atomicAdd(&a.members[(size_t)seg * a.k + tid], s_mem[tid]);
  if (tid == 0 && s_changed) a.changed[seg] = 1;
}

// after pass p: a node whose assignments did not change has converged, one at ORBX_VOCAB_MAX_ITERS is capped; both keep
// the centres and the member counts of this pass.  Otherwise: majority means, counters cleared for the next pass.
__global__ void __launch_bounds__(kVT) vocab_update_kernel(const VbArgs a, int pass)
{
  const int seg = blockIdx.x, tid = threadIdx.x;
  if (!a.active[seg]) return;
  const bool changed = pass == 1 || a.changed[seg];
  if (!changed || pass >= ORBX_VOCAB_MAX_ITERS)
  {
    if (tid == 0) a.active[seg] = 0, a.iters[seg] = pass, a.capped[seg] = changed ? 1 : 0;
    return;
  }
  const int nk = a.kk[seg];
  unsigned *g_cnt = a.cnt + (size_t)seg * a.k * 256;
  unsigned *cw = reinterpret_cast<unsigned *>(a.cent + 2 * (size_t)seg * a.k);
  for (int c = 0; c < nk; ++c)
  {
    const unsigned m = a.members[(size_t)seg * a.k + c];
    if (m == 0) continue; // an empty cluster keeps its centre
    const unsigned w = __ballot_sync(kFull, g_cnt[c * 256 + tid] >= (m + 1) / 2);
    if ((tid & 31) == 0) cw[c * 8 + (tid >> 5)] = w;
  }
  __syncthreads();
  for (int c = 0; c < nk; ++c) g_cnt[c * 256 + tid] = 0;
  if (tid < nk) a.members[(size_t)seg * a.k + tid] = 0;
  if (tid == 0)
  {
    a.changed[seg] = 0;
    atomicAdd(a.n_active, 1);
  }
}

__global__ void __launch_bounds__(kVT) vocab_tile_count_kernel(const VbArgs a)
{
  __shared__ int s_n[ORBX_VOCAB_MAX_K];
  const int t = blockIdx.x;
  if (threadIdx.x < a.k) s_n[threadIdx.x] = 0;
  __syncthreads();
  const int base = a.tile_start[t], len = a.tile_len[t];
  for (int e = threadIdx.x; e < len; e += kVT) atomicAdd(&s_n[a.asg[(size_t)base + e]], 1);
  __syncthreads();
  if (threadIdx.x < a.k) a.tile_cnt[(size_t)t * a.k + threadIdx.x] = s_n[threadIdx.x];
}

// members of cluster c keep their order: destination = tile_dst[t][c] + members of c before them in the tile
__global__ void __launch_bounds__(kVT) vocab_scatter_kernel(const VbArgs a)
{
  __shared__ int s_wc[kVT / 32][ORBX_VOCAB_MAX_K];
  const int t = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nk = a.kk[a.tile_seg[t]];
  const int base = a.tile_start[t], len = a.tile_len[t];
  const int per = ((len + kVT / 32 - 1) / (kVT / 32) + 31) & ~31; // each warp: a contiguous, 32-aligned part of the tile
  const int w0 = min(wid * per, len), w1 = min(w0 + per, len);
  int cnt_c = 0; // lane c: members of cluster c in this warp's part
  for (int ch = w0; ch < w1; ch += 32)
  {
    const int e = ch + lane;
    const int bc = e < w1 ? (int)a.asg[(size_t)base + e] : -1;
    for (int c = 0; c < nk; ++c)
    {
      const unsigned m = __ballot_sync(kFull, bc == c);
      if (lane == c) cnt_c += __popc(m);
    }
  }
  if (lane < nk) s_wc[wid][lane] = cnt_c;
  __syncthreads();
  int run = 0; // lane c: members of c before the current chunk
  if (lane < nk)
    for (int w = 0; w < wid; ++w) run += s_wc[w][lane];
  const int *dst = a.tile_dst + (size_t)t * a.k;
  for (int ch = w0; ch < w1; ch += 32)
  {
    const int e = ch + lane;
    const bool valid = e < w1;
    const int bc = valid ? (int)a.asg[(size_t)base + e] : -1;
    unsigned mine = 0;
    int add = 0;
    for (int c = 0; c < nk; ++c)
    {
      const unsigned m = __ballot_sync(kFull, bc == c);
      if (bc == c) mine = m;
      if (lane == c) add = __popc(m);
    }
    const int before = __shfl_sync(kFull, run, valid ? bc : 0);
    if (valid && dst[bc] >= 0)
    {
      const size_t o = (size_t)dst[bc] + before + __popc(mine & ((1u << lane) - 1u));
      const size_t g = (size_t)base + e;
      a.Dn[2 * o] = a.D[2 * g];
      a.Dn[2 * o + 1] = a.D[2 * g + 1];
    }
    run += add;
  }
}

// one warp per node with n <= k: its descriptors (one child each) to out[out_off[s] ..]
__global__ void __launch_bounds__(kVT) vocab_trivial_copy_kernel(const uint4 *D, const int *start, const int *n, const int *out_off, int n_segs, uint4 *out)
{
  const int s = blockIdx.x * (kVT / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (s >= n_segs || lane >= n[s]) return;
  const size_t g = (size_t)start[s] + lane, o = (size_t)out_off[s] + lane;
  out[2 * o] = D[2 * g];
  out[2 * o + 1] = D[2 * g + 1];
}

// device scratch of one build, freed on every return path
struct Scratch
{
  std::vector<void *> p;
  int dev = 0;
  ~Scratch()
  {
    cudaSetDevice(dev);
    for (void *q : p) cudaFree(q);
  }
  template <class T> cudaError_t get(T **out, size_t n)
  {
    *out = nullptr;
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, n * sizeof(T) + 16);
    if (e == cudaSuccess) p.push_back(q), *out = (T *)q;
    return e;
  }
};

struct Events
{
  cudaEvent_t a = nullptr, b = nullptr;
  ~Events()
  {
    if (a) cudaEventDestroy(a);
    if (b) cudaEventDestroy(b);
  }
};

struct HostNode
{
  int parent, first_child = -1, n_child = 0;
  uint8_t desc[32];
};

struct Seg
{
  int node, start, n;
  unsigned long long key;
};

} // namespace

} // namespace orbx

using namespace orbx;

extern "C" int orbx_vocab_build(orbx_ctx *c, const orbx_vocab_train *in, orbx_vocab **out)
{
  if (!c || !in || !out) return ORBX_ERR_INVALID_ARG;
  *out = nullptr;
  const int k = in->k, L = in->L, F = in->n_frames, stride = in->stride;
  if (!in->desc || !in->n_kps || F < 1 || stride < 1) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary training set: desc / n_kps missing, n_frames < 1 or stride < 1");
  if (k < 2 || k > ORBX_VOCAB_MAX_K || L < 1) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary build: k must be 2..ORBX_VOCAB_MAX_K and L >= 1");
  {
    // a full tree of k^1 + .. + k^L nodes (+ the root) must fit int32 node ids
    double nodes = 1.0, lev = 1.0;
    for (int l = 0; l < L && nodes <= 2147483647.0; ++l) lev *= k, nodes += lev;
    if (nodes > 2147483647.0) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary build: k^L overflows int32 node ids");
  }
  cudaStream_t s = c->stream;
  ORBX_CUDA(c, cudaSetDevice(c->device));
  if (int rc = bow_configure(c, stride, ORBX_ERR_INVALID_ARG)) return rc; // the TF_IDF step sorts a frame row in shared memory
  Scratch sc;
  sc.dev = c->device;
  // counts on the host: row offsets of the gather, validation
  std::vector<int32_t> h_n((size_t)F);
  if (in->on_device)
  {
    ORBX_CUDA(c, cudaMemcpyAsync(h_n.data(), in->n_kps, (size_t)F * 4, cudaMemcpyDeviceToHost, s));
    ORBX_CUDA(c, cudaStreamSynchronize(s));
  }
  else
    std::memcpy(h_n.data(), in->n_kps, (size_t)F * 4);
  std::vector<long long> row_off((size_t)F);
  long long N = 0;
  for (int f = 0; f < F; ++f)
  {
    if (h_n[(size_t)f] < 0 || h_n[(size_t)f] > stride) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary training set: a count lies outside 0..stride");
    row_off[(size_t)f] = N;
    N += h_n[(size_t)f];
  }
  if (N == 0) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary training set holds no descriptor");
  if (N > 2147483647LL) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary training set: more than INT32_MAX descriptors");
  const size_t rows = (size_t)F * stride;
  const uint8_t *d_train = in->desc;
  const int32_t *d_n = in->n_kps;
  if (!in->on_device)
  {
    uint8_t *td;
    int32_t *tn;
    ORBX_CUDA(c, sc.get(&td, rows * 32));
    ORBX_CUDA(c, sc.get(&tn, (size_t)F));
    ORBX_CUDA(c, cudaMemcpyAsync(td, in->desc, rows * 32, cudaMemcpyHostToDevice, s));
    ORBX_CUDA(c, cudaMemcpyAsync(tn, in->n_kps, (size_t)F * 4, cudaMemcpyHostToDevice, s));
    d_train = td, d_n = tn;
  }
  uint4 *D, *Dn;
  uint16_t *md;
  uint8_t *asg;
  long long *d_row_off;
  ORBX_CUDA(c, sc.get(&D, (size_t)N * 2));
  ORBX_CUDA(c, sc.get(&Dn, (size_t)N * 2));
  ORBX_CUDA(c, sc.get(&md, (size_t)N));
  ORBX_CUDA(c, sc.get(&asg, (size_t)N));
  ORBX_CUDA(c, sc.get(&d_row_off, (size_t)F));
  ORBX_CUDA(c, cudaMemcpyAsync(d_row_off, row_off.data(), (size_t)F * 8, cudaMemcpyHostToDevice, s));
  vocab_gather_kernel<<<(unsigned)((rows + kVT - 1) / kVT), kVT, 0, s>>>(reinterpret_cast<const uint4 *>(d_train), d_n, d_row_off, stride, (long long)rows, D);
  ++c->launches;
  ORBX_CUDA(c, cudaGetLastError());

  // per-level device state, grown on demand
  int cap_S = 0, cap_T = 0;
  VbArgs a{};
  a.k = k, a.md = md, a.asg = asg;
  int *d_n_active;
  ORBX_CUDA(c, sc.get(&d_n_active, 1));
  a.n_active = d_n_active;
  Scratch lvl; // buffers that grow are replaced inside `lvl` (freed with the build)
  lvl.dev = c->device;

  std::vector<HostNode> nodes(1);
  nodes[0].parent = -1;
  std::vector<Seg> segs{{0, 0, (int)N, splitmix64(in->seed)}};
  std::vector<int32_t> level_iters((size_t)L, 0);
  std::vector<float> level_ms((size_t)L + 1, 0.f);
  int n_capped = 0;
  Events ev;
  ORBX_CUDA(c, cudaEventCreate(&ev.a));
  ORBX_CUDA(c, cudaEventCreate(&ev.b));
  for (int level = 1; level <= L && !segs.empty(); ++level)
  {
    ORBX_CUDA(c, cudaEventRecord(ev.a, s));
    std::vector<int> km, tr; // indices into segs: k-means nodes, nodes with n <= k
    for (int i = 0; i < (int)segs.size(); ++i) (segs[(size_t)i].n > k ? km : tr).push_back(i);
    const int S = (int)km.size();
    std::vector<int> h_seg_start(S), h_seg_n(S), h_tile0(S), h_ntiles(S), h_tseg, h_tstart, h_tlen;
    std::vector<unsigned long long> h_key(S);
    for (int j = 0; j < S; ++j)
    {
      const Seg &g = segs[(size_t)km[(size_t)j]];
      h_seg_start[j] = g.start, h_seg_n[j] = g.n, h_key[j] = g.key, h_tile0[j] = (int)h_tseg.size();
      for (int o = 0; o < g.n; o += kTile) h_tseg.push_back(j), h_tstart.push_back(g.start + o), h_tlen.push_back(std::min(kTile, g.n - o));
      h_ntiles[j] = (int)h_tseg.size() - h_tile0[j];
    }
    const int T = (int)h_tseg.size();
    std::vector<int> h_kk(S), h_members((size_t)S * k), h_iters(S), h_capped(S), h_tcnt((size_t)T * k);
    std::vector<uint8_t> h_cent((size_t)S * k * 32);
    if (S > 0)
    {
      if (S > cap_S || T > cap_T)
      {
        cap_S = std::max(S, cap_S), cap_T = std::max(T, cap_T);
        int *i32;
        ORBX_CUDA(c, lvl.get(&i32, (size_t)cap_S * (5 + 6 + 2 * (size_t)k) + (size_t)cap_T * (3 + 2 * (size_t)k)));
        a.seg_start = i32, a.seg_n = i32 + cap_S, a.seg_tile0 = i32 + 2 * (size_t)cap_S, a.seg_ntiles = i32 + 3 * (size_t)cap_S;
        a.kk = i32 + 4 * (size_t)cap_S, a.changed = i32 + 5 * (size_t)cap_S, a.active = i32 + 6 * (size_t)cap_S, a.iters = i32 + 7 * (size_t)cap_S;
        a.capped = i32 + 8 * (size_t)cap_S;
        a.members = reinterpret_cast<unsigned *>(i32 + 11 * (size_t)cap_S);
        int *ti = i32 + (11 + (size_t)k) * cap_S + (size_t)k * cap_S;
        a.tile_seg = ti, a.tile_start = ti + cap_T, a.tile_len = ti + 2 * (size_t)cap_T;
        a.tile_cnt = ti + 3 * (size_t)cap_T, a.tile_dst = ti + (3 + (size_t)k) * cap_T;
        unsigned long long *u64;
        ORBX_CUDA(c, lvl.get(&u64, (size_t)cap_S + cap_T));
        a.seg_key = u64, a.tile_sum = u64 + cap_S;
        ORBX_CUDA(c, lvl.get(&a.cent, (size_t)cap_S * k * 2));
        ORBX_CUDA(c, lvl.get(&a.cnt, (size_t)cap_S * k * 256));
      }
      a.D = D, a.Dn = Dn;
      ORBX_CUDA(c, cudaMemcpyAsync((void *)a.seg_start, h_seg_start.data(), (size_t)S * 4, cudaMemcpyHostToDevice, s));
      ORBX_CUDA(c, cudaMemcpyAsync((void *)a.seg_n, h_seg_n.data(), (size_t)S * 4, cudaMemcpyHostToDevice, s));
      ORBX_CUDA(c, cudaMemcpyAsync((void *)a.seg_tile0, h_tile0.data(), (size_t)S * 4, cudaMemcpyHostToDevice, s));
      ORBX_CUDA(c, cudaMemcpyAsync((void *)a.seg_ntiles, h_ntiles.data(), (size_t)S * 4, cudaMemcpyHostToDevice, s));
      ORBX_CUDA(c, cudaMemcpyAsync((void *)a.seg_key, h_key.data(), (size_t)S * 8, cudaMemcpyHostToDevice, s));
      ORBX_CUDA(c, cudaMemcpyAsync((void *)a.tile_seg, h_tseg.data(), (size_t)T * 4, cudaMemcpyHostToDevice, s));
      ORBX_CUDA(c, cudaMemcpyAsync((void *)a.tile_start, h_tstart.data(), (size_t)T * 4, cudaMemcpyHostToDevice, s));
      ORBX_CUDA(c, cudaMemcpyAsync((void *)a.tile_len, h_tlen.data(), (size_t)T * 4, cudaMemcpyHostToDevice, s));
      std::vector<int> ones((size_t)S, 1);
      ORBX_CUDA(c, cudaMemcpyAsync(a.active, ones.data(), (size_t)S * 4, cudaMemcpyHostToDevice, s));
      ORBX_CUDA(c, cudaMemsetAsync(a.changed, 0, (size_t)S * 4, s));
      ORBX_CUDA(c, cudaMemsetAsync(a.capped, 0, (size_t)S * 4, s));
      ORBX_CUDA(c, cudaMemsetAsync(a.kk, 0, (size_t)S * 4, s));
      ORBX_CUDA(c, cudaMemsetAsync(a.members, 0, (size_t)S * k * 4, s));
      ORBX_CUDA(c, cudaMemsetAsync(a.cnt, 0, (size_t)S * k * 256 * 4, s));
      // k-means++ seeding: pick 0, then (min_dist update, pick) per further centre
      vocab_kpp_pick_kernel<<<S, kVT, 0, s>>>(a, 0);
      for (int r = 1; r < k; ++r)
      {
        vocab_kpp_dist_kernel<<<T, kVT, 0, s>>>(a, r);
        vocab_kpp_pick_kernel<<<S, kVT, 0, s>>>(a, r);
      }
      c->launches += 2 * k - 1;
      ORBX_CUDA(c, cudaGetLastError());
      // Lloyd passes until every node of the level has converged or is capped
      int h_active = 0;
      for (int pass = 1; pass <= ORBX_VOCAB_MAX_ITERS; ++pass)
      {
        ORBX_CUDA(c, cudaMemsetAsync(d_n_active, 0, 4, s));
        vocab_assign_kernel<<<T, kVT, 0, s>>>(a, pass);
        vocab_update_kernel<<<S, kVT, 0, s>>>(a, pass);
        c->launches += 2;
        ORBX_CUDA(c, cudaGetLastError());
        ORBX_CUDA(c, cudaMemcpyAsync(&h_active, d_n_active, 4, cudaMemcpyDeviceToHost, s));
        ORBX_CUDA(c, cudaStreamSynchronize(s));
        if (h_active == 0) break;
      }
      vocab_tile_count_kernel<<<T, kVT, 0, s>>>(a);
      ++c->launches;
      ORBX_CUDA(c, cudaGetLastError());
      ORBX_CUDA(c, cudaMemcpyAsync(h_kk.data(), a.kk, (size_t)S * 4, cudaMemcpyDeviceToHost, s));
      ORBX_CUDA(c, cudaMemcpyAsync(h_members.data(), a.members, (size_t)S * k * 4, cudaMemcpyDeviceToHost, s));
      ORBX_CUDA(c, cudaMemcpyAsync(h_iters.data(), a.iters, (size_t)S * 4, cudaMemcpyDeviceToHost, s));
      ORBX_CUDA(c, cudaMemcpyAsync(h_capped.data(), a.capped, (size_t)S * 4, cudaMemcpyDeviceToHost, s));
      ORBX_CUDA(c, cudaMemcpyAsync(h_cent.data(), a.cent, (size_t)S * k * 32, cudaMemcpyDeviceToHost, s));
      ORBX_CUDA(c, cudaMemcpyAsync(h_tcnt.data(), a.tile_cnt, (size_t)T * k * 4, cudaMemcpyDeviceToHost, s));
    }
    // descriptors of the nodes with n <= k
    std::vector<int> t_start(tr.size()), t_n(tr.size()), t_off(tr.size());
    int t_total = 0;
    for (size_t j = 0; j < tr.size(); ++j)
    {
      const Seg &g = segs[(size_t)tr[j]];
      t_start[j] = g.start, t_n[j] = g.n, t_off[j] = t_total;
      t_total += g.n;
    }
    std::vector<uint8_t> h_triv((size_t)t_total * 32);
    if (!tr.empty())
    {
      int *ti;
      uint4 *tout;
      ORBX_CUDA(c, lvl.get(&ti, tr.size() * 3));
      ORBX_CUDA(c, lvl.get(&tout, (size_t)t_total * 2));
      ORBX_CUDA(c, cudaMemcpyAsync(ti, t_start.data(), tr.size() * 4, cudaMemcpyHostToDevice, s));
      ORBX_CUDA(c, cudaMemcpyAsync(ti + tr.size(), t_n.data(), tr.size() * 4, cudaMemcpyHostToDevice, s));
      ORBX_CUDA(c, cudaMemcpyAsync(ti + 2 * tr.size(), t_off.data(), tr.size() * 4, cudaMemcpyHostToDevice, s));
      vocab_trivial_copy_kernel<<<(unsigned)((tr.size() + kVT / 32 - 1) / (kVT / 32)), kVT, 0, s>>>(D, ti, ti + tr.size(), ti + 2 * tr.size(), (int)tr.size(), tout);
      ++c->launches;
      ORBX_CUDA(c, cudaGetLastError());
      ORBX_CUDA(c, cudaMemcpyAsync(h_triv.data(), tout, (size_t)t_total * 32, cudaMemcpyDeviceToHost, s));
    }
    ORBX_CUDA(c, cudaEventRecord(ev.b, s));
    ORBX_CUDA(c, cudaStreamSynchronize(s));
    ORBX_CUDA(c, cudaEventElapsedTime(&level_ms[(size_t)level - 1], ev.a, ev.b));
    // children in cluster order; the next level's segments in (node, cluster) order
    std::vector<Seg> next;
    std::vector<int> dst_base((size_t)S * k, -1);
    int run = 0;
    for (size_t j = 0; j < tr.size(); ++j)
    {
      const Seg &g = segs[(size_t)tr[j]];
      nodes[(size_t)g.node].first_child = (int)nodes.size(), nodes[(size_t)g.node].n_child = g.n;
      for (int i = 0; i < g.n; ++i)
      {
        HostNode h;
        h.parent = g.node;
        std::memcpy(h.desc, h_triv.data() + ((size_t)t_off[j] + i) * 32, 32);
        nodes.push_back(h);
      }
    }
    for (int j = 0; j < S; ++j)
    {
      const Seg &g = segs[(size_t)km[(size_t)j]];
      level_iters[(size_t)level - 1] = std::max(level_iters[(size_t)level - 1], h_iters[j]);
      n_capped += h_capped[j];
      const int first = (int)nodes.size();
      nodes[(size_t)g.node].first_child = first, nodes[(size_t)g.node].n_child = h_kk[j];
      for (int cl = 0; cl < h_kk[j]; ++cl)
      {
        HostNode h;
        h.parent = g.node;
        std::memcpy(h.desc, h_cent.data() + ((size_t)j * k + cl) * 32, 32);
        nodes.push_back(h);
        const int m = h_members[(size_t)j * k + cl];
        if (level < L && m > 1)
        {
          next.push_back({first + cl, run, m, splitmix64(g.key + (unsigned long long)cl + 1)});
          dst_base[(size_t)j * k + cl] = run;
          run += m;
        }
      }
    }
    if (nodes.size() > (size_t)2147483647) return fail(c, ORBX_ERR_CAPACITY, "vocabulary build: more than INT32_MAX nodes");
    if (!next.empty())
    {
      // order-preserving scatter into the child segments
      std::vector<int> h_tdst((size_t)T * k, -1);
      std::vector<int> acc((size_t)k);
      for (int j = 0; j < S; ++j)
      {
        for (int cl = 0; cl < k; ++cl) acc[(size_t)cl] = dst_base[(size_t)j * k + cl];
        for (int t = h_tile0[j]; t < h_tile0[j] + h_ntiles[j]; ++t)
          for (int cl = 0; cl < h_kk[j]; ++cl)
            if (acc[(size_t)cl] >= 0)
            {
              h_tdst[(size_t)t * k + cl] = acc[(size_t)cl];
              acc[(size_t)cl] += h_tcnt[(size_t)t * k + cl];
            }
      }
      ORBX_CUDA(c, cudaMemcpyAsync((void *)a.tile_dst, h_tdst.data(), (size_t)T * k * 4, cudaMemcpyHostToDevice, s));
      vocab_scatter_kernel<<<T, kVT, 0, s>>>(a);
      ++c->launches;
      ORBX_CUDA(c, cudaGetLastError());
      std::swap(D, Dn);
    }
    segs.swap(next);
  }

  // DBoW's ids: children consecutive, nodes split depth first (pre-order)
  const size_t nn = nodes.size();
  if (nn < 2) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary build produced no node");
  std::vector<int> id(nn, 0);
  {
    int next_id = 1;
    std::vector<int> stack{0};
    while (!stack.empty())
    {
      const int v = stack.back();
      stack.pop_back();
      const HostNode &h = nodes[(size_t)v];
      for (int ch = 0; ch < h.n_child; ++ch) id[(size_t)h.first_child + ch] = next_id++;
      for (int ch = h.n_child - 1; ch >= 0; --ch) stack.push_back(h.first_child + ch); // first child is visited first
    }
  }
  const int n_rec = (int)nn - 1;
  std::vector<int32_t> parent((size_t)n_rec);
  std::vector<uint8_t> leaf((size_t)n_rec), rdesc((size_t)n_rec * 32);
  std::vector<double> weight((size_t)n_rec, 0.0);
  for (size_t v = 1; v < nn; ++v)
  {
    const size_t r = (size_t)id[v] - 1;
    parent[r] = id[(size_t)nodes[v].parent];
    leaf[r] = nodes[v].n_child == 0;
    std::memcpy(rdesc.data() + r * 32, nodes[v].desc, 32);
  }
  orbx_vocab *v = nullptr;
  int rc = orbx_vocab_create(c, k, L, n_rec, parent.data(), leaf.data(), rdesc.data(), weight.data(), &v);
  if (rc) return rc;
  // TF_IDF: descend every training descriptor (the transform's descent), count each word once per frame
  auto fail_v = [&](int code, const std::string &msg) {
    orbx_vocab_destroy(v);
    return fail(c, code, msg);
  };
  int *f_word, *f_nid, *ni;
  double *f_weight;
  cudaError_t e = sc.get(&f_word, rows);
  if (e == cudaSuccess) e = sc.get(&f_nid, rows);
  if (e == cudaSuccess) e = sc.get(&f_weight, rows);
  if (e == cudaSuccess) e = sc.get(&ni, (size_t)v->n_words);
  if (e == cudaSuccess) e = cudaMemsetAsync(ni, 0, (size_t)v->n_words * 4, s);
  if (e != cudaSuccess) return fail_v(ORBX_ERR_CUDA, std::string("vocabulary IDF buffers: ") + cudaGetErrorString(e));
  BowArgs b{};
  b.child_start = v->child_start, b.child_ids = v->child_ids, b.v_desc = v->desc, b.v_weight = v->weight, b.v_word = v->word;
  b.L = L, b.levelsup = 0, b.image_stride = 1;
  e = cudaEventRecord(ev.a, s);
  for (int f0 = 0; f0 < F && e == cudaSuccess; f0 += 65535) // grid.y of the descent carries the frame
  {
    const int nf = std::min(65535, F - f0);
    Params p{};
    p.n_features = stride;
    p.desc = const_cast<uint8_t *>(d_train) + (size_t)f0 * stride * 32;
    p.n_kps = const_cast<int *>(d_n) + f0;
    BowArgs bb = b;
    bb.f_word = f_word + (size_t)f0 * stride, bb.f_nid = f_nid + (size_t)f0 * stride, bb.f_weight = f_weight + (size_t)f0 * stride;
    launch_bow_descend(p, bb, nf, s);
    launch_bow_word_frames(p, bb, nf, ni, s);
    c->launches += 2;
  }
  std::vector<int> h_ni((size_t)v->n_words);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaEventRecord(ev.b, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(h_ni.data(), ni, (size_t)v->n_words * 4, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e == cudaSuccess) e = cudaEventElapsedTime(&level_ms[(size_t)L], ev.a, ev.b);
  if (e != cudaSuccess) return fail_v(ORBX_ERR_CUDA, std::string("vocabulary IDF: ") + cudaGetErrorString(e));
  // setNodeWeights: log(N / N_i) in double on the host, from the integer counts
  std::vector<double> node_w((size_t)v->n_nodes, 0.0);
  for (int r = 0, w = 0; r < n_rec; ++r)
    if (leaf[(size_t)r])
    {
      const int n_i = h_ni[(size_t)w++];
      weight[(size_t)r] = n_i > 0 ? std::log((double)F / (double)n_i) : 0.0;
      node_w[(size_t)r + 1] = weight[(size_t)r];
    }
  v->rec_weight = weight;
  e = cudaMemcpyAsync(v->weight, node_w.data(), node_w.size() * sizeof(double), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return fail_v(ORBX_ERR_CUDA, std::string("vocabulary weights: ") + cudaGetErrorString(e));
  if (in->iters) std::memcpy(in->iters, level_iters.data(), (size_t)L * 4);
  if (in->n_capped) *in->n_capped = n_capped;
  if (in->level_ms) std::memcpy(in->level_ms, level_ms.data(), ((size_t)L + 1) * sizeof(float));
  *out = v;
  return ORBX_OK;
}
