// orbx_bow.cu -- bag-of-words transform (SURVEY.md section 8(f) rank 3), sm_100a.
//
// Replaces VirtualFrame::computeBow (include/ORB_SLAM2/Frame.h:224-231) = DBoW3::Vocabulary::transform(descriptors,
// BowVector&, FeatureVector&, levelsup = 4).  DBoW3 is an un-vendored dependency of the reference: the kernels follow its
// published algorithm (see oracle/orb_oracle.c for the restatement they are tested against; parity unpinned).
//   bow_descend_kernel   one warp per descriptor: at every tree level the child with the smallest Hamming distance, the
//                        first among equals (lanes <-> children, packed (distance, position) minimum through REDUX)
//   bow_assemble_kernel  one CTA per frame: BowVector (std::map<WordId, double>: ids ascending, weights accumulated in
//                        feature order, then L1-normalised with the sum taken in id order) and FeatureVector
//                        (std::map<NodeId, vector<unsigned>>) from two stable sorts of (key << 16 | feature index)
//   bow_word_frames_kernel  one CTA per frame: the frame's distinct words (the same sort), one integer atomic per word;
//                        N_i of TF_IDF for orbx_vocab_build (setNodeWeights)
#include "orbx_device.cuh"

namespace orbx
{

namespace
{

constexpr int kBowWarps = 8;
constexpr int kAsmThreads = 256;
constexpr unsigned kFullMask = 0xffffffffu;

__global__ void __launch_bounds__(kBowWarps * 32) bow_descend_kernel(const Params p, const BowArgs a)
{
  const int frame = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * kBowWarps + (threadIdx.x >> 5);
  const int img = frame * a.image_stride;
  if (i >= p.n_kps[img]) return;
  const uint4 *d4 = reinterpret_cast<const uint4 *>(p.desc + ((size_t)img * p.n_features + i) * 32);
  const uint4 f0 = __ldg(d4), f1 = __ldg(d4 + 1);
  const uint4 *vdesc = reinterpret_cast<const uint4 *>(a.v_desc);
  const int nid_level = a.L - a.levelsup;
  int node = 0, at = 0, level = 0;
  for (;;)
  {
    ++level;
    const int c0 = a.child_start[node], c1 = a.child_start[node + 1];
    if (c0 == c1) break; // only a degenerate root gets here
    unsigned best = 0xffffffffu;
    for (int cb = c0; cb < c1; cb += 32)
    {
      const int c = cb + lane;
      if (c < c1)
      {
        const int id = a.child_ids[c];
        const uint4 g0 = __ldg(vdesc + 2 * (size_t)id), g1 = __ldg(vdesc + 2 * (size_t)id + 1);
        const unsigned d = __popc(f0.x ^ g0.x) + __popc(f0.y ^ g0.y) + __popc(f0.z ^ g0.z) + __popc(f0.w ^ g0.w) + __popc(f1.x ^ g1.x) +
                           __popc(f1.y ^ g1.y) + __popc(f1.z ^ g1.z) + __popc(f1.w ^ g1.w);
        best = min(best, (d << 20) | (unsigned)(c - c0)); // strict < over children in id order == lexicographic minimum
      }
    }
    best = __reduce_min_sync(kFullMask, best);
    node = a.child_ids[c0 + (int)(best & 0xfffffu)];
    if (level == nid_level) at = node;
    if (a.child_start[node] == a.child_start[node + 1]) break; // leaf
  }
  if (lane == 0)
  {
    const size_t o = (size_t)frame * p.n_features + i;
    a.f_word[o] = a.v_word[node];
    a.f_weight[o] = a.v_weight[node];
    a.f_nid[o] = nid_level <= 0 ? 0 : at;
  }
}

__device__ __forceinline__ int asm_block_scan(int v, int &total, int *s_warp)
{
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1)
  {
    const int t = __shfl_up_sync(kFullMask, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_warp[wid] = inc;
  __syncthreads();
  int base = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < kAsmThreads / 32; ++w)
  {
    const int t = s_warp[w];
    if (w < wid) base += t;
    tot += t;
  }
  __syncthreads();
  total = tot;
  return base + inc - v;
}

// ascending bitonic sort of P (power of two) 64-bit keys in shared memory
__device__ void bitonic_sort(unsigned long long *key, int P)
{
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1)
    {
      for (int i = threadIdx.x; i < P; i += kAsmThreads)
      {
        const int x = i ^ j;
        if (x > i)
        {
          const unsigned long long u = key[i], v = key[x];
          const bool asc = (i & k) == 0;
          if ((u > v) == asc)
          {
            key[i] = v;
            key[x] = u;
          }
        }
      }
      __syncthreads();
    }
}

// segments of equal (key >> 16) in the sorted prefix [0, nv): returns the number of segments; seg_of(j) via the scan
template <typename HeadFn> __device__ int for_each_head(const unsigned long long *key, int nv, int P, int *s_warp, HeadFn fn)
{
  const int per = P / kAsmThreads > 0 ? P / kAsmThreads : 1;
  const int j0 = threadIdx.x * per, j1 = min(j0 + per, nv);
  int mine = 0;
  for (int j = j0; j < j1; ++j) mine += (j == 0) || ((key[j] >> 16) != (key[j - 1] >> 16));
  int total;
  int seg = asm_block_scan(mine, total, s_warp);
  for (int j = j0; j < j1; ++j)
    if ((j == 0) || ((key[j] >> 16) != (key[j - 1] >> 16))) fn(seg++, j);
  return total;
}

__global__ void __launch_bounds__(kAsmThreads) bow_assemble_kernel(const Params p, const BowArgs a, int P)
{
  extern __shared__ unsigned long long s_key[]; // [P]
  __shared__ int s_warp[kAsmThreads / 32];
  __shared__ int s_nv;
  __shared__ double s_norm;
  const int frame = blockIdx.x, tid = threadIdx.x;
  const int n = min(p.n_kps[frame * a.image_stride], P);
  const size_t fo = (size_t)frame * p.n_features;
  const int *f_word = a.f_word + fo, *f_nid = a.f_nid + fo;
  const double *f_weight = a.f_weight + fo;
  int *bow_ids = a.bow_ids + fo, *fv_nodes = a.fv_nodes + fo, *fv_feats = a.fv_feats + fo;
  int *fv_start = a.fv_start + (size_t)frame * (p.n_features + 1);
  double *bow_vals = a.bow_vals + fo;
  constexpr unsigned long long kPad = ~0ull;

  for (int pass = 0; pass < 2; ++pass)
  {
    // pass 0: keys (word << 16 | feature) -> BowVector; pass 1: keys (node << 16 | feature) -> FeatureVector.
    // Features with weight 0 are stopped words (`if (w > 0)` in Vocabulary::transform) and take part in neither.
    if (tid == 0) s_nv = 0;
    __syncthreads();
    int cnt = 0;
    for (int i = tid; i < P; i += kAsmThreads)
    {
      unsigned long long k = kPad;
      if (i < n && f_weight[i] > 0.0)
      {
        k = ((unsigned long long)(unsigned)(pass == 0 ? f_word[i] : f_nid[i]) << 16) | (unsigned long long)i;
        ++cnt;
      }
      s_key[i] = k;
    }
    atomicAdd(&s_nv, cnt);
    __syncthreads();
    const int nv = s_nv;
    bitonic_sort(s_key, P);
    if (pass == 0)
    {
      // BowVector::addWeight in feature order: the first feature of a word inserts its weight, the others add to it
      const int m = for_each_head(s_key, nv, P, s_warp, [&](int seg, int j) {
        const unsigned long long w = s_key[j] >> 16;
        double sum = f_weight[s_key[j] & 0xffffull];
        for (int t = j + 1; t < nv && (s_key[t] >> 16) == w; ++t) sum = __dadd_rn(sum, f_weight[s_key[t] & 0xffffull]);
        bow_ids[seg] = (int)w;
        bow_vals[seg] = sum;
      });
      __syncthreads();
      // BowVector::normalize(L1): the norm is accumulated over the map in id order (a serial chain, by one thread)
      if (tid == 0)
      {
        double norm = 0.0;
        for (int k = 0; k < m; ++k) norm = __dadd_rn(norm, fabs(bow_vals[k]));
        s_norm = norm;
        a.n_bow[frame] = m;
      }
      __syncthreads();
      const double norm = s_norm;
      if (norm > 0.0)
        for (int k = tid; k < m; k += kAsmThreads) bow_vals[k] = __ddiv_rn(bow_vals[k], norm);
    }
    else
    {
      const int m = for_each_head(s_key, nv, P, s_warp, [&](int seg, int j) {
        fv_nodes[seg] = (int)(s_key[j] >> 16);
        fv_start[seg] = j;
      });
      for (int j = tid; j < nv; j += kAsmThreads) fv_feats[j] = (int)(s_key[j] & 0xffffull);
      if (tid == 0)
      {
        fv_start[m] = nv;
        a.n_fv[frame] = m;
      }
    }
    __syncthreads();
  }
}

// N_i of setNodeWeights: n_frames_of_word[w] += 1 for every distinct word w among the frame's descents (f_word)
__global__ void __launch_bounds__(kAsmThreads) bow_word_frames_kernel(const Params p, const BowArgs a, int P, int *n_frames_of_word)
{
  extern __shared__ unsigned long long s_key[]; // [P]
  __shared__ int s_warp[kAsmThreads / 32];
  const int frame = blockIdx.x;
  const int n = min(p.n_kps[frame * a.image_stride], P);
  const int *f_word = a.f_word + (size_t)frame * p.n_features;
  for (int i = threadIdx.x; i < P; i += kAsmThreads)
    s_key[i] = i < n ? ((unsigned long long)(unsigned)f_word[i] << 16) | (unsigned long long)i : ~0ull;
  __syncthreads();
  bitonic_sort(s_key, P);
  for_each_head(s_key, n, P, s_warp, [&](int, int j) { atomicAdd(&n_frames_of_word[s_key[j] >> 16], 1); });
}

} // namespace

void launch_bow_descend(const Params &p, const BowArgs &a, int n_frames, cudaStream_t s)
{
  dim3 grid((p.n_features + kBowWarps - 1) / kBowWarps, n_frames);
  bow_descend_kernel<<<grid, kBowWarps * 32, 0, s>>>(p, a);
}

int bow_sort_size(int n_features)
{
  int P = 256;
  while (P < n_features) P <<= 1;
  return P;
}

void launch_bow_assemble(const Params &p, const BowArgs &a, int n_frames, cudaStream_t s)
{
  const int P = bow_sort_size(p.n_features);
  bow_assemble_kernel<<<n_frames, kAsmThreads, (size_t)P * sizeof(unsigned long long), s>>>(p, a, P);
}

void launch_bow_word_frames(const Params &p, const BowArgs &a, int n_frames, int *n_frames_of_word, cudaStream_t s)
{
  const int P = bow_sort_size(p.n_features);
  bow_word_frames_kernel<<<n_frames, kAsmThreads, (size_t)P * sizeof(unsigned long long), s>>>(p, a, P, n_frames_of_word);
}

int bow_configure(int n_features)
{
  const size_t bytes = (size_t)bow_sort_size(n_features) * sizeof(unsigned long long);
  if (bytes <= 48 * 1024) return 0;
  static SmemOptIn state, state_words;
  if (raise_dynamic_smem(bow_assemble_kernel, state, bytes)) return -1;
  return raise_dynamic_smem(bow_word_frames_kernel, state_words, bytes);
}

} // namespace orbx
