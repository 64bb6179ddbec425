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
// and the host code the bag-of-words entry points share: the tree arguments, the transform launch, the builders' training-set
// intake and bow_frames, the chunked transform of the keyframe database and the loop verifier.
#include <algorithm>
#include <cstring>

#include "orbx_internal.h"

namespace orbx
{

namespace
{

constexpr int kBowWarps = 8;
constexpr int kAsmThreads = 256;

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
        const unsigned d = (unsigned)hamming256(f0, f1, g0, g1);
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

// segments of equal (key >> 16) in the sorted prefix [0, nv): returns the number of segments; seg_of(j) via the scan
template <typename HeadFn> __device__ int for_each_head(const unsigned long long *key, int nv, int P, int *s_warp, HeadFn fn)
{
  const int per = P / kAsmThreads > 0 ? P / kAsmThreads : 1;
  const int j0 = threadIdx.x * per, j1 = min(j0 + per, nv);
  int mine = 0;
  for (int j = j0; j < j1; ++j) mine += (j == 0) || ((key[j] >> 16) != (key[j - 1] >> 16));
  int total;
  int seg = block_exclusive_scan<kAsmThreads>(mine, total, s_warp);
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
    bitonic_sort<kAsmThreads>(s_key, P);
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
  bitonic_sort<kAsmThreads>(s_key, P);
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

int bow_configure(orbx_ctx *c, int n_features, int too_large)
{
  if (n_features > ORBX_BOW_MAX_STRIDE) return fail(c, too_large, "the bag-of-words sort holds at most ORBX_BOW_MAX_STRIDE (16384) features per frame");
  const size_t bytes = (size_t)bow_sort_size(n_features) * sizeof(unsigned long long);
  if (bytes <= 48 * 1024) return ORBX_OK;
  static SmemOptIn state, state_words;
  if (raise_dynamic_smem(bow_assemble_kernel, state, bytes) || raise_dynamic_smem(bow_word_frames_kernel, state_words, bytes))
    return fail(c, ORBX_ERR_CUDA, "cannot reserve shared memory for the bag-of-words sort");
  return ORBX_OK;
}

BowArgs bow_args(const orbx_vocab *v, int levelsup, int image_stride, BowArgs b)
{
  b.child_start = v->child_start, b.child_ids = v->child_ids, b.v_desc = v->desc, b.v_weight = v->weight, b.v_word = v->word;
  b.L = v->L, b.levelsup = levelsup, b.image_stride = image_stride;
  return b;
}

void launch_bow_transform(orbx_ctx *c, const Params &p, const BowArgs &a, int n_frames, cudaStream_t s)
{
  launch_bow_descend(p, a, n_frames, s);
  launch_bow_assemble(p, a, n_frames, s);
  c->launches += 2;
}

int read_training_set(orbx_ctx *c, const uint8_t *desc, const int32_t *n_kps, int F, int stride, bool on_device, const char *what, TrainingSet &ts)
{
  cudaStream_t s = c->stream;
  ts.n.resize((size_t)F);
  if (on_device)
  {
    ORBX_CUDA(c, cudaMemcpyAsync(ts.n.data(), n_kps, (size_t)F * 4, cudaMemcpyDeviceToHost, s));
    ORBX_CUDA(c, cudaStreamSynchronize(s));
  }
  else
    std::memcpy(ts.n.data(), n_kps, (size_t)F * 4);
  for (int32_t x : ts.n)
    if (x < 0 || x > stride) return fail(c, ORBX_ERR_INVALID_ARG, std::string(what) + ": a count lies outside 0..stride");
  ts.desc = desc, ts.d_n = n_kps;
  if (on_device) return ORBX_OK;
  // the kernels read no byte past rows * 32 of the descriptors and F * 4 of the counts
  const size_t desc_bytes = up16((size_t)F * stride * 32);
  if (int rc = ts.staged.reserve(c, desc_bytes + (size_t)F * 4)) return rc;
  ORBX_CUDA(c, cudaMemcpyAsync(ts.staged.p, desc, (size_t)F * stride * 32, cudaMemcpyHostToDevice, s));
  ORBX_CUDA(c, cudaMemcpyAsync(ts.staged.p + desc_bytes, n_kps, (size_t)F * 4, cudaMemcpyHostToDevice, s));
  ts.desc = ts.staged.p, ts.d_n = (const int32_t *)(ts.staged.p + desc_bytes);
  return ORBX_OK;
}

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
  BowArgs b = bow_args(v, levelsup, 1);
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
    launch_bow_transform(c, p, bb, nf, s);
  }
  ORBX_CUDA(c, cudaGetLastError());
  // the scratch is freed on return: the work that reads it has to finish first
  ORBX_CUDA(c, cudaStreamSynchronize(s));
  return ORBX_OK;
}

} // namespace orbx
