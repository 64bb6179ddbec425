// orbx_serialize.cu -- result serialisation (SURVEY.md section 8(f) rank 4), sm_100a.
//
// serialize_kernel writes, for every frame of the last call, the orbslam2.KeyFrameData record (proto3 wire format,
// proto/Keyframe.proto:45-64) that KeyFrame::serializeToProtobuf (src/KeyFrame.cc:553-647) produces for a keyframe made
// from a fresh frame, straight from the device-resident results: one CTA per frame, so that only the finished records
// cross PCIe.  Layout of a record (fields in number order, as every protobuf serializer emits them):
//   1 id | 2-5 max_u max_v min_u min_v | 6 keypoints[] | 7 right_u (packed) | 8 depths (packed) | 9 descriptors[] |
//   10 bow_vector | 11 feature_vector | 12 pose | 16 map_points (packed, -1 each)
// proto3 scalars whose bit pattern is zero are not written.  Keypoint entries have variable size (block scan for their
// offsets, byte stores); everything behind them is fixed-stride and written as aligned words assembled byte by byte.
// Fields 10 / 11 are present and empty unless the launch carries the frames' BoW results (SerArgs::bow_ids ...), as
// KeyFrame::serializeToProtobuf fills them from mBowVec / mFeatVec (src/KeyFrame.cc:585-599): then they are byte-stored
// entries at offsets from closed forms (sorted ids -> varint sizes by binary search) and a block scan over the nodes.
#include "orbx_device.cuh"

namespace orbx
{

namespace
{

constexpr int kSerThreads = 256;

__device__ __forceinline__ int put_varint(uint8_t *o, unsigned long long v)
{
  int n = 0;
  while (v >= 0x80ull)
  {
    o[n++] = (uint8_t)(v | 0x80ull);
    v >>= 7;
  }
  o[n++] = (uint8_t)v;
  return n;
}

__device__ __forceinline__ int put_f32(uint8_t *o, float f)
{
  const uint32_t u = __float_as_uint(f);
  o[0] = (uint8_t)u, o[1] = (uint8_t)(u >> 8), o[2] = (uint8_t)(u >> 16), o[3] = (uint8_t)(u >> 24);
  return 4;
}

// size and bytes of one KeyPoint entry: tag 0x32, length, then x (1), y (2), octave (3), angle (4) when non-zero
__device__ __forceinline__ int keypoint_entry(const orbx_keypoint &k, uint8_t *m /* >= 28 bytes */)
{
  int l = 2;
  if (__float_as_uint(k.x)) m[l++] = 0x0D, l += put_f32(m + l, k.x);
  if (__float_as_uint(k.y)) m[l++] = 0x15, l += put_f32(m + l, k.y);
  if (k.octave) m[l++] = 0x18, l += put_varint(m + l, (unsigned long long)(long long)k.octave);
  if (__float_as_uint(k.angle)) m[l++] = 0x25, l += put_f32(m + l, k.angle);
  m[0] = 0x32;
  m[1] = (uint8_t)(l - 2); // <= 26
  return l;
}

__device__ __forceinline__ int varint_len(unsigned long long v)
{
  int n = 1;
  while (v >= 0x80ull) v >>= 7, ++n;
  return n;
}

// FeatureVector.FeatureNode j: 0A len [08 node_id, left out when 0] 12 plen <packed varint feature ids>.  Feature ids
// ascend inside a node and are < 2^16, so plen = count + (count >= 128) + (count >= 16384) from two binary searches.
struct FvNode
{
  int s, e, lb1, lb2; // features [s, e); the first >= 128 / >= 16384
  int node, plen, inner, len;
};
__device__ __forceinline__ FvNode fv_node(const int *fv_nodes, const int *fv_start, const int *fv_feats, int j)
{
  FvNode d;
  d.s = fv_start[j], d.e = fv_start[j + 1];
  d.lb1 = lower_bound(fv_feats, d.s, d.e, 1 << 7);
  d.lb2 = lower_bound(fv_feats, d.lb1, d.e, 1 << 14);
  d.node = fv_nodes[j];
  d.plen = (d.e - d.s) + (d.e - d.lb1) + (d.e - d.lb2);
  d.inner = (d.node ? 1 + varint_len((unsigned)d.node) : 0) + 1 + varint_len((unsigned)d.plen) + d.plen;
  d.len = 1 + varint_len((unsigned)d.inner) + d.inner;
  return d;
}

__global__ void __launch_bounds__(kSerThreads) serialize_kernel(const Params p, const SerArgs a)
{
  __shared__ uint8_t s_head[40], s_tail[64], s_pk[3][12]; // s_pk: the length-delimited headers of fields 7, 8, 16
  __shared__ int s_warp[kSerThreads / 32];
  __shared__ int s_len[4]; // head, tail, and the header lengths of the packed fields
  __shared__ int s_lb[4];  // BowVector: first entry whose word id needs 2, 3, 4, 5 varint bytes
  __shared__ int s_fv[5][kSerThreads]; // FeatureVector chunk: s, e, lb1, lb2 and payload offset of each node
  const int frame = blockIdx.x, tid = threadIdx.x;
  const int img = frame * a.image_stride;
  const int n = p.n_kps[img];
  const orbx_keypoint *kps = p.kps_und + (size_t)img * p.n_features;
  const uint8_t *desc = p.desc + (size_t)img * p.n_features * 32;
  const double *ur = p.u_right + (size_t)frame * p.n_features, *dp = p.depth + (size_t)frame * p.n_features;
  uint8_t *out = a.out + (size_t)frame * a.stride;

  if (tid == 0)
  {
    int h = 0;
    const unsigned long long id = a.id0 + (unsigned long long)frame;
    if (id) s_head[h++] = 0x08, h += put_varint(s_head + h, id);
    const float b[4] = {a.max_u, a.max_v, a.min_u, a.min_v};
    for (int k = 0; k < 4; ++k)
      if (__float_as_uint(b[k])) s_head[h++] = (uint8_t)(((2 + k) << 3) | 5), h += put_f32(s_head + h, b[k]);
    s_len[0] = h;
    int t = 0;
    s_tail[t++] = 0x52, s_tail[t++] = 0; // bow_vector = 10, feature_vector = 11: present and empty
    s_tail[t++] = 0x5A, s_tail[t++] = 0;
    s_tail[t++] = 0x62, s_tail[t++] = 52; // pose = 12 { rotation = 1 [9 floats, packed], translation = 2 [3 floats] }
    s_tail[t++] = 0x0A, s_tail[t++] = 36;
    for (int k = 0; k < 9; ++k) t += put_f32(s_tail + t, a.pose ? a.pose[(size_t)frame * 12 + k] : ((k & 3) == 0 ? 1.f : 0.f));
    s_tail[t++] = 0x12, s_tail[t++] = 12;
    for (int k = 9; k < 12; ++k) t += put_f32(s_tail + t, a.pose ? a.pose[(size_t)frame * 12 + k] : 0.f);
    s_len[1] = t;
    int q = 0;
    s_pk[0][q++] = 0x3A, q += put_varint(s_pk[0] + q, 4ull * (unsigned long long)n);
    s_pk[1][0] = 0x42;
    for (int k = 1; k < q; ++k) s_pk[1][k] = s_pk[0][k];
    s_len[2] = q;
    int r = 0;
    r += put_varint(s_pk[2] + r, (16u << 3) | 2u);
    r += put_varint(s_pk[2] + r, 10ull * (unsigned long long)n);
    s_len[3] = r;
  }
  __syncthreads();
  const int H = s_len[0], T = s_len[1], PH = s_len[2], MH = s_len[3];
  for (int i = tid; i < H; i += kSerThreads) out[i] = s_head[i];

  // field 6: variable-size entries; offsets by a block scan per chunk of kSerThreads keypoints
  int base = H;
  for (int i0 = 0; i0 < n; i0 += kSerThreads)
  {
    const int i = i0 + tid;
    uint8_t m[28];
    int len = 0;
    if (i < n) len = keypoint_entry(kps[i], m);
    int total;
    const int off = block_exclusive_scan<kSerThreads>(len, total, s_warp);
    uint8_t *o = out + base + off;
    for (int k = 0; k < len; ++k) o[k] = m[k];
    base += total;
  }

  // fields 10 and 11 with content: sizes first (their headers precede them), from closed forms and one block reduction
  const bool bow = a.bow_ids != nullptr;
  const size_t fo = (size_t)frame * p.n_features;
  const int *bow_ids = bow ? a.bow_ids + fo : nullptr, *fv_nodes = bow ? a.fv_nodes + fo : nullptr, *fv_feats = bow ? a.fv_feats + fo : nullptr;
  const int *fv_start = bow ? a.fv_start + (size_t)frame * (p.n_features + 1) : nullptr;
  int n_bow = 0, n_fv = 0;
  long long sz_bow = 0, sz_fv = 0;
  if (bow)
  {
    n_bow = a.n_bow[frame], n_fv = a.n_fv[frame];
    // entry k = 0A len 08 <varint id> 11 <double>: 12 + varint_len(id) bytes; ids ascend, so the bytes before entry k are
    // 13 k + sum over t of max(0, k - s_lb[t])
    if (tid < 4) s_lb[tid] = lower_bound(bow_ids, 0, n_bow, 1 << (7 * (tid + 1)));
    int mine = 0;
    for (int j = tid; j < n_fv; j += kSerThreads) mine += fv_node(fv_nodes, fv_start, fv_feats, j).len;
    int fv_total;
    block_exclusive_scan<kSerThreads>(mine, fv_total, s_warp); // its barriers also publish s_lb
    sz_bow = 13ll * n_bow;
    for (int t = 0; t < 4; ++t) sz_bow += n_bow - s_lb[t];
    sz_fv = fv_total;
  }

  // everything behind the keypoints except the BoW sections is a function of the byte position
  const long long off_ru = base;
  const long long sec_pk = n ? (long long)PH + 4ll * n : 0;            // fields 7 and 8 (absent when empty)
  const long long off_dp = off_ru + sec_pk, off_desc = off_dp + sec_pk;
  const long long off_bow = off_desc + 36ll * n;
  const long long off_bow_e = off_bow + 1 + varint_len((unsigned long long)sz_bow), off_fv = off_bow_e + sz_bow;
  const long long off_fv_e = off_fv + 1 + varint_len((unsigned long long)sz_fv);
  // without BoW inputs s_tail starts with the empty fields 10 / 11; with them it starts at the pose
  const int tail_skip = bow ? 4 : 0;
  const long long off_tail = bow ? off_fv_e + sz_fv : off_bow, off_mp = off_tail + T - tail_skip;
  const long long total = off_mp + ((a.with_map_points && n) ? (long long)MH + 10ll * n : 0);
  auto byte_at = [&](long long pos) -> uint32_t {
    if (pos < off_desc)
    {
      const bool second = pos >= off_dp;
      const long long q = pos - (second ? off_dp : off_ru);
      if (q < PH) return s_pk[second ? 1 : 0][q];
      const long long e = (q - PH) >> 2;
      const float v = (float)(second ? dp[e] : ur[e]); // the writer narrows the doubles to float (src/KeyFrame.cc:575-576)
      return (__float_as_uint(v) >> (8 * (int)((q - PH) & 3))) & 0xffu;
    }
    if (pos < off_tail)
    {
      const long long q = pos - off_desc, e = q / 36;
      const int r = (int)(q - 36 * e);
      if (r < 4) return (0x200A224Au >> (8 * r)) & 0xffu; // 0x4A, 34, 0x0A, 32
      return desc[e * 32 + (r - 4)];
    }
    if (pos < off_mp) return s_tail[tail_skip + (pos - off_tail)];
    const long long q = pos - off_mp;
    if (q < MH) return s_pk[2][q];
    return ((q - MH) % 10 == 9) ? 0x01u : 0xffu; // int64 -1 as a 10-byte varint
  };
  // aligned output words of [lo, hi) (out and stride are 4-byte aligned); bytes of the edge words outside the range belong
  // to the byte-stored sections
  auto write_words = [&](long long lo, long long hi) {
    const long long w0 = lo >> 2, w1 = (hi + 3) >> 2;
    for (long long w = w0 + tid; w < w1; w += kSerThreads)
    {
      const long long pos = w << 2;
      if (pos >= lo && pos + 4 <= hi)
      {
        const uint32_t v = byte_at(pos) | (byte_at(pos + 1) << 8) | (byte_at(pos + 2) << 16) | (byte_at(pos + 3) << 24);
        *reinterpret_cast<uint32_t *>(out + pos) = v;
      }
      else
      {
        for (int k = 0; k < 4; ++k)
          if (pos + k >= lo && pos + k < hi) out[pos + k] = (uint8_t)byte_at(pos + k);
      }
    }
  };
  if (!bow)
  {
    write_words(off_ru, total);
    if (tid == 0) a.sizes[frame] = total;
    return;
  }
  write_words(off_ru, off_bow);
  write_words(off_tail, total);

  // field 10 BowVector { map<uint32, double> words = 1 }: entries in ascending word id (std::map order), key and value
  // always written
  if (tid == 0)
  {
    out[off_bow] = 0x52, put_varint(out + off_bow + 1, (unsigned long long)sz_bow);
    out[off_fv] = 0x5A, put_varint(out + off_fv + 1, (unsigned long long)sz_fv);
  }
  const double *bow_vals = a.bow_vals + fo;
  for (int k = tid; k < n_bow; k += kSerThreads)
  {
    long long pos = off_bow_e + 13ll * k;
    for (int t = 0; t < 4; ++t) pos += max(0, k - s_lb[t]);
    uint8_t *o = out + pos;
    const unsigned id = (unsigned)bow_ids[k];
    o[0] = 0x0A, o[1] = (uint8_t)(10 + varint_len(id)), o[2] = 0x08;
    int l = 3 + put_varint(o + 3, id);
    o[l++] = 0x11;
    const unsigned long long v = (unsigned long long)__double_as_longlong(bow_vals[k]);
    for (int b = 0; b < 8; ++b) o[l + b] = (uint8_t)(v >> (8 * b));
  }

  // field 11 FeatureVector { repeated FeatureNode nodes = 1 }: nodes in ascending id; node headers by one thread per node
  // at block-scan offsets, then the packed feature ids by one warp per node at closed-form offsets
  const int lane = tid & 31, wid = tid >> 5;
  long long fbase = off_fv_e;
  for (int j0 = 0; j0 < n_fv; j0 += kSerThreads)
  {
    const int j = j0 + tid, cnt = min(kSerThreads, n_fv - j0);
    FvNode d{};
    if (j < n_fv) d = fv_node(fv_nodes, fv_start, fv_feats, j);
    int chunk_total;
    const int off = block_exclusive_scan<kSerThreads>(j < n_fv ? d.len : 0, chunk_total, s_warp);
    if (j < n_fv)
    {
      uint8_t *o = out + fbase + off;
      int q = 0;
      o[q++] = 0x0A, q += put_varint(o + q, (unsigned)d.inner);
      if (d.node) o[q++] = 0x08, q += put_varint(o + q, (unsigned)d.node);
      o[q++] = 0x12, q += put_varint(o + q, (unsigned)d.plen);
      s_fv[0][tid] = d.s, s_fv[1][tid] = d.e, s_fv[2][tid] = d.lb1, s_fv[3][tid] = d.lb2, s_fv[4][tid] = (int)(fbase + off + q);
    }
    __syncthreads();
    for (int q = wid; q < cnt; q += kSerThreads / 32)
    {
      const int s = s_fv[0][q], e = s_fv[1][q], lb1 = s_fv[2][q], lb2 = s_fv[3][q], pay = s_fv[4][q];
      for (int t = s + lane; t < e; t += 32)
        put_varint(out + pay + (t - s) + max(0, t - lb1) + max(0, t - lb2), (unsigned)fv_feats[t]);
    }
    fbase += chunk_total;
    __syncthreads(); // s_fv is reused by the next chunk
  }
  if (tid == 0) a.sizes[frame] = total;
}

} // namespace

void launch_serialize(const Params &p, const SerArgs &a, int n_frames, cudaStream_t s) { serialize_kernel<<<n_frames, kSerThreads, 0, s>>>(p, a); }

} // namespace orbx
