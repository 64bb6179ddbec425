// orbx_match.cuh -- device code of the Hamming matchers, shared by orbx_match.cu (one query per launch) and orbx_loop.cu
// (every (query, candidate) pair of a loop-candidate table in one launch).
#pragma once

#include "orbx_device.cuh"

namespace orbx
{

// One chunk of up to 32 candidates (lane order == the reference's candidate order; id < 0: no candidate on this lane) of
// ORBMatcher::getBestMatch (src/ORBMatcher.cc:967-990).  The sequential rule
//   if (d < min) { min = d; idx = i; } else if (d < second) second = d;
// is evaluated with an exclusive prefix-minimum over the lanes: a candidate is a "new minimum" iff its distance is below
// every earlier one (the running minimum included); `second` is the minimum over all the others.
__device__ __forceinline__ void best_match_chunk(int id, int d, int lane, int &n_cand, int &min_d, int &second_d, int &min_idx)
{
  const unsigned valid = __ballot_sync(kFullMask, id >= 0);
  if (!valid) return;
  n_cand += __popc(valid);
  int pm = d; // exclusive prefix minimum over the lanes, seeded with the running minimum
#pragma unroll
  for (int s = 1; s < 32; s <<= 1)
  {
    const int t = __shfl_up_sync(kFullMask, pm, s);
    if (lane >= s) pm = min(pm, t);
  }
  int ex = __shfl_up_sync(kFullMask, pm, 1);
  if (lane == 0) ex = 0x7fffffff;
  ex = min(ex, min_d);
  const bool is_new = id >= 0 && d < ex;
  int sec = (id >= 0 && !is_new) ? d : 0x7fffffff;
#pragma unroll
  for (int s = 16; s; s >>= 1) sec = min(sec, __shfl_xor_sync(kFullMask, sec, s));
  second_d = min(second_d, sec);
  // the last "new minimum" lane of the chunk holds the chunk's minimum at its first occurrence
  const unsigned news = __ballot_sync(kFullMask, is_new);
  if (news)
  {
    const int src = 31 - __clz(news);
    min_d = __shfl_sync(kFullMask, d, src);
    min_idx = __shfl_sync(kFullMask, id, src);
  }
}

// One row of the matching loop of ORBMatcher::searchByBow (src/ORBMatcher.cc:170-255), for a whole warp: entry e of the
// keyframe's FeatureVector.  Its vocabulary node is looked up in the frame's FeatureVector (both sorted by node id: binary
// searches replace the reference's merge-join); candidates = the frame's features of that node that pass the mask.
__device__ __forceinline__ void bow_match_row(const BowMatchArgs &a, int e, int lane, int &n_cand, int &min_d, int &second_d, int &min_idx)
{
  n_cand = 0, min_d = 0x7fffffff, second_d = 0x7fffffff, min_idx = -1;
  const int pk = a.k_feats[e];
  if (a.kf_query_ok && !a.kf_query_ok[pk]) return;
  // keyframe node segment containing entry e: last j with k_start[j] <= e
  int lo = 0, hi = a.k_n_nodes;
  while (hi - lo > 1)
  {
    const int mid = (lo + hi) >> 1;
    if (a.k_start[mid] <= e) lo = mid; else hi = mid;
  }
  const int node = a.k_nodes[lo];
  const int f_n = *a.f_n_nodes;
  const int l2 = lower_bound(a.f_nodes, 0, f_n, node);
  if (l2 >= f_n || a.f_nodes[l2] != node) return;
  const uint4 *qd = reinterpret_cast<const uint4 *>(a.k_desc + (size_t)pk * 32);
  const uint4 q0 = __ldg(qd), q1 = __ldg(qd + 1);
  const uint4 *fd = reinterpret_cast<const uint4 *>(a.f_desc);
  const int t0 = a.f_start[l2], t1 = a.f_start[l2 + 1];
  for (int t = t0; t < t1; t += 32)
  {
    int id = -1, d = 0x7fffffff;
    if (t + lane < t1)
    {
      id = a.f_feats[t + lane];
      if (a.frame_cand_ok && !a.frame_cand_ok[id]) id = -1;
    }
    if (id >= 0) d = hamming256(q0, q1, __ldg(fd + 2 * id), __ldg(fd + 2 * id + 1));
    best_match_chunk(id, d, lane, n_cand, min_d, second_d, min_idx);
  }
}

constexpr int kVaThreads = 256;
constexpr int kVaBins = 30;   // ORBMatcher::mnBinNum   (src/ORBMatcher.cc:1091)
constexpr int kVaChoose = 3;  // ORBMatcher::mnBinChoose (src/ORBMatcher.cc:1092)

// the rotation bin of a match whose keypoint angles are a1 (kps1[queryIdx]) and a2 (kps2[trainIdx])
__device__ __forceinline__ int angle_bin(float a1, float a2)
{
  float diff = __fsub_rn(a1, a2);
  diff = diff >= 0.f ? diff : __fadd_rn(360.f, diff);
  int b = (int)__fdiv_rn(diff, 12.f); // 360 / mnBinNum is an integer division in the reference
  if (b == 30) b = 0;
  return min(max(b, 0), kVaBins - 1);
}

// ORBMatcher::verifyAngle (src/ORBMatcher.cc:1013-1051) over matches 0 .. n-1, run by one CTA of kVaThreads threads: keeps the
// matches in the three fullest of the 30 bins; emit(out, i) stores match i at position `out` of the reference's order
// (ascending bin, original order inside a bin).  Returns the number kept, in every thread.
template <class BinOf, class Emit> __device__ __forceinline__ int verify_angle_block(int n, BinOf bin_of, Emit emit)
{
  __shared__ int s_count[kVaBins], s_base[kVaBins], s_wcount[kVaThreads / 32][kVaBins], s_total;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < kVaBins) s_count[tid] = 0;
  __syncthreads();
  for (int i = tid; i < n; i += kVaThreads) atomicAdd(&s_count[bin_of(i)], 1);
  __syncthreads();
  if (tid == 0)
  {
    bool good[kVaBins];
    for (int b = 0; b < kVaBins; ++b) good[b] = false;
    for (int k = 0; k < kVaChoose; ++k)
    {
      int max_size = 0, max_id = 0;
      bool init = false;
      for (int b = 0; b < kVaBins; ++b)
      {
        if (good[b]) continue;
        if (s_count[b] > max_size) max_id = b, max_size = s_count[b], init = true;
      }
      if (init) good[max_id] = true;
    }
    int off = 0;
    for (int b = 0; b < kVaBins; ++b) // std::set iteration: ascending bin id
    {
      s_base[b] = good[b] ? off : -1;
      if (good[b]) off += s_count[b];
    }
    s_total = off;
  }
  __syncthreads();
  // stable scatter: chunks of kVaThreads matches in order; rank inside a chunk from warp match masks + per-warp counts
  for (int i0 = 0; i0 < n; i0 += kVaThreads)
  {
    for (int k = tid; k < (kVaThreads / 32) * kVaBins; k += kVaThreads) (&s_wcount[0][0])[k] = 0;
    __syncthreads();
    const int i = i0 + tid;
    const int b = i < n ? bin_of(i) : -1;
    const unsigned same = __match_any_sync(kFullMask, b);
    const int rank = __popc(same & ((1u << lane) - 1));
    if (b >= 0 && rank == 0) s_wcount[warp][b] = __popc(same);
    __syncthreads();
    if (b >= 0 && s_base[b] >= 0)
    {
      int off = s_base[b] + rank;
      for (int w = 0; w < warp; ++w) off += s_wcount[w][b];
      emit(off, i);
    }
    __syncthreads();
    if (tid < kVaBins && s_base[tid] >= 0)
    {
      int add = 0;
      for (int w = 0; w < kVaThreads / 32; ++w) add += s_wcount[w][tid];
      s_base[tid] += add;
    }
    __syncthreads();
  }
  return s_total;
}

} // namespace orbx
