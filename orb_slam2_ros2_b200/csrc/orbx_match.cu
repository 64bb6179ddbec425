// orbx_match.cu -- tracking-side Hamming matchers (SURVEY.md section 8(f) rank 2), sm_100a.
//
//   area_match_kernel    VirtualFrame::findFeaturesInArea (src/Frame.cc:286-311) + the exclusion filter of
//                        ORBMatcher::searchByProjection (src/ORBMatcher.cc:322-331) + ORBMatcher::getBestMatch
//                        (src/ORBMatcher.cc:967-990), one warp per query, over the frame's device-resident CSR grid
//   bow_match_kernel     the matching loop of ORBMatcher::searchByBow (src/ORBMatcher.cc:170-255), one warp per keyframe
//                        feature, candidates = the frame's features under the same vocabulary node
//   verify_angle_kernel  ORBMatcher::verifyAngle (src/ORBMatcher.cc:1013-1051), one CTA per match list
//
// Both reproduce the reference's candidate ORDER (grid cells row-major, ascending keypoint index inside a cell), which
// decides ties of the best match and the value of the reference's order-dependent "second best".
#include "orbx_match.cuh"

namespace orbx
{

namespace
{

constexpr int kAreaWarps = 8;

// One warp per query.  Candidates are visited 32 at a time in the reference's order; getBestMatch's sequential rule
//   if (d < min) { min = d; idx = i; } else if (d < second) second = d;
// is evaluated per chunk with an exclusive prefix-minimum over the lanes: a candidate is a "new minimum" iff its
// distance is below every earlier one (the running minimum included); `second` is the minimum over all the others.
__global__ void __launch_bounds__(kAreaWarps * 32, 8) area_match_kernel(const Params p, const AreaArgs a)
{
  const int frame = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int qi = blockIdx.x * kAreaWarps + (threadIdx.x >> 5);
  const int n_q = a.n_q ? a.n_q[frame] : a.n_q_all;
  if (qi >= min(n_q, a.q_stride)) return;
  const size_t qo = (size_t)frame * a.q_stride + qi;
  const orbx_area_query q = a.q[qo];
  const int img = frame * a.image_stride;
  const orbx_keypoint *kps = p.kps_und + (size_t)img * p.n_features;
  const uint4 *desc = reinterpret_cast<const uint4 *>(p.desc + (size_t)img * p.n_features * 32);
  const int nc = p.grid_rows * p.grid_cols;
  const int *start = p.grid_start + (size_t)frame * (nc + 1);
  const uint16_t *entries = p.grid_entries + (size_t)frame * p.n_features;
  const uint8_t *excl = a.exclude ? a.exclude + (size_t)frame * p.n_features : nullptr;

  // findFeaturesInArea (src/Frame.cc:289-297); getScaledFactor2 = float(pow(double(sf), 2)) (Frame.h:207)
  const int oct = min(max(q.octave, 0), p.n_levels - 1);
  const double sfd = (double)p.levels[oct].sf;
  const float sf2 = (float)(sfd * sfd);
  const float radius = __fmul_rn(q.radius, sf2);
  const int min_x = max(0, __float2int_rn(__fsub_rn(q.x, radius)));
  const int max_x = min((int)a.max_u, __float2int_rn(__fadd_rn(q.x, radius)));
  const int min_y = max(0, __float2int_rn(__fsub_rn(q.y, radius)));
  const int max_y = min((int)a.max_v, __float2int_rn(__fadd_rn(q.y, radius)));
  int n_cand = 0, min_d = 0x7fffffff, second_d = 0x7fffffff, min_idx = -1;
  if (max_x >= 0 && max_y >= 0) // a window left of / above the image is undefined behaviour in the reference
  {
    const int c0 = __float2int_rd(__fdiv_rn((float)min_x, 64.f)), c1 = min(__float2int_rd(__fdiv_rn((float)max_x, 64.f)), p.grid_cols - 1);
    const int r0 = __float2int_rd(__fdiv_rn((float)min_y, 48.f)), r1 = min(__float2int_rd(__fdiv_rn((float)max_y, 48.f)), p.grid_rows - 1);
    const uint4 *qd = reinterpret_cast<const uint4 *>(a.q_desc + qo * 32);
    const uint4 q0 = __ldg(qd), q1 = __ldg(qd + 1);
    for (int r = r0; r <= r1; ++r)
    {
      // the cells c0..c1 of one grid row are contiguous in the CSR: one entry range per row
      const int e0 = (c0 <= c1) ? start[r * p.grid_cols + c0] : 0, e1 = (c0 <= c1) ? start[r * p.grid_cols + c1 + 1] : 0;
      for (int e = e0; e < e1; e += 32)
      {
        int id = -1, d = 0x7fffffff;
        if (e + lane < e1)
        {
          id = entries[e + lane];
          const int o = kps[id].octave;
          if (o > q.max_level || o < q.min_level || (excl && excl[id])) id = -1;
        }
        if (id >= 0) d = hamming256(q0, q1, __ldg(desc + 2 * id), __ldg(desc + 2 * id + 1));
        best_match_chunk(id, d, lane, n_cand, min_d, second_d, min_idx);
      }
    }
  }
  if (lane == 0)
  {
    a.n_cand[qo] = n_cand;
    a.best_idx[qo] = n_cand ? min_idx : -1;
    a.best_dist[qo] = min_d;
    a.ratio[qo] = n_cand ? __fdiv_rn((float)min_d, (float)second_d) : 0.f; // :988
  }
}

// The matching loop of ORBMatcher::searchByBow (src/ORBMatcher.cc:170-255): one warp per entry of the keyframe's
// FeatureVector (bow_match_row).
__global__ void __launch_bounds__(kAreaWarps * 32) bow_match_kernel(const BowMatchArgs a)
{
  const int lane = threadIdx.x & 31;
  const int e = blockIdx.x * kAreaWarps + (threadIdx.x >> 5);
  if (e >= a.k_n_listed) return;
  int n_cand, min_d, second_d, min_idx;
  bow_match_row(a, e, lane, n_cand, min_d, second_d, min_idx);
  if (lane == 0)
  {
    a.n_cand[e] = n_cand;
    a.best_idx[e] = n_cand ? min_idx : -1;
    a.best_dist[e] = min_d;
    a.ratio[e] = n_cand ? __fdiv_rn((float)min_d, (float)second_d) : 0.f;
  }
}

__global__ void __launch_bounds__(kVaThreads) verify_angle_kernel(const VerifyArgs a)
{
  const int n_out = verify_angle_block(
      a.n, [&](int i) { return angle_bin(a.kps1[a.query_idx[i]].angle, a.kps2[a.train_idx[i]].angle); },
      [&](int off, int i) {
        a.out_query[off] = a.query_idx[i];
        a.out_train[off] = a.train_idx[i];
        a.out_dist[off] = a.distance[i];
      });
  if (threadIdx.x == 0) *a.n_out = n_out;
}

} // namespace

void launch_area_match(const Params &p, const AreaArgs &a, int n_frames, cudaStream_t s)
{
  dim3 grid((a.q_stride + kAreaWarps - 1) / kAreaWarps, n_frames);
  area_match_kernel<<<grid, kAreaWarps * 32, 0, s>>>(p, a);
}

void launch_verify_angle(const VerifyArgs &a, cudaStream_t s) { verify_angle_kernel<<<1, kVaThreads, 0, s>>>(a); }

void launch_bow_match(const BowMatchArgs &a, cudaStream_t s)
{
  bow_match_kernel<<<(a.k_n_listed + kAreaWarps - 1) / kAreaWarps, kAreaWarps * 32, 0, s>>>(a);
}

} // namespace orbx
