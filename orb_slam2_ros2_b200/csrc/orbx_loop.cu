// orbx_loop.cu -- loop verification (orbx_loopver_*): searchByBow + verifyAngle + a fixed-scale Horn RANSAC for every
// (query, candidate) pair of a loop-candidate table, sm_100a.
//
// Restates the geometric check of ORB-SLAM2's LoopClosing::ComputeSim3 (SearchByBoW, the rotation check, Sim3Solver with a
// fixed scale) under the rules of include/orbx.h; tests/loopver_oracle.c is the sequential restatement the kernels are tested
// against bit for bit.
//   build: loopver_extract_kernel copies keypoints (x, y, angle, octave), descriptors and depth out of the records into
//   arrays the verifier owns; the FeatureVectors come from bow_frames (bow_descend_kernel + bow_assemble_kernel, orbx_bow.cu).
//   verify: loopver_pair_kernel, one 256-thread CTA per pair (a grid-stride loop over the pairs), per-CTA scratch in global
//   memory:
//     rows          a warp per row of the candidate's FeatureVector (bow_match_row, orbx_match.cuh)
//     compaction    the kept rows in row order (block scans over chunks of 256 rows)
//     verifyAngle   verify_angle_block (orbx_match.cuh), the body of verify_angle_kernel
//     points        the matches with two depths, compacted in match order, back-projected in double
//     RANSAC        rounds of 8 hypotheses, one per warp: lane 0 draws the 3 samples and solves Horn (a serial 4x4 Jacobi),
//                   the warp's lanes count the inliers over the points; after each round thread 0 walks the round's
//                   counts in hypothesis order (the first > min_inliers stops, else the last among the maxima)
//     refit         warp 0: the rule's 32 slot partials over the inliers are the lanes, the tree is __shfl_down_sync
//   loopver_loop_frame_kernel turns the per-query minimum (hypothesis / 5, table position) into loop_frame.
//   Every double operation on the solver path is an explicit __dadd_rn / __dsub_rn / __dmul_rn / __ddiv_rn / __dsqrt_rn.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "orbx_internal.h"
#include "orbx_match.cuh"

struct orbx_loopver
{
  const orbx_ctx *ctx = nullptr;
  const orbx_vocab *vocab = nullptr;
  int device = 0;
  int F = 0, N = 0;
  float4 *kp = nullptr;       // [F][N] x, y, angle, octave (int bits)
  uint8_t *desc = nullptr;    // [F][N][32]
  double *depth = nullptr;    // [F][N]
  int *n = nullptr;           // [F]
  int *fv_nodes = nullptr, *fv_start = nullptr, *fv_feats = nullptr, *n_fv = nullptr; // FeatureVector CSR per frame
  int grid_max = 0;           // resident CTAs of the pair kernel
  orbx::DeviceBuffer scratch; // [grid_max][per-CTA scratch]
  orbx::DeviceBuffer staging; // iteration table, host tables and outputs of host-io calls
};

namespace orbx
{

namespace
{

constexpr int kLT = 256;   // threads of the pair CTA
constexpr int kLW = kLT / 32;
constexpr int kRound = kLW; // hypotheses per RANSAC round: one per warp
constexpr int kRecChunk = 64; // host records staged per extraction launch

// one correspondence: candidate / query point in its camera, the keypoints and their inlier bounds 9.210 * sigma2
struct Corr
{
  double c[3], q[3];
  double thr_c, thr_q;
  float uc, vc, uq, vq;
};

struct LvArgs
{
  const float4 *kp;
  const uint8_t *desc;
  const double *depth;
  const int *n, *fv_nodes, *fv_start, *fv_feats, *n_fv;
  int F, N;
  double fx, fy, cx, cy;
  double thr[kMaxLevels];
  const int *iters; // [N + 1] RANSAC iterations per n_corr
  const int *table;
  int top_k, n_queries;
  long long q_lo;
  float ratio;
  int min_matches, min_inliers;
  unsigned long long seed_key; // splitmix64(seed)
  uint8_t *scratch;
  size_t cta_bytes;
  int *n_bow, *n_matches, *n_corr, *n_iters, *hypothesis, *n_inliers, *accepted, *match;
  double *T;
  unsigned long long *loop_key; // [n_queries]
};

__device__ __forceinline__ double dA(double x, double y) { return __dadd_rn(x, y); }
__device__ __forceinline__ double dS(double x, double y) { return __dsub_rn(x, y); }
__device__ __forceinline__ double dM(double x, double y) { return __dmul_rn(x, y); }
__device__ __forceinline__ double dD(double x, double y) { return __ddiv_rn(x, y); }

// the sum rule of include/orbx.h for three points in slots 0, 1, 2: p_j = 0 + x_j, the tree adds p_2 to p_0, then p_1
__device__ __forceinline__ double sum3(double x0, double x1, double x2) { return dA(dA(dA(0.0, x0), dA(0.0, x2)), dA(0.0, x1)); }

// Horn's closed form after the sums: N from M, cyclic Jacobi, quaternion of the largest eigenvalue, R / |q|^2, t.
// T[0..8] = R row-major, T[9..11] = t, T[12..14] = -R^T t (the inverse's translation, for the inlier test)
__device__ __noinline__ void horn_finish(const double cc[3], const double cq[3], const double M[9], double *T)
{
  double a[4][4], v[4][4];
  a[0][0] = dA(dA(M[0], M[4]), M[8]);
  a[0][1] = dS(M[5], M[7]);
  a[0][2] = dS(M[6], M[2]);
  a[0][3] = dS(M[1], M[3]);
  a[1][1] = dS(dS(M[0], M[4]), M[8]);
  a[1][2] = dA(M[1], M[3]);
  a[1][3] = dA(M[6], M[2]);
  a[2][2] = dS(dA(-M[0], M[4]), M[8]);
  a[2][3] = dA(M[5], M[7]);
  a[3][3] = dA(dS(-M[0], M[4]), M[8]);
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
    {
      if (j < i) a[i][j] = a[j][i];
      v[i][j] = i == j ? 1.0 : 0.0;
    }
  for (int sweep = 0; sweep < ORBX_LOOPVER_JACOBI_SWEEPS; ++sweep)
  {
    if (a[0][1] == 0.0 && a[0][2] == 0.0 && a[0][3] == 0.0 && a[1][2] == 0.0 && a[1][3] == 0.0 && a[2][3] == 0.0) break;
#pragma unroll
    for (int p = 0; p < 3; ++p)
#pragma unroll
      for (int q = p + 1; q < 4; ++q)
      {
        const double apq = a[p][q];
        if (apq == 0.0) continue;
        const double theta = dD(dS(a[q][q], a[p][p]), dM(2.0, apq));
        double t = dD(1.0, dA(fabs(theta), __dsqrt_rn(dA(dM(theta, theta), 1.0))));
        if (theta < 0.0) t = -t;
        const double c = dD(1.0, __dsqrt_rn(dA(dM(t, t), 1.0))), s = dM(t, c);
#pragma unroll
        for (int k = 0; k < 4; ++k)
        {
          const double akp = a[k][p], akq = a[k][q];
          a[k][p] = dS(dM(c, akp), dM(s, akq));
          a[k][q] = dA(dM(s, akp), dM(c, akq));
        }
#pragma unroll
        for (int k = 0; k < 4; ++k)
        {
          const double apk = a[p][k], aqk = a[q][k];
          a[p][k] = dS(dM(c, apk), dM(s, aqk));
          a[q][k] = dA(dM(s, apk), dM(c, aqk));
        }
        a[p][q] = 0.0;
        a[q][p] = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
        {
          const double vkp = v[k][p], vkq = v[k][q];
          v[k][p] = dS(dM(c, vkp), dM(s, vkq));
          v[k][q] = dA(dM(s, vkp), dM(c, vkq));
        }
      }
  }
  double best = a[0][0], w = v[0][0], x = v[1][0], y = v[2][0], z = v[3][0];
#pragma unroll
  for (int m = 1; m < 4; ++m)
    if (a[m][m] > best) best = a[m][m], w = v[0][m], x = v[1][m], y = v[2][m], z = v[3][m];
  const double ww = dM(w, w), xx = dM(x, x), yy = dM(y, y), zz = dM(z, z);
  const double n2 = dA(dA(dA(ww, xx), yy), zz);
  const double xy = dM(x, y), xz = dM(x, z), yz = dM(y, z), wx = dM(w, x), wy = dM(w, y), wz = dM(w, z);
  T[0] = dD(dS(dS(dA(ww, xx), yy), zz), n2);
  T[1] = dD(dM(2.0, dS(xy, wz)), n2);
  T[2] = dD(dM(2.0, dA(xz, wy)), n2);
  T[3] = dD(dM(2.0, dA(xy, wz)), n2);
  T[4] = dD(dS(dA(dS(ww, xx), yy), zz), n2);
  T[5] = dD(dM(2.0, dS(yz, wx)), n2);
  T[6] = dD(dM(2.0, dS(xz, wy)), n2);
  T[7] = dD(dM(2.0, dA(yz, wx)), n2);
  T[8] = dD(dA(dS(dS(ww, xx), yy), zz), n2);
#pragma unroll
  for (int r = 0; r < 3; ++r) T[9 + r] = dS(cq[r], dA(dA(dM(T[3 * r], cc[0]), dM(T[3 * r + 1], cc[1])), dM(T[3 * r + 2], cc[2])));
#pragma unroll
  for (int r = 0; r < 3; ++r) T[12 + r] = -dA(dA(dM(T[r], T[9]), dM(T[3 + r], T[10])), dM(T[6 + r], T[11]));
}

__device__ __forceinline__ bool is_inlier(const Corr &k, const double *T, const LvArgs &a)
{
  double Y[3], Z[3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
  {
    Y[r] = dA(dA(dA(dM(T[3 * r], k.c[0]), dM(T[3 * r + 1], k.c[1])), dM(T[3 * r + 2], k.c[2])), T[9 + r]);
    Z[r] = dA(dA(dA(dM(T[r], k.q[0]), dM(T[3 + r], k.q[1])), dM(T[6 + r], k.q[2])), T[12 + r]);
  }
  const double iy = dD(1.0, Y[2]), iz = dD(1.0, Z[2]);
  const double du1 = dS((double)k.uq, dA(dM(a.fx, dM(Y[0], iy)), a.cx)), dv1 = dS((double)k.vq, dA(dM(a.fy, dM(Y[1], iy)), a.cy));
  const double du2 = dS((double)k.uc, dA(dM(a.fx, dM(Z[0], iz)), a.cx)), dv2 = dS((double)k.vc, dA(dM(a.fy, dM(Z[1], iz)), a.cy));
  return dA(dM(du1, du1), dM(dv1, dv1)) < k.thr_q && dA(dM(du2, du2), dM(dv2, dv2)) < k.thr_c;
}

// Horn over the three samples of hypothesis h (include/orbx.h: draws, avail swaps, slots 0, 1, 2)
__device__ __noinline__ void hypothesis_solve(const Corr *corr, int n, unsigned long long K, int h, double *T)
{
  int r[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) r[j] = (int)(splitmix64(K ^ ((unsigned long long)(3 * h + j) * kGolden)) % (unsigned long long)(n - j));
  // avail after the first draw: avail1(k) = k == r0 ? n - 1 : k; after the second: avail2(k) = k == r1 ? avail1(n - 2) : avail1(k)
  auto avail1 = [&](int k) { return k == r[0] ? n - 1 : k; };
  auto avail2 = [&](int k) { return k == r[1] ? avail1(n - 2) : avail1(k); };
  const Corr &k0 = corr[r[0]], &k1 = corr[avail1(r[1])], &k2 = corr[avail2(r[2])];
  double cc[3], cq[3], M[9];
#pragma unroll
  for (int d = 0; d < 3; ++d)
  {
    cc[d] = dD(sum3(k0.c[d], k1.c[d], k2.c[d]), 3.0);
    cq[d] = dD(sum3(k0.q[d], k1.q[d], k2.q[d]), 3.0);
  }
#pragma unroll
  for (int x = 0; x < 3; ++x)
#pragma unroll
    for (int y = 0; y < 3; ++y)
      M[3 * x + y] = sum3(dM(dS(k0.c[x], cc[x]), dS(k0.q[y], cq[y])), dM(dS(k1.c[x], cc[x]), dS(k1.q[y], cq[y])),
                          dM(dS(k2.c[x], cc[x]), dS(k2.q[y], cq[y])));
  horn_finish(cc, cq, M, T);
}

__device__ __forceinline__ double tree_sum(double p)
{
#pragma unroll
  for (int s = 16; s; s >>= 1) p = dA(p, __shfl_down_sync(kMatchFull, p, s));
  return __shfl_sync(kMatchFull, p, 0);
}

// Horn over the inliers of T0 in correspondence order, by one warp (lane l = the rule's partial of slot l)
__device__ __noinline__ void refit_warp(const Corr *corr, int n, int m, const double *T0, const LvArgs &a, double *T)
{
  const int lane = threadIdx.x & 31;
  double cc[3], cq[3], M[9];
  {
    double p[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int i = lane; i < n; i += 32)
      if (is_inlier(corr[i], T0, a))
#pragma unroll
        for (int d = 0; d < 3; ++d) p[d] = dA(p[d], corr[i].c[d]), p[3 + d] = dA(p[3 + d], corr[i].q[d]);
#pragma unroll
    for (int d = 0; d < 3; ++d) cc[d] = dD(tree_sum(p[d]), (double)m), cq[d] = dD(tree_sum(p[3 + d]), (double)m);
  }
  double p[9];
#pragma unroll
  for (int j = 0; j < 9; ++j) p[j] = 0.0;
  for (int i = lane; i < n; i += 32)
  {
    const Corr &k = corr[i];
    if (!is_inlier(k, T0, a)) continue;
#pragma unroll
    for (int x = 0; x < 3; ++x)
#pragma unroll
      for (int y = 0; y < 3; ++y) p[3 * x + y] = dA(p[3 * x + y], dM(dS(k.c[x], cc[x]), dS(k.q[y], cq[y])));
  }
#pragma unroll
  for (int j = 0; j < 9; ++j) M[j] = tree_sum(p[j]);
  if (lane == 0) horn_finish(cc, cq, M, T);
}

__global__ void __launch_bounds__(kLT) loopver_pair_kernel(const LvArgs a)
{
  __shared__ int s_warp[kLW];
  __shared__ double s_T[kRound][15], s_best[15], s_fit[15];
  __shared__ int s_cnt[kRound], s_best_h, s_best_n, s_acc;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int N = a.N;
  uint8_t *cta = a.scratch + (size_t)blockIdx.x * a.cta_bytes;
  Corr *corr = reinterpret_cast<Corr *>(cta);
  int *row = reinterpret_cast<int *>(cta + (size_t)N * sizeof(Corr));
  int *kq = row + N, *kc = kq + N, *mq = kc + N, *mc = mq + N;
  const long long n_pairs = (long long)a.n_queries * a.top_k;
  for (long long pair = blockIdx.x; pair < n_pairs; pair += gridDim.x)
  {
    const int qi = (int)(pair / a.top_k), slot = (int)(pair - (long long)qi * a.top_k);
    const int qf = (int)(a.q_lo + qi);
    int cf = a.table[pair];
    if (cf < 0 || cf >= a.F) cf = -1;
    int nb = 0, nm = 0, ncorr = 0, nit = 0;
    if (tid == 0) s_best_h = -1, s_best_n = 0, s_acc = 0;
    if (cf >= 0)
    {
      const size_t qo = (size_t)qf * N, co = (size_t)cf * N;
      const float4 *kp_q = a.kp + qo, *kp_c = a.kp + co;
      const double *dep_q = a.depth + qo, *dep_c = a.depth + co;
      // 1. searchByBow rows: the candidate is the keyframe, the query the frame, no masks
      BowMatchArgs m{};
      m.f_nodes = a.fv_nodes + qo, m.f_start = a.fv_start + (size_t)qf * (N + 1), m.f_feats = a.fv_feats + qo, m.f_n_nodes = a.n_fv + qf;
      m.f_desc = a.desc + qo * 32;
      m.k_nodes = a.fv_nodes + co, m.k_start = a.fv_start + (size_t)cf * (N + 1), m.k_feats = a.fv_feats + co, m.k_n_nodes = a.n_fv[cf];
      m.k_desc = a.desc + co * 32;
      const int n_rows = m.k_start[m.k_n_nodes];
      for (int e = warp; e < n_rows; e += kLW)
      {
        int n_cand, min_d, second_d, min_idx;
        bow_match_row(m, e, lane, n_cand, min_d, second_d, min_idx);
        if (lane == 0)
        {
          const float ratio = n_cand ? __fdiv_rn((float)min_d, (float)second_d) : 0.f;
          row[e] = (n_cand && min_d <= 50 && !(ratio > a.ratio)) ? min_idx : -1;
        }
      }
      __syncthreads();
      // 2. the kept rows, in row order
      for (int e0 = 0; e0 < n_rows; e0 += kLT)
      {
        const int e = e0 + tid;
        const bool keep = e < n_rows && row[e] >= 0;
        int tot;
        const int pos = nb + block_exscan<kLT>(keep, &tot, s_warp);
        if (keep) kq[pos] = row[e], kc[pos] = m.k_feats[e];
        nb += tot;
      }
      __syncthreads();
      // 3. verifyAngle: kps1 = the query's, kps2 = the candidate's keypoints
      nm = verify_angle_block(
          nb, [&](int i) { return angle_bin(kp_q[kq[i]].z, kp_c[kc[i]].z); },
          [&](int off, int i) {
            mq[off] = kq[i];
            mc[off] = kc[i];
          });
      if (nm >= a.min_matches)
      {
        // 4. correspondences: both depths > 0, in match order
        for (int i0 = 0; i0 < nm; i0 += kLT)
        {
          const int i = i0 + tid;
          const bool ok = i < nm && dep_c[mc[i]] > 0.0 && dep_q[mq[i]] > 0.0;
          int tot;
          const int pos = ncorr + block_exscan<kLT>(ok, &tot, s_warp);
          if (ok)
          {
            Corr k;
            const float4 pc = kp_c[mc[i]], pq = kp_q[mq[i]];
            const double zc = dep_c[mc[i]], zq = dep_q[mq[i]];
            k.c[0] = dD(dM(dS((double)pc.x, a.cx), zc), a.fx), k.c[1] = dD(dM(dS((double)pc.y, a.cy), zc), a.fy), k.c[2] = zc;
            k.q[0] = dD(dM(dS((double)pq.x, a.cx), zq), a.fx), k.q[1] = dD(dM(dS((double)pq.y, a.cy), zq), a.fy), k.q[2] = zq;
            k.thr_c = a.thr[min(max(__float_as_int(pc.w), 0), kMaxLevels - 1)];
            k.thr_q = a.thr[min(max(__float_as_int(pq.w), 0), kMaxLevels - 1)];
            k.uc = pc.x, k.vc = pc.y, k.uq = pq.x, k.vq = pq.y;
            corr[pos] = k;
          }
          ncorr += tot;
        }
        __syncthreads();
        // 5. RANSAC in rounds of kRound hypotheses
        nit = a.iters[ncorr];
        const unsigned long long K = splitmix64(splitmix64(a.seed_key + (unsigned long long)qf + 1) + (unsigned long long)cf + 1);
        for (int h0 = 0; h0 < nit; h0 += kRound)
        {
          const int h = h0 + warp;
          if (h < nit)
          {
            if (lane == 0) hypothesis_solve(corr, ncorr, K, h, s_T[warp]);
            __syncwarp();
            int cnt = 0;
            for (int i = lane; i < ncorr; i += 32) cnt += is_inlier(corr[i], s_T[warp], a);
#pragma unroll
            for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(kMatchFull, cnt, o);
            if (lane == 0) s_cnt[warp] = cnt;
          }
          __syncthreads();
          if (tid == 0)
            for (int w = 0; w < kRound && h0 + w < nit; ++w)
              if (s_cnt[w] >= s_best_n)
              {
                s_best_n = s_cnt[w], s_best_h = h0 + w;
                for (int j = 0; j < 15; ++j) s_best[j] = s_T[w][j];
                if (s_cnt[w] > a.min_inliers)
                {
                  s_acc = 1;
                  break;
                }
              }
          __syncthreads();
          if (s_acc) break;
        }
        // 6. the refit over the inliers of the reported hypothesis
        if (s_best_h >= 0 && warp == 0)
        {
          if (s_best_n >= 3) refit_warp(corr, ncorr, s_best_n, s_best, a, s_fit);
          else if (lane == 0)
            for (int j = 0; j < 15; ++j) s_fit[j] = s_best[j];
        }
      }
    }
    __syncthreads();
    const size_t o = (size_t)pair;
    if (a.match)
    {
      int *mrow = a.match + o * N;
      for (int j = tid; j < N; j += kLT) mrow[j] = -1;
      __syncthreads();
      for (int i = tid; i < nm; i += kLT) mrow[mc[i]] = mq[i];
    }
    if (tid == 0)
    {
      const int hyp = s_best_h, acc = s_acc;
      if (a.n_bow) a.n_bow[o] = nb;
      if (a.n_matches) a.n_matches[o] = nm;
      if (a.n_corr) a.n_corr[o] = ncorr;
      if (a.n_iters) a.n_iters[o] = acc ? hyp + 1 : nit;
      if (a.hypothesis) a.hypothesis[o] = hyp;
      if (a.n_inliers) a.n_inliers[o] = hyp >= 0 ? s_best_n : 0;
      if (a.accepted) a.accepted[o] = acc;
      if (a.T)
        for (int j = 0; j < 12; ++j) a.T[o * 12 + j] = hyp >= 0 ? s_fit[j] : 0.0;
      if (acc && a.loop_key) atomicMin(&a.loop_key[qi], ((unsigned long long)(hyp / 5) << 32) | (unsigned)slot);
    }
    __syncthreads(); // the scratch and the shared state are reused by the next pair
  }
}

__global__ void __launch_bounds__(256) loopver_loop_frame_kernel(const int *table, int top_k, int n_queries, const unsigned long long *key, int *loop_frame)
{
  const int q = blockIdx.x * 256 + threadIdx.x;
  if (q >= n_queries) return;
  const unsigned long long k = key[q];
  loop_frame[q] = k == ~0ull ? -1 : table[(size_t)q * top_k + (unsigned)(k & 0xffffffffu)];
}

// frame f0 + f's record -> the verifier's arrays
__global__ void __launch_bounds__(256) loopver_extract_kernel(const uint8_t *rec, size_t stride, orbx_record_layout lay, int f0, int N, float4 *kp,
                                                              uint8_t *desc, double *depth, int *n)
{
  const int f = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
  const uint8_t *r = rec + (size_t)f * stride;
  const int nl = *reinterpret_cast<const int *>(r);
  const size_t o = (size_t)(f0 + f) * N + i;
  if (i == 0) n[f0 + f] = nl;
  if (i >= N) return;
  float4 k = make_float4(0.f, 0.f, 0.f, 0.f);
  double z = 0.0;
  uint4 d0 = make_uint4(0, 0, 0, 0), d1 = d0;
  if (i < nl)
  {
    const orbx_keypoint *kps = reinterpret_cast<const orbx_keypoint *>(r + lay.off_kps_left);
    k = make_float4(kps[i].x, kps[i].y, kps[i].angle, __int_as_float(kps[i].octave));
    const uint4 *dd = reinterpret_cast<const uint4 *>(r + lay.off_desc_left) + 2 * i;
    d0 = dd[0], d1 = dd[1];
    z = reinterpret_cast<const double *>(r + lay.off_depth)[i];
  }
  kp[o] = k;
  reinterpret_cast<uint4 *>(desc)[2 * o] = d0;
  reinterpret_cast<uint4 *>(desc)[2 * o + 1] = d1;
  depth[o] = z;
}

size_t up16(size_t v) { return (v + 15) & ~(size_t)15; }

size_t cta_bytes(int N) { return up16((size_t)N * sizeof(Corr) + (size_t)N * 5 * 4); }

} // namespace

} // namespace orbx

using namespace orbx;

namespace
{

struct LvGuard
{
  orbx_loopver *lv;
  ~LvGuard()
  {
    if (lv) orbx_loopver_destroy(lv);
  }
};

// SetRansacParameters (include/orbx.h: iterations) for every n_corr in 0..N
std::vector<int32_t> iteration_table(int N, const orbx_loopver_params *p)
{
  std::vector<int32_t> t((size_t)N + 1, 0);
  for (int n = p->min_inliers; n <= N; ++n)
  {
    double it = 1.0;
    if (n != p->min_inliers)
    {
      const float eps = (float)p->min_inliers / (float)n;
      it = std::ceil(std::log(1.0 - p->probability) / std::log(1.0 - std::pow((double)eps, 3.0)));
    }
    t[(size_t)n] = it < 1.0 ? 1 : it > (double)p->max_iterations ? p->max_iterations : (int32_t)it;
  }
  return t;
}

} // namespace

extern "C"
{

  void orbx_loopver_destroy(orbx_loopver *lv)
  {
    if (!lv) return;
    cudaSetDevice(lv->device);
    for (void *p : {(void *)lv->kp, (void *)lv->desc, (void *)lv->depth, (void *)lv->n, (void *)lv->fv_nodes, (void *)lv->fv_start, (void *)lv->fv_feats,
                    (void *)lv->n_fv})
      cudaFree(p);
    delete lv;
  }

  int orbx_loopver_build(orbx_ctx *c, const orbx_vocab *v, int32_t levelsup, const void *records, size_t record_stride, int32_t F, int32_t on_device,
                         orbx_loopver **out)
  {
    if (!c || !v || !records || !out) return ORBX_ERR_INVALID_ARG;
    *out = nullptr;
    if (v->ctx != c || v->device != c->device) return fail(c, ORBX_ERR_INVALID_ARG, "the vocabulary belongs to another context");
    orbx_record_layout lay;
    orbx_record_layout_get(c, &lay);
    if (F < 1) return fail(c, ORBX_ERR_INVALID_ARG, "loop verifier: n_frames < 1");
    if (record_stride < (size_t)lay.record_bytes || record_stride % 16) return fail(c, ORBX_ERR_INVALID_ARG, "loop verifier: record_stride below record_bytes or not a multiple of 16");
    // device records are read in place with 16-byte loads; host records go through the (aligned) staging buffer
    if (on_device && ((uintptr_t)records & 15)) return fail(c, ORBX_ERR_INVALID_ARG, "loop verifier: device records must be 16-byte aligned");
    if (levelsup < 0) return fail(c, ORBX_ERR_INVALID_ARG, "loop verifier: levelsup < 0");
    const int N = c->cfg.n_features;
    cudaStream_t s = c->stream;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    if (int rc = bow_configure(c, N, ORBX_ERR_CAPACITY)) return rc;
    orbx_loopver *lv = new orbx_loopver();
    LvGuard guard{lv};
    lv->ctx = c, lv->vocab = v, lv->device = c->device, lv->F = F, lv->N = N;
    const size_t e = (size_t)F * N;
    ORBX_CUDA(c, cudaMalloc((void **)&lv->kp, e * sizeof(float4)));
    ORBX_CUDA(c, cudaMalloc((void **)&lv->desc, e * 32));
    ORBX_CUDA(c, cudaMalloc((void **)&lv->depth, e * 8));
    ORBX_CUDA(c, cudaMalloc((void **)&lv->n, (size_t)F * 4));
    ORBX_CUDA(c, cudaMalloc((void **)&lv->fv_nodes, e * 4));
    ORBX_CUDA(c, cudaMalloc((void **)&lv->fv_start, (size_t)F * (N + 1) * 4));
    ORBX_CUDA(c, cudaMalloc((void **)&lv->fv_feats, e * 4));
    ORBX_CUDA(c, cudaMalloc((void **)&lv->n_fv, (size_t)F * 4));
    // the records' fields, in chunks of kRecChunk frames through a staging buffer when they live on the host
    DeviceBuffer stage;
    if (!on_device)
      if (int rc = stage.reserve(c, (size_t)std::min(F, kRecChunk) * record_stride)) return rc;
    const dim3 blk(256);
    for (int f0 = 0; f0 < F; f0 += kRecChunk)
    {
      const int nf = std::min(kRecChunk, F - f0);
      const uint8_t *src = (const uint8_t *)records + (size_t)f0 * record_stride;
      if (!on_device)
      {
        ORBX_CUDA(c, cudaMemcpyAsync(stage.p, src, (size_t)nf * record_stride, cudaMemcpyHostToDevice, s));
        src = stage.p;
      }
      loopver_extract_kernel<<<dim3((N + 255) / 256, nf), blk, 0, s>>>(src, record_stride, lay, f0, N, lv->kp, lv->desc, lv->depth, lv->n);
      ++c->launches;
    }
    ORBX_CUDA(c, cudaGetLastError());
    std::vector<int32_t> h_n((size_t)F);
    ORBX_CUDA(c, cudaMemcpyAsync(h_n.data(), lv->n, (size_t)F * 4, cudaMemcpyDeviceToHost, s));
    ORBX_CUDA(c, cudaStreamSynchronize(s));
    for (int32_t x : h_n)
      if (x < 0 || x > N) return fail(c, ORBX_ERR_INVALID_ARG, "loop verifier: a record's n_left lies outside 0..n_features");
    BowArgs fv{};
    fv.fv_nodes = lv->fv_nodes, fv.fv_start = lv->fv_start, fv.fv_feats = lv->fv_feats, fv.n_fv = lv->n_fv;
    if (int rc = bow_frames(c, v, levelsup, lv->desc, lv->n, F, N, fv)) return rc;
    int per_sm = 0, n_sm = 0;
    ORBX_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, loopver_pair_kernel, kLT, 0));
    ORBX_CUDA(c, cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, c->device));
    if (per_sm < 1) return fail(c, ORBX_ERR_CUDA, "the loop verification kernel does not fit an SM");
    lv->grid_max = per_sm * n_sm;
    if (int rc = lv->scratch.reserve(c, (size_t)lv->grid_max * cta_bytes(N))) return rc;
    guard.lv = nullptr;
    *out = lv;
    return ORBX_OK;
  }

  int orbx_loopver_verify(orbx_ctx *c, const orbx_loopver *lv_, int64_t q_lo, int64_t nq, const orbx_loopver_params *prm, const orbx_loopver_io *io)
  {
    if (!c || !lv_ || !prm || !io) return ORBX_ERR_INVALID_ARG;
    orbx_loopver *lv = const_cast<orbx_loopver *>(lv_);
    if (lv->ctx != c || lv->device != c->device) return fail(c, ORBX_ERR_INVALID_ARG, "the verifier belongs to another context");
    if (std::isnan(prm->ratio)) return fail(c, ORBX_ERR_INVALID_ARG, "ratio is NaN");
    if (!(prm->probability > 0.0 && prm->probability < 1.0)) return fail(c, ORBX_ERR_INVALID_ARG, "probability outside (0, 1)");
    if (prm->min_inliers < 3) return fail(c, ORBX_ERR_INVALID_ARG, "min_inliers < 3");
    if (prm->max_iterations < 1) return fail(c, ORBX_ERR_INVALID_ARG, "max_iterations < 1");
    if (io->top_k < 1) return fail(c, ORBX_ERR_INVALID_ARG, "top_k < 1");
    if (q_lo < 0 || nq < 0 || q_lo + nq > lv->F) return fail(c, ORBX_ERR_INVALID_ARG, "queries outside [0, n_frames)");
    if (nq > 0 && !io->cand_frame) return fail(c, ORBX_ERR_INVALID_ARG, "no candidate table");
    const size_t n_pairs = (size_t)nq * io->top_k;
    if (!io->on_device)
      for (size_t i = 0; i < n_pairs; ++i)
        if (io->cand_frame[i] < -1 || io->cand_frame[i] >= lv->F) return fail(c, ORBX_ERR_INVALID_ARG, "a candidate lies outside [-1, n_frames)");
    if (nq == 0) return ORBX_OK;
    ORBX_CUDA(c, cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    const int N = lv->N;
    const std::vector<int32_t> iters = iteration_table(N, prm);
    // staging: iteration table, loop keys, then (host io) the table and the outputs
    const size_t o_it = 0, o_key = o_it + up16(((size_t)N + 1) * 4), o_tab = o_key + up16((size_t)nq * 8);
    const size_t o_i32 = o_tab + (io->on_device ? 0 : up16(n_pairs * 4)), n_i32 = 7;
    const size_t o_T = o_i32 + n_i32 * up16(n_pairs * 4), o_match = o_T + (io->on_device ? 0 : up16(n_pairs * 96));
    const size_t o_lf = o_match + (io->on_device || !io->match ? 0 : up16(n_pairs * (size_t)N * 4)), total = o_lf + up16((size_t)nq * 4);
    if (int rc = lv->staging.reserve(c, total)) return rc;
    uint8_t *st = lv->staging.p;
    ORBX_CUDA(c, cudaMemcpyAsync(st + o_it, iters.data(), iters.size() * 4, cudaMemcpyHostToDevice, s));
    LvArgs a{};
    a.kp = lv->kp, a.desc = lv->desc, a.depth = lv->depth, a.n = lv->n;
    a.fv_nodes = lv->fv_nodes, a.fv_start = lv->fv_start, a.fv_feats = lv->fv_feats, a.n_fv = lv->n_fv;
    a.F = lv->F, a.N = N;
    a.fx = c->cfg.fx, a.fy = c->cfg.fy, a.cx = c->cfg.cx, a.cy = c->cfg.cy;
    for (int l = 0; l < kMaxLevels; ++l)
    {
      const float sf = l < (int)c->levels.size() ? c->levels[(size_t)l].sf : 1.f;
      const float s2 = sf * sf; // mvLevelSigma2: the float square of the level scale factor
      a.thr[l] = 9.210 * (double)s2;
    }
    a.iters = (const int *)(st + o_it);
    a.top_k = io->top_k, a.n_queries = (int)nq, a.q_lo = q_lo;
    a.ratio = prm->ratio, a.min_matches = prm->min_matches, a.min_inliers = prm->min_inliers;
    a.seed_key = splitmix64(prm->seed);
    a.scratch = lv->scratch.p, a.cta_bytes = cta_bytes(N);
    a.loop_key = (unsigned long long *)(st + o_key);
    int *i32[7];
    int *const user[7] = {io->n_bow, io->n_matches, io->n_corr, io->n_iters, io->hypothesis, io->n_inliers, io->accepted};
    for (int j = 0; j < 7; ++j) i32[j] = io->on_device ? user[j] : (user[j] ? (int *)(st + o_i32 + j * up16(n_pairs * 4)) : nullptr);
    a.n_bow = i32[0], a.n_matches = i32[1], a.n_corr = i32[2], a.n_iters = i32[3], a.hypothesis = i32[4], a.n_inliers = i32[5], a.accepted = i32[6];
    int *loop_frame = io->loop_frame;
    if (io->on_device)
      a.table = io->cand_frame, a.T = io->T, a.match = io->match;
    else
    {
      ORBX_CUDA(c, cudaMemcpyAsync(st + o_tab, io->cand_frame, n_pairs * 4, cudaMemcpyHostToDevice, s));
      a.table = (const int *)(st + o_tab);
      a.T = io->T ? (double *)(st + o_T) : nullptr;
      a.match = io->match ? (int *)(st + o_match) : nullptr;
      loop_frame = io->loop_frame ? (int *)(st + o_lf) : nullptr;
    }
    if (!loop_frame) a.loop_key = nullptr;
    if (a.loop_key) ORBX_CUDA(c, cudaMemsetAsync(a.loop_key, 0xff, (size_t)nq * 8, s));
    const int grid = (int)std::min<size_t>(n_pairs, (size_t)lv->grid_max);
    loopver_pair_kernel<<<grid, kLT, 0, s>>>(a);
    ++c->launches;
    if (loop_frame)
    {
      loopver_loop_frame_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(a.table, a.top_k, (int)nq, a.loop_key, loop_frame);
      ++c->launches;
    }
    ORBX_CUDA(c, cudaGetLastError());
    if (io->on_device) return ORBX_OK;
    auto back = [&](void *dst, const void *src, size_t bytes) -> cudaError_t {
      return dst ? cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s) : cudaSuccess;
    };
    for (int j = 0; j < 7; ++j) ORBX_CUDA(c, back(user[j], i32[j], n_pairs * 4));
    ORBX_CUDA(c, back(io->T, a.T, n_pairs * 96));
    ORBX_CUDA(c, back(io->match, a.match, n_pairs * (size_t)N * 4));
    ORBX_CUDA(c, back(io->loop_frame, loop_frame, (size_t)nq * 4));
    ORBX_CUDA(c, cudaStreamSynchronize(s));
    return ORBX_OK;
  }

} // extern "C"
