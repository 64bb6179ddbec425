/* loopver_oracle.c -- plain-C restatement of loop verification (orbx_loopver_*, include/orbx.h): for every (query, candidate)
 * pair of a table, ORBMatcher::searchByBow with the candidate as the keyframe (oracle_search_by_bow), the kept rows,
 * oracle_verify_angle, the correspondences with two depths, and Sim3Solver-style RANSAC with Horn's closed form at a fixed
 * scale -- one hypothesis after another, as ORB-SLAM2's Sim3Solver::iterate runs them.  FeatureVectors come from
 * oracle_bow_transform (oracle/orb_oracle.c, compiled into the same library).  Compiled with -ffp-contract=off so that every
 * double operation rounds once.
 *
 *   oracle_loopver(v, levelsup, F, N, kps, desc, depth, n,      frame f: kps / desc / depth + f * N, n[f] features
 *                  fx, fy, cx, cy, sf, n_levels,                camera and level scale factors
 *                  q_lo, n_queries, table, top_k,               query i is frame q_lo + i, its candidates table[i][0 .. top_k)
 *                  ratio, min_matches, min_inliers, max_iterations, probability, seed,
 *                  counts, T, match, loop_frame)                [nq][top_k][7]: n_bow n_matches n_corr n_iters hypothesis
 *                                                               n_inliers accepted; [nq][top_k][12]; [nq][top_k][N]; [nq]
 * The sums follow the rule of include/orbx.h: 32 slot partials, then the tree; the sweep bound is ORBX_LOOPVER_JACOBI_SWEEPS.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "orb_oracle.h"

#define JACOBI_SWEEPS 16 /* ORBX_LOOPVER_JACOBI_SWEEPS */
#define GOLDEN 0x9E3779B97F4A7C15ull

static uint64_t splitmix64(uint64_t x)
{
  uint64_t z = x + GOLDEN;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

typedef struct
{
  double c[3], q[3];
  double thr_c, thr_q;
  float uc, vc, uq, vq;
} corr_t;

/* sum of x[0 .. m) with slots slot[k]: 32 partials, then p_l += p_{l+s} for s = 16 .. 1 */
static double slot_sum(const double *x, const int *slot, int m)
{
  double p[32];
  for (int l = 0; l < 32; ++l) p[l] = 0.0;
  for (int k = 0; k < m; ++k) p[slot[k] % 32] += x[k];
  for (int s = 16; s; s >>= 1)
    for (int l = 0; l < s; ++l) p[l] += p[l + s];
  return p[0];
}

/* Horn on the listed points (pts[k], slot[k]); T = R row-major, t, then the inverse's translation -R^T t */
static void horn(const corr_t *const *pts, const int *slot, int m, double *T)
{
  double *x = malloc(sizeof(double) * (size_t)m);
  double cc[3], cq[3], M[9];
  for (int d = 0; d < 3; ++d)
  {
    for (int k = 0; k < m; ++k) x[k] = pts[k]->c[d];
    cc[d] = slot_sum(x, slot, m) / (double)m;
    for (int k = 0; k < m; ++k) x[k] = pts[k]->q[d];
    cq[d] = slot_sum(x, slot, m) / (double)m;
  }
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b)
    {
      for (int k = 0; k < m; ++k) x[k] = (pts[k]->c[a] - cc[a]) * (pts[k]->q[b] - cq[b]);
      M[3 * a + b] = slot_sum(x, slot, m);
    }
  free(x);
  /* N (Sim3Solver::ComputeSim3: M = Pr2 * Pr1^T with the candidate as set 2) */
  double A[4][4], V[4][4];
  A[0][0] = M[0] + M[4] + M[8];
  A[0][1] = M[5] - M[7];
  A[0][2] = M[6] - M[2];
  A[0][3] = M[1] - M[3];
  A[1][1] = M[0] - M[4] - M[8];
  A[1][2] = M[1] + M[3];
  A[1][3] = M[6] + M[2];
  A[2][2] = -M[0] + M[4] - M[8];
  A[2][3] = M[5] + M[7];
  A[3][3] = -M[0] - M[4] + M[8];
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j)
    {
      if (j < i) A[i][j] = A[j][i];
      V[i][j] = i == j ? 1.0 : 0.0;
    }
  /* cyclic Jacobi */
  for (int sweep = 0; sweep < JACOBI_SWEEPS; ++sweep)
  {
    if (A[0][1] == 0 && A[0][2] == 0 && A[0][3] == 0 && A[1][2] == 0 && A[1][3] == 0 && A[2][3] == 0) break;
    for (int p = 0; p < 3; ++p)
      for (int q = p + 1; q < 4; ++q)
      {
        if (A[p][q] == 0) continue;
        const double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
        double t = 1.0 / (fabs(theta) + sqrt(theta * theta + 1.0));
        if (theta < 0) t = -t;
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 4; ++k)
        {
          const double akp = A[k][p], akq = A[k][q];
          A[k][p] = c * akp - s * akq;
          A[k][q] = s * akp + c * akq;
        }
        for (int k = 0; k < 4; ++k)
        {
          const double apk = A[p][k], aqk = A[q][k];
          A[p][k] = c * apk - s * aqk;
          A[q][k] = s * apk + c * aqk;
        }
        A[p][q] = A[q][p] = 0;
        for (int k = 0; k < 4; ++k)
        {
          const double vkp = V[k][p], vkq = V[k][q];
          V[k][p] = c * vkp - s * vkq;
          V[k][q] = s * vkp + c * vkq;
        }
      }
  }
  int mx = 0;
  for (int i = 1; i < 4; ++i)
    if (A[i][i] > A[mx][mx]) mx = i;
  const double w = V[0][mx], x_ = V[1][mx], y = V[2][mx], z = V[3][mx];
  const double ww = w * w, xx = x_ * x_, yy = y * y, zz = z * z, n2 = ww + xx + yy + zz;
  T[0] = (ww + xx - yy - zz) / n2;
  T[1] = 2.0 * (x_ * y - w * z) / n2;
  T[2] = 2.0 * (x_ * z + w * y) / n2;
  T[3] = 2.0 * (x_ * y + w * z) / n2;
  T[4] = (ww - xx + yy - zz) / n2;
  T[5] = 2.0 * (y * z - w * x_) / n2;
  T[6] = 2.0 * (x_ * z - w * y) / n2;
  T[7] = 2.0 * (y * z + w * x_) / n2;
  T[8] = (ww - xx - yy + zz) / n2;
  for (int r = 0; r < 3; ++r) T[9 + r] = cq[r] - (T[3 * r] * cc[0] + T[3 * r + 1] * cc[1] + T[3 * r + 2] * cc[2]);
  for (int r = 0; r < 3; ++r) T[12 + r] = -(T[r] * T[9] + T[3 + r] * T[10] + T[6 + r] * T[11]);
}

static int is_inlier(const corr_t *k, const double *T, double fx, double fy, double cx, double cy)
{
  double Y[3], Z[3];
  for (int r = 0; r < 3; ++r)
  {
    Y[r] = T[3 * r] * k->c[0] + T[3 * r + 1] * k->c[1] + T[3 * r + 2] * k->c[2] + T[9 + r];
    Z[r] = T[r] * k->q[0] + T[3 + r] * k->q[1] + T[6 + r] * k->q[2] + T[12 + r];
  }
  const double iy = 1.0 / Y[2], iz = 1.0 / Z[2];
  const double du1 = (double)k->uq - (fx * (Y[0] * iy) + cx), dv1 = (double)k->vq - (fy * (Y[1] * iy) + cy);
  const double du2 = (double)k->uc - (fx * (Z[0] * iz) + cx), dv2 = (double)k->vc - (fy * (Z[1] * iz) + cy);
  return du1 * du1 + dv1 * dv1 < k->thr_q && du2 * du2 + dv2 * dv2 < k->thr_c;
}

int oracle_loopver(const oracle_vocab *v, int levelsup, int32_t F, int32_t N, const oracle_keypoint *kps, const uint8_t *desc, const double *depth,
                   const int32_t *n, float fx_, float fy_, float cx_, float cy_, const float *sf, int n_levels, int64_t q_lo, int32_t n_queries,
                   const int32_t *table, int32_t top_k, float ratio, int32_t min_matches, int32_t min_inliers, int32_t max_iterations,
                   double probability, uint64_t seed, int32_t *counts, double *T_out, int32_t *match, int32_t *loop_frame)
{
  const double fx = fx_, fy = fy_, cx = cx_, cy = cy_;
  const size_t NN = (size_t)N;
  /* the FeatureVectors of the frames the table uses */
  int32_t *fv_nodes = malloc(sizeof(int32_t) * (size_t)F * (NN + 1)), *fv_start = malloc(sizeof(int32_t) * (size_t)F * (NN + 2));
  int32_t *fv_feats = malloc(sizeof(int32_t) * (size_t)F * (NN + 1)), *n_fv = malloc(sizeof(int32_t) * (size_t)F);
  int32_t *bids = malloc(sizeof(int32_t) * (NN + 1));
  double *bvals = malloc(sizeof(double) * (NN + 1));
  /* the frames the queries and their candidates use */
  uint8_t *need = calloc((size_t)F, 1);
  for (int32_t qi = 0; qi < n_queries; ++qi)
  {
    need[q_lo + qi] = 1;
    for (int32_t sl = 0; sl < top_k; ++sl)
      if (table[(size_t)qi * top_k + sl] >= 0 && table[(size_t)qi * top_k + sl] < F) need[table[(size_t)qi * top_k + sl]] = 1;
  }
  for (int f = 0; f < F; ++f)
    if (need[f])
      oracle_bow_transform(v, desc + (size_t)f * NN * 32, n[f], levelsup, bids, bvals, fv_nodes + (size_t)f * (NN + 1), fv_start + (size_t)f * (NN + 2),
                         fv_feats + (size_t)f * (NN + 1), &n_fv[f]);
  free(bids);
  free(bvals);
  free(need);
  /* SetRansacParameters for every n_corr */
  int32_t *iters = calloc(NN + 1, sizeof(int32_t));
  for (int m = min_inliers; m <= N; ++m)
  {
    double it = 1.0;
    if (m != min_inliers)
    {
      const float eps = (float)min_inliers / (float)m;
      it = ceil(log(1.0 - probability) / log(1.0 - pow((double)eps, 3.0)));
    }
    iters[m] = it < 1.0 ? 1 : it > (double)max_iterations ? max_iterations : (int32_t)it;
  }
  int32_t *ki = malloc(sizeof(int32_t) * (NN + 1)), *bi = malloc(sizeof(int32_t) * (NN + 1)), *bd = malloc(sizeof(int32_t) * (NN + 1));
  int32_t *nc = malloc(sizeof(int32_t) * (NN + 1));
  float *ra = malloc(sizeof(float) * (NN + 1)), *di = malloc(sizeof(float) * (NN + 1));
  int32_t *mq = malloc(sizeof(int32_t) * (NN + 1)), *mc = malloc(sizeof(int32_t) * (NN + 1)), *slot = malloc(sizeof(int32_t) * (NN + 1));
  corr_t *corr = malloc(sizeof(corr_t) * (NN + 1));
  const corr_t **pts = malloc(sizeof(corr_t *) * (NN + 1));
  double thr[64];
  for (int l = 0; l < 64; ++l)
  {
    const float s = l < n_levels ? sf[l] : 1.f, s2 = s * s;
    thr[l] = 9.210 * (double)s2;
  }
  const uint64_t seed_key = splitmix64(seed);
  for (int32_t qi = 0; qi < n_queries; ++qi)
  {
    const int qf = (int)(q_lo + qi);
    uint64_t best_key = ~0ull;
    for (int32_t sl = 0; sl < top_k; ++sl)
    {
      const size_t o = (size_t)qi * top_k + sl;
      int32_t *cnt = counts + 7 * o;
      double *T = T_out + 12 * o;
      int32_t *mrow = match + o * NN;
      for (int j = 0; j < 7; ++j) cnt[j] = 0;
      cnt[4] = -1;
      for (int j = 0; j < 12; ++j) T[j] = 0.0;
      for (int j = 0; j < N; ++j) mrow[j] = -1;
      const int cf = table[o];
      if (cf < 0 || cf >= F) continue;
      const oracle_keypoint *kq = kps + (size_t)qf * NN, *kc = kps + (size_t)cf * NN;
      const double *dq = depth + (size_t)qf * NN, *dc = depth + (size_t)cf * NN;
      /* searchByBow(pFrame = query, pKframe = candidate, bLoop): the rows, then the kept ones */
      const int rows = oracle_search_by_bow(fv_nodes + (size_t)qf * (NN + 1), fv_start + (size_t)qf * (NN + 2), fv_feats + (size_t)qf * (NN + 1), n_fv[qf],
                                            desc + (size_t)qf * NN * 32, NULL, fv_nodes + (size_t)cf * (NN + 1), fv_start + (size_t)cf * (NN + 2),
                                            fv_feats + (size_t)cf * (NN + 1), n_fv[cf], desc + (size_t)cf * NN * 32, NULL, ki, bi, bd, ra, nc);
      int nb = 0;
      for (int r = 0; r < rows; ++r)
        if (bd[r] <= 50 && !(ra[r] > ratio))
        {
          mq[nb] = bi[r];
          mc[nb] = ki[r];
          di[nb] = (float)bd[r];
          ++nb;
        }
      const int nm = oracle_verify_angle(nb, mq, mc, di, kq, kc);
      cnt[0] = nb;
      cnt[1] = nm;
      for (int i = 0; i < nm; ++i) mrow[mc[i]] = mq[i];
      if (nm < min_matches) continue;
      /* correspondences */
      int m = 0;
      for (int i = 0; i < nm; ++i)
      {
        const double zc = dc[mc[i]], zq = dq[mq[i]];
        if (!(zc > 0) || !(zq > 0)) continue;
        const oracle_keypoint *pc = &kc[mc[i]], *pq = &kq[mq[i]];
        corr_t *k = &corr[m++];
        k->c[0] = ((double)pc->x - cx) * zc / fx, k->c[1] = ((double)pc->y - cy) * zc / fy, k->c[2] = zc;
        k->q[0] = ((double)pq->x - cx) * zq / fx, k->q[1] = ((double)pq->y - cy) * zq / fy, k->q[2] = zq;
        k->thr_c = thr[pc->octave < 0 ? 0 : pc->octave > 63 ? 63 : pc->octave];
        k->thr_q = thr[pq->octave < 0 ? 0 : pq->octave > 63 ? 63 : pq->octave];
        k->uc = pc->x, k->vc = pc->y, k->uq = pq->x, k->vq = pq->y;
      }
      cnt[2] = m;
      /* Sim3Solver::iterate, one hypothesis after another */
      const int nit = iters[m];
      const uint64_t K = splitmix64(splitmix64(seed_key + (uint64_t)qf + 1) + (uint64_t)cf + 1);
      int best_h = -1, best_n = 0, acc = 0;
      double bestT[15], Th[15];
      int *avail = malloc(sizeof(int) * (size_t)(m > 0 ? m : 1));
      for (int h = 0; h < nit; ++h)
      {
        for (int i = 0; i < m; ++i) avail[i] = i;
        const corr_t *smp[3];
        const int sslot[3] = {0, 1, 2};
        for (int j = 0; j < 3; ++j)
        {
          const int r = (int)(splitmix64(K ^ ((uint64_t)(3 * h + j) * GOLDEN)) % (uint64_t)(m - j));
          smp[j] = &corr[avail[r]];
          avail[r] = avail[m - 1 - j];
        }
        horn(smp, sslot, 3, Th);
        int ninl = 0;
        for (int i = 0; i < m; ++i) ninl += is_inlier(&corr[i], Th, fx, fy, cx, cy);
        if (ninl >= best_n)
        {
          best_n = ninl, best_h = h;
          memcpy(bestT, Th, sizeof(Th));
          if (ninl > min_inliers)
          {
            acc = 1;
            break;
          }
        }
      }
      free(avail);
      cnt[3] = acc ? best_h + 1 : nit;
      cnt[4] = best_h;
      cnt[5] = best_h >= 0 ? best_n : 0;
      cnt[6] = acc;
      if (best_h < 0) continue;
      /* the refit over the inliers of the reported hypothesis (slot = correspondence index) */
      double Tf[15];
      if (best_n >= 3)
      {
        int k = 0;
        for (int i = 0; i < m; ++i)
          if (is_inlier(&corr[i], bestT, fx, fy, cx, cy)) pts[k] = &corr[i], slot[k] = i, ++k;
        horn(pts, slot, k, Tf);
      }
      else
        memcpy(Tf, bestT, sizeof(Tf));
      memcpy(T, Tf, 12 * sizeof(double));
      if (acc)
      {
        const uint64_t key = ((uint64_t)(best_h / 5) << 32) | (uint32_t)sl;
        if (key < best_key) best_key = key;
      }
    }
    loop_frame[qi] = best_key == ~0ull ? -1 : table[(size_t)qi * top_k + (uint32_t)(best_key & 0xffffffffu)];
  }
  free(fv_nodes), free(fv_start), free(fv_feats), free(n_fv), free(iters);
  free(ki), free(bi), free(bd), free(nc), free(ra), free(di), free(mq), free(mc), free(slot), free(corr), free(pts);
  return 0;
}
