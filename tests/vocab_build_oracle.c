/*
 * vocab_build_oracle.c -- plain-C restatement of the vocabulary construction (orbx_vocab_build), the sequential checker
 * the CUDA build is tested against bit for bit.  TEST INFRASTRUCTURE ONLY: tests/vocab_build_restatement.py compiles it
 * with the host C compiler into a temporary directory and loads it through ctypes.
 */
#include <limits.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static int desc_distance(const uint8_t *a, const uint8_t *b) {
  int d = 0;
  for (int i = 0; i < 32; ++i) d += __builtin_popcount((unsigned)(a[i] ^ b[i]));
  return d;
}

/* ---------------------------------------------------------------------------------------------------------------
 * Vocabulary construction.  PARITY UNPINNED, as the transform of oracle/orb_oracle.c: a restatement of DBoW2 / DBoW3
 * TemplatedVocabulary::create -> HKmeansStep (hierarchical k-means, DBoW's recursion order), initiateClustersKMpp
 * (k-means++ seeding, here with integer distances and a counter-based generator instead of rand()), FORB::meanValue
 * (bitwise majority), createWords (word ids = leaves in node id order) and setNodeWeights (TF_IDF).  The rules are the
 * ones include/orbx.h states for orbx_vocab_build; the CUDA build is tested against this function bit for bit.
 * --------------------------------------------------------------------------------------------------------------- */
#include "../include/orbx.h" /* ORBX_VOCAB_MAX_ITERS: the checker and the kernels stop at the same pass */

static uint64_t vb_splitmix64(uint64_t x) {
  uint64_t z = x + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

typedef struct vb_state {
  int k, L, cap, n_nodes, failed;
  const uint8_t *d;  /* training descriptors, compacted: [n][32] */
  int32_t *parent, *first_child, *n_child;
  uint8_t *desc, *capped;
  int32_t *iters, *leaf_of, n_capped;
  int32_t *root_picks; /* optional [k]: the root's k-means++ picks, positions in its segment */
} vb_state;

static void vb_step(vb_state *s, int node, uint64_t key, const int32_t *idx, int n, int level) {
  const int k = s->k;
  uint8_t *cent = (uint8_t *)malloc((size_t)k * 32);
  int32_t *asg = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
  int kk = 0, capped = 0;
  if (n <= k) { /* one cluster per descriptor */
    for (int i = 0; i < n; ++i) {
      memcpy(cent + 32 * (size_t)i, s->d + 32 * (size_t)idx[i], 32);
      asg[i] = i;
    }
    kk = n;
  } else {
    /* initiateClustersKMpp with integer distances: S = sum of min_dist, cut = 1 + r_j % S, first i whose running sum
     * reaches cut; S == 0 stops the seeding with fewer than k centres */
    uint32_t *md = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)n);
    int pick = (int)(vb_splitmix64(key) % (uint64_t)n);
    for (;;) {
      memcpy(cent + 32 * (size_t)kk, s->d + 32 * (size_t)idx[pick], 32);
      if (node == 0 && s->root_picks) s->root_picks[kk] = pick;
      ++kk;
      if (kk == k) break;
      uint64_t S = 0;
      for (int i = 0; i < n; ++i) {
        const uint32_t dd = (uint32_t)desc_distance(s->d + 32 * (size_t)idx[i], cent + 32 * (size_t)(kk - 1));
        if (kk == 1 || dd < md[i]) md[i] = dd;
        S += md[i];
      }
      if (S == 0) break;
      const uint64_t cut = 1 + vb_splitmix64(key ^ ((uint64_t)kk * 0x9E3779B97F4A7C15ull)) % S;
      uint64_t run = 0;
      for (pick = 0; pick < n; ++pick) {
        run += md[pick];
        if (run >= cut) break;
      }
    }
    free(md);
    /* Lloyd iterations until no assignment changes (at most ORBX_VOCAB_MAX_ITERS assignment passes) */
    uint32_t *cnt = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)kk * 257);
    int pass = 0;
    for (;;) {
      ++pass;
      int changed = pass == 1;
      for (int i = 0; i < n; ++i) {
        const uint8_t *x = s->d + 32 * (size_t)idx[i];
        int best = desc_distance(x, cent), bc = 0;
        for (int c = 1; c < kk; ++c) {
          const int dd = desc_distance(x, cent + 32 * (size_t)c);
          if (dd < best) {
            best = dd;
            bc = c;
          }
        }
        if (pass > 1 && asg[i] != bc) changed = 1;
        asg[i] = bc;
      }
      if (!changed) break;
      if (pass == ORBX_VOCAB_MAX_ITERS) {
        capped = 1;
        break;
      }
      /* FORB::meanValue: bit b set iff at least ceil(m/2) of the m members have it; an empty cluster keeps its centre */
      memset(cnt, 0, sizeof(uint32_t) * (size_t)kk * 257);
      for (int i = 0; i < n; ++i) {
        const uint8_t *x = s->d + 32 * (size_t)idx[i];
        uint32_t *cc = cnt + 257 * (size_t)asg[i];
        ++cc[256];
        for (int b = 0; b < 256; ++b) cc[b] += (x[b >> 3] >> (b & 7)) & 1;
      }
      for (int c = 0; c < kk; ++c) {
        const uint32_t *cc = cnt + 257 * (size_t)c, m = cc[256];
        if (m == 0) continue;
        uint8_t *y = cent + 32 * (size_t)c;
        memset(y, 0, 32);
        for (int b = 0; b < 256; ++b)
          if (cc[b] >= (m + 1) / 2) y[b >> 3] |= (uint8_t)(1u << (b & 7));
      }
    }
    free(cnt);
    if (pass > s->iters[level - 1]) s->iters[level - 1] = pass;
    s->n_capped += capped;
  }
  s->capped[node] = (uint8_t)capped;
  /* children of the node get consecutive ids, in cluster order */
  const int first = s->n_nodes;
  if (first + kk > s->cap) {
    s->failed = 1;
    free(cent);
    free(asg);
    return;
  }
  for (int c = 0; c < kk; ++c) {
    const int id = s->n_nodes++;
    s->parent[id] = node;
    s->first_child[id] = -1;
    s->n_child[id] = 0;
    s->capped[id] = 0;
    memcpy(s->desc + 32 * (size_t)id, cent + 32 * (size_t)c, 32);
  }
  s->first_child[node] = first;
  s->n_child[node] = kk;
  free(cent);
  /* then the children, depth first; a child's members keep their order in the node's list */
  int32_t *mem = (int32_t *)malloc(sizeof(int32_t) * (size_t)(n > 0 ? n : 1));
  for (int c = 0; c < kk && !s->failed; ++c) {
    int m = 0;
    for (int i = 0; i < n; ++i)
      if (asg[i] == c) mem[m++] = idx[i];
    if (level < s->L && m > 1)
      vb_step(s, first + c, vb_splitmix64(key + (uint64_t)c + 1), mem, m, level + 1);
    else
      for (int i = 0; i < m; ++i) s->leaf_of[mem[i]] = first + c;
  }
  free(mem);
  free(asg);
}

/* DBoW2/DBoW3 TemplatedVocabulary::create on the descriptors desc[f][i] (i < n_kps[f]) of n_frames frame rows of `stride`
 * descriptors each, under the rules include/orbx.h states for orbx_vocab_build.  Outputs in the text format's record order
 * (record i = node i + 1): parent, is_leaf, node_desc [cap][32], weight.  iters[L]: most assignment passes of a k-means
 * node per level; *n_capped: nodes stopped by ORBX_VOCAB_MAX_ITERS.  Optional (NULL): leaf_of[n_frames * stride] = node
 * id each training descriptor was trained into (-1 for padding), node_capped[n_records + 1] per node id, root_picks[k] =
 * the root's k-means++ picks as positions among the training descriptors in frame order (-1 past the last pick, and all -1
 * when the root has n <= k descriptors).  Returns the
 * number of records, or -1 (bad arguments, no descriptors, more than cap_records records). */
int oracle_vocab_build(const uint8_t *desc, const int32_t *n_kps, int n_frames, int stride, int k, int L, uint64_t seed,
                       int cap_records, int32_t *parent, uint8_t *is_leaf, uint8_t *node_desc, double *weight,
                       int32_t *iters, int32_t *n_capped, int32_t *leaf_of, uint8_t *node_capped, int32_t *root_picks) {
  if (k < 2 || L < 1 || n_frames < 1 || stride < 1 || cap_records < 1) return -1;
  int n = 0;
  for (int f = 0; f < n_frames; ++f) {
    if (n_kps[f] < 0 || n_kps[f] > stride) return -1;
    n += n_kps[f];
  }
  if (n == 0) return -1;
  uint8_t *d = (uint8_t *)malloc((size_t)n * 32);
  int32_t *idx = (int32_t *)malloc(sizeof(int32_t) * (size_t)n), *pos = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
  for (int f = 0, o = 0; f < n_frames; ++f)
    for (int i = 0; i < n_kps[f]; ++i, ++o) {
      memcpy(d + 32 * (size_t)o, desc + 32 * ((size_t)f * stride + i), 32);
      idx[o] = o;
      pos[o] = f * stride + i;
    }
  const int cap = cap_records + 1;
  vb_state s;
  memset(&s, 0, sizeof(s));
  s.k = k, s.L = L, s.cap = cap, s.n_nodes = 1, s.d = d;
  s.parent = (int32_t *)malloc(sizeof(int32_t) * (size_t)cap);
  s.first_child = (int32_t *)malloc(sizeof(int32_t) * (size_t)cap);
  s.n_child = (int32_t *)malloc(sizeof(int32_t) * (size_t)cap);
  s.desc = (uint8_t *)calloc((size_t)cap, 32);
  s.capped = (uint8_t *)calloc((size_t)cap, 1);
  s.iters = iters;
  s.root_picks = root_picks;
  if (root_picks)
    for (int c = 0; c < k; ++c) root_picks[c] = -1;
  s.leaf_of = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
  for (int l = 0; l < L; ++l) iters[l] = 0;
  s.parent[0] = -1, s.first_child[0] = -1, s.n_child[0] = 0;
  vb_step(&s, 0, vb_splitmix64(seed), idx, n, 1);
  int rc = -1;
  if (!s.failed) {
    const int nn = s.n_nodes;
    /* createWords: word ids to the leaves in node id order; setNodeWeights (TF_IDF): N_i = frames with at least one
     * descriptor whose DESCENT ends at word i, weight = log(N / N_i), N = n_frames, 0 when N_i = 0 */
    int32_t *word = (int32_t *)malloc(sizeof(int32_t) * (size_t)nn);
    int nw = 0;
    for (int i = 0; i < nn; ++i) word[i] = (i > 0 && s.n_child[i] == 0) ? nw++ : -1;
    int32_t *ni = (int32_t *)calloc((size_t)(nw > 0 ? nw : 1), sizeof(int32_t)), *stamp = (int32_t *)malloc(sizeof(int32_t) * (size_t)(nw > 0 ? nw : 1));
    for (int w = 0; w < nw; ++w) stamp[w] = -1;
    for (int f = 0; f < n_frames; ++f)
      for (int i = 0; i < n_kps[f]; ++i) {
        const uint8_t *x = desc + 32 * ((size_t)f * stride + i);
        int node = 0;
        while (s.n_child[node] > 0) {
          const int c0 = s.first_child[node];
          int best = INT_MAX, bc = c0;
          for (int c = c0; c < c0 + s.n_child[node]; ++c) {
            const int dd = desc_distance(x, s.desc + 32 * (size_t)c);
            if (dd < best) {
              best = dd;
              bc = c;
            }
          }
          node = bc;
        }
        const int w = word[node];
        if (stamp[w] != f) {
          stamp[w] = f;
          ++ni[w];
        }
      }
    for (int i = 1; i < nn; ++i) {
      parent[i - 1] = s.parent[i];
      is_leaf[i - 1] = s.n_child[i] == 0;
      memcpy(node_desc + 32 * (size_t)(i - 1), s.desc + 32 * (size_t)i, 32);
      weight[i - 1] = (word[i] >= 0 && ni[word[i]] > 0) ? log((double)n_frames / (double)ni[word[i]]) : 0.0;
    }
    if (n_capped) *n_capped = s.n_capped;
    if (node_capped) memcpy(node_capped, s.capped, (size_t)nn);
    if (leaf_of) {
      for (size_t t = 0; t < (size_t)n_frames * stride; ++t) leaf_of[t] = -1;
      for (int o = 0; o < n; ++o) leaf_of[pos[o]] = s.leaf_of[o];
    }
    free(word);
    free(ni);
    free(stamp);
    rc = nn - 1;
  }
  free(s.parent);
  free(s.first_child);
  free(s.n_child);
  free(s.desc);
  free(s.capped);
  free(s.leaf_of);
  free(d);
  free(idx);
  free(pos);
  return rc;
}
