// orbx_kernels.cu -- hand-written sm_100a kernels of the ORB front-end.
//
// One kernel per stage of the reference's CPU path (citations relative to /root/reference/src/ORB_SLAM2/):
//   pyramid_level0_kernel / pyramid_levels_kernel  ORBExtractor::initPyramid  src/ORBExtractor.cc:304-319  (cv::resize + cv::GaussianBlur)
//   fast_cells_kernel    ORBExtractor::extractFast, FAST part  src/ORBExtractor.cc:346-375  (cv::FAST + threshold fallback)
//   quadtree_kernel      Quadtree::split / nodes2kpoints       src/ORBExtractor.cc:19-192,376-386
//   orient_brief_kernel  getGrayCentroid + computeBRIEF        src/ORBExtractor.cc:397-487,534-540
//   stereo_kernel        ORBMatcher::searchByStereo            src/ORBMatcher.cc:18-81,841-1011
//   rgbd_kernel          Frame::Frame (RGB-D)                  src/Frame.cc:125-159
// All arithmetic that decides a result bit is integer, or IEEE float/double with explicit round-to-nearest
// intrinsics (no FMA contraction), so results equal the CPU path bit for bit.
#include "orbx_device.cuh"
#include <cstdio>

namespace orbx
{

// ------------------------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int refl101(int i, int n)
{
  // BORDER_REFLECT_101 for an overshoot of at most 3 pixels on images of at least 4 pixels
  if (i < 0) i = -i;
  if (i >= n) i = 2 * (n - 1) - i;
  return i;
}

__device__ __forceinline__ const uint8_t *input_image(const Params &p, int img)
{
  if (p.stereo) return ((img & 1) ? p.in_right : p.in_left) + (size_t)(img >> 1) * p.in_frame_stride;
  return p.in_left + (size_t)img * p.in_frame_stride;
}

__device__ __forceinline__ int warp_sum(int v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
  return v;
}

// shared-memory accesses of the compaction lists by 32-bit shared address: one LDS / STS each, no generic-pointer arithmetic
__device__ __forceinline__ void sts_u16_if(uint32_t addr, uint32_t v, bool pred)
{
  asm volatile("{\n .reg .pred p;\n setp.ne.u32 p, %2, 0;\n @p st.shared.u16 [%0], %1;\n}" ::"r"(addr), "h"((unsigned short)v), "r"((uint32_t)pred) : "memory");
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr)
{
  unsigned short v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr) : "memory");
  return v;
}

// ---- TMA (cp.async.bulk.tensor) + mbarrier helpers -------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// one 3-D box {x .. x + boxW, y .. y + boxH, z} of a byte tensor -> shared memory, completion on an mbarrier
__device__ __forceinline__ void tma_load_3d(void *smem_dst, const CUtensorMap *map, int x, int y, int z, uint64_t *bar)
{
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(smem_u32(smem_dst)),
               "l"(map), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr)
{
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}

// ------------------------------------------------------------------------------------------------------------------
// K1: pyramid level (resize from level 0) fused with the 7x7 Gaussian blur.  One CTA per kTileW x kTileH output tile.
//   cv::resize INTER_LINEAR 8UC1: 11-bit coefficient tables (built on the host exactly like OpenCV does), int32 maths.
//   cv::GaussianBlur 7x7 sigma 2: 8.8 fixed-point kernel {18,34,48,56,48,34,18}, u16 rows, (v + 32768) >> 16.
// Two launches per batch:
//   pyramid_level0_kernel   level 0 = the caller's image.  Stage A copies the tile (+ 3-px halo) with aligned word loads
//                           (two LDG.32 + one funnel shift per 4 pixels whatever the row's alignment; the caller's rows
//                           have an arbitrary stride) into shared memory; the level-0 image lands in the 16-byte
//                           aligned pyramid buffer.
//   pyramid_levels_kernel   levels >= 1, resized FROM THAT ALIGNED COPY (L2-resident): a row of it starts 16-byte aligned,
//                           so a thread's word alignment is the same in every row.  Stage A: thread <-> two adjacent
//                           columns; the 2 x 2 bytes they need from a source row lie inside one aligned 8-byte window
//                           (scale < 3), fetched with two LDG.32; each horizontal tap pair is one PRMT (per-thread
//                           constant selector) + one DP2A against the packed 11-bit coefficients; vertical weights by
//                           multiply-high (no clamp: the weights sum to 2048).
//   Stage B  horizontal pass on packed bytes: 3 aligned LDS.32 + funnel shifts + 8 DP4A per 4 pixels -> u16
//   Stage C  vertical pass: one item per 4 columns x 2 rows, LDS.128 of vertically paired u16, DP2A (exact integers)
//   The tile is stored with pixel 0 at byte 16 of a 96-byte row, so the level image leaves as LDS.128 / STG.128.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kSrcW = kTileW + 2 * kHalo;      // 70
constexpr int kSrcH = kTileH + 2 * kHalo;      // tile rows + halo
constexpr int kSrcPitch = 96;                  // bytes, 16-byte multiple
constexpr int kSrcCol0 = 13;                   // byte of source column 0 inside a row: tile pixel 0 sits at byte 16 (LDS.128 rows)
constexpr int kSrcWord0 = 3;                   // first word of a row that holds tile (+ halo) pixels: bytes 12..83 = columns -4..67
constexpr int kSrcWords = 18;
constexpr int kPairs = 36;                     // stage A of the resized levels: byte pairs 12 + 2q, 13 + 2q <-> columns 2q - 4, 2q - 3
constexpr int kPairRows = kPyrThreads / kPairs; // 7 rows per pass (252 threads)
constexpr int kWordRows = kPyrThreads / kSrcWords; // level 0: 14 rows per pass (252 threads)

constexpr int kPyrBoxBytes = 18 * 1024; // largest level-0 source rectangle staged through TMA (levels whose box fits)

template <int kHBytes> struct PyrSharedT
{
  __align__(16) uint8_t src[kSrcH * kSrcPitch];
  // horizontal-pass output (u16); in pyramid_levels_kernel the same bytes first receive the tile's level-0 source rectangle (TMA box)
  __align__(128) uint8_t hbuf[kHBytes];
  __device__ __forceinline__ uint16_t *h() { return reinterpret_cast<uint16_t *>(hbuf); }
  __device__ __forceinline__ const uint16_t *h() const { return reinterpret_cast<const uint16_t *>(hbuf); }
  // per source row: byte offsets of the two level-0 rows and the vertical coefficients pre-shifted by 16, so that
  // (b * (h >> 4)) >> 16 is one multiply-high (level 0: .x = row offset, .z = 1 when the row may be read with word loads)
  __align__(16) uint4 row[kSrcH];
};
using PyrShared = PyrSharedT<kSrcH * kTileW * 2>;
using PyrSharedBox = PyrSharedT<kPyrBoxBytes>;

// rows of the tile (+ halo) that exist: rows beyond level row lh + kHalo - 1 are never consumed
__device__ __forceinline__ int tile_rows(const Tile &t, int lh) { return min(kSrcH, lh + 2 * kHalo - t.y0); }

// the level image itself (getPyramid(); FAST, orientation and the stereo SAD read it): 16 pixels per load/store
template <class S> __device__ __forceinline__ void pyr_store_level(const S &sm, const Tile &t, int lh, int pitch, uint8_t *__restrict__ pyr)
{
  for (int i = threadIdx.x; i < kTileH * (kTileW / 16); i += kPyrThreads)
  {
    const int ty = i >> 2, tx = (i & 3) * 16;
    const int gx = t.x0 + tx, gy = t.y0 + ty;
    if (gy < lh && gx < pitch)
      *reinterpret_cast<uint4 *>(pyr + (size_t)gy * pitch + gx) = *reinterpret_cast<const uint4 *>(&sm.src[(ty + kHalo) * kSrcPitch + 16 + tx]);
  }
}

// stage B: horizontal pass, 2 rows x 4 outputs per item from 3 aligned words per row; output pixel 4g + k needs source
// bytes 4g + 13 + k .. + 6 of the row = words 3 + g .. 5 + g shifted by 8 (k + 1) bits; sums fit u16 (255 * 256).
// The two rows of a pair share a word (row 2j low, row 2j + 1 high) so that the vertical pass can use DP2A.
template <class S> __device__ __forceinline__ void pyr_blur_rows(S &sm, int rows)
{
  constexpr uint32_t K0 = 18u | (34u << 8) | (48u << 16) | (56u << 24); // taps 0..3
  constexpr uint32_t K1 = 48u | (34u << 8) | (18u << 16);               // taps 4..6
  const uint32_t *s32 = reinterpret_cast<const uint32_t *>(sm.src);
  uint4 *h4 = reinterpret_cast<uint4 *>(sm.h());
  const int g = threadIdx.x & 15;
  const int n_pairs = (rows + 1) >> 1;
  for (int j = threadIdx.x >> 4; j < n_pairs; j += kPyrThreads / 16)
  {
    const uint32_t *row = s32 + (2 * j) * (kSrcPitch / 4) + 3 + g;
    uint32_t o[2][4];
#pragma unroll
    for (int r = 0; r < 2; ++r)
    {
      const uint32_t w0 = row[r * (kSrcPitch / 4)], w1 = row[r * (kSrcPitch / 4) + 1], w2 = row[r * (kSrcPitch / 4) + 2];
      o[r][0] = __dp4a(__funnelshift_r(w0, w1, 8), K0, __dp4a(__funnelshift_r(w1, w2, 8), K1, 0u));
      o[r][1] = __dp4a(__funnelshift_r(w0, w1, 16), K0, __dp4a(__funnelshift_r(w1, w2, 16), K1, 0u));
      o[r][2] = __dp4a(__funnelshift_r(w0, w1, 24), K0, __dp4a(__funnelshift_r(w1, w2, 24), K1, 0u));
      o[r][3] = __dp4a(w1, K0, __dp4a(w2, K1, 0u));
    }
    h4[j * 16 + g] = make_uint4(o[0][0] | (o[1][0] << 16), o[0][1] | (o[1][1] << 16), o[0][2] | (o[1][2] << 16), o[0][3] | (o[1][3] << 16));
  }
}

// stage C: vertical pass + rounding; one item per 4 columns x 2 output rows (2y, 2y + 1).  Both rows read the same four
// row pairs y .. y + 3: the even row weighs them (18,34) (48,56) (48,34) (18,0), the odd row (0,18) (34,48) (56,48)
// (34,18) -- low / high byte pairs of the same weight registers (DP2A.LO / DP2A.HI).
template <class S> __device__ __forceinline__ void pyr_blur_cols(const S &sm, const Tile &t, int lh, int pitch, uint8_t *__restrict__ blr)
{
  const int g = threadIdx.x & 15;
  const int gx = t.x0 + g * 4;
  if (gx >= pitch) return;
  const int n_out = min(kTileH / 2, (lh - t.y0 + 1) >> 1);
  const uint4 *h4 = reinterpret_cast<const uint4 *>(sm.h());
  for (int yp = threadIdx.x >> 4; yp < n_out; yp += kPyrThreads / 16)
  {
    const int gy = t.y0 + 2 * yp;
    constexpr uint32_t W0 = 18u | (34u << 8) | (0u << 16) | (18u << 24), W1 = 48u | (56u << 8) | (34u << 16) | (48u << 24);
    constexpr uint32_t W2 = 48u | (34u << 8) | (56u << 16) | (48u << 24), W3 = 18u | (0u << 8) | (34u << 16) | (18u << 24);
    const uint4 p0 = h4[yp * 16 + g], p1 = h4[(yp + 1) * 16 + g], p2 = h4[(yp + 2) * 16 + g], p3 = h4[(yp + 3) * 16 + g];
    const uint32_t c0[4] = {p0.x, p0.y, p0.z, p0.w}, c1[4] = {p1.x, p1.y, p1.z, p1.w}, c2[4] = {p2.x, p2.y, p2.z, p2.w}, c3[4] = {p3.x, p3.y, p3.z, p3.w};
    uint32_t we = 0, wo = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
    {
      const uint32_t e = __dp2a_lo(c3[k], W3, __dp2a_lo(c2[k], W2, __dp2a_lo(c1[k], W1, __dp2a_lo(c0[k], W0, 32768u))));
      const uint32_t o = __dp2a_hi(c3[k], W3, __dp2a_hi(c2[k], W2, __dp2a_hi(c1[k], W1, __dp2a_hi(c0[k], W0, 32768u))));
      we |= (e >> 16) << (8 * k);
      wo |= (o >> 16) << (8 * k);
    }
    *reinterpret_cast<uint32_t *>(blr + (size_t)gy * pitch + gx) = we;
    if (gy + 1 < lh) *reinterpret_cast<uint32_t *>(blr + (size_t)(gy + 1) * pitch + gx) = wo;
  }
}

// Colour input (orbx_set_input_format): cv::cvtColor's 8-bit RGB -> gray rule, gray = (w0 c0 + w1 c1 + w2 c2 + 16384) >> 15
// with the weights of the channel order (9798 R, 19235 G, 3735 B; they sum to 32768, so the result is at most 255).  `px`
// holds one pixel's first three bytes in bytes 0..2; byte 3 (alpha, or the next pixel's first byte) weighs 0.
__device__ __forceinline__ uint32_t gray_of(uint32_t px, uint32_t w01, uint32_t w2) { return __dp2a_lo(w01, px, __dp2a_hi(w2, px, 16384u)) >> 15; }

// one gray pixel of the caller's image: q = its first byte
template <int kBpp> __device__ __forceinline__ uint32_t gray_at(const uint8_t *q, const Params &p)
{
  if constexpr (kBpp == 1)
    return *q;
  else
    return gray_of((uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16), p.cvt_w01, p.cvt_w2);
}

// the 4 gray bytes of 4 consecutive pixels held in b[0 .. kBpp) (4 * kBpp bytes, pixel k at byte k * kBpp)
template <int kBpp> __device__ __forceinline__ uint32_t gray4(const uint32_t (&b)[kBpp], uint32_t w01, uint32_t w2)
{
  uint32_t px[4];
  if constexpr (kBpp == 4)
    px[0] = b[0], px[1] = b[1], px[2] = b[2], px[3] = b[3];
  else
    px[0] = b[0], px[1] = __funnelshift_r(b[0], b[1], 24), px[2] = __funnelshift_r(b[1], b[2], 16), px[3] = b[2] >> 8;
  uint32_t v = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) v |= gray_of(px[k], w01, w2) << (8 * k);
  return v;
}

// kBpp = bytes per pixel of the caller's images (1 gray, 3 RGB / BGR, 4 RGBA / BGRA); the channel order travels as weights
template <int kBpp> __global__ void __launch_bounds__(kPyrThreads) pyramid_level0_kernel(const Params p)
{
  __shared__ PyrShared sm;
  const Tile t = p.tiles[blockIdx.x];
  const int img = blockIdx.y;
  const Level &L = p.levels[0];
  const int lw = L.w, lh = L.h, pitch = L.pitch;
  const uint8_t *__restrict__ src = input_image(p, img);
  const uint32_t sstride = (uint32_t)p.in_stride;
  const int tid = threadIdx.x;
  const int rows = tile_rows(t, lh);

  // Row table for all kSrcH entries (rows beyond `rows` repeat row 0 and are never consumed): .x = byte offset of the source row,
  // .z = 1 when the row may be read with aligned word loads.  Rows 0 and lh - 1 are gathered byte by byte: an aligned word
  // may reach up to 3 bytes outside the caller's buffer there.
  if (tid < kSrcH)
  {
    const int gy = tid < rows ? refl101(t.y0 + tid - kHalo, lh) : 0;
    sm.row[tid] = make_uint4((uint32_t)gy * sstride, 0u, (tid < rows && gy > 0 && gy < lh - 1) ? 1u : 0u, 0u);
  }
  __syncthreads();

  // stage A: thread <-> word column j (source columns x0 - 4 + 4 j .. + 3), kWordRows rows per pass.  Word columns jl .. jh lie
  // completely inside the image: two aligned loads + a funnel shift per word, no per-row branch.  The others (the left / right
  // borders: REFLECT_101, zero beyond the level + halo) and the first / last image row are patched byte by byte afterwards.
  // Colour: the 4 pixels of a word column are a 12- / 16-byte window at any alignment, read as 4 / 5 aligned words (at most
  // 3 bytes before and 4 after the window, as for gray) and funnel-shifted into place, then converted to 4 gray bytes.
  const int jl = t.x0 == 0 ? 1 : 0, jh = min(kSrcWords - 1, (lw - t.x0) >> 2);
  {
    const int j = tid % kSrcWords, grp = tid / kSrcWords;
    if (grp < kWordRows && j >= jl && j <= jh)
    {
      uint32_t *dst = reinterpret_cast<uint32_t *>(sm.src) + kSrcWord0 + j + grp * (kSrcPitch / 4);
      const uint8_t *col_src = src + (t.x0 - 4 + 4 * j) * kBpp;
      asm volatile("" : "+l"(col_src)); // one register pair: a row address is one IMAD.WIDE.U32
      const uint4 *rp = sm.row + grp;
      constexpr int U = 5; // 70 rows = 14 rows per pass x 5: all loads of a tile are issued before the first use
      static_assert(kWordRows * U == kSrcH, "the row passes tile the buffer exactly");
      if constexpr (kBpp == 1)
      {
        uint32_t w0[U], w1[U], sh[U], ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
        {
          const uint4 r = rp[u * kWordRows];
          const uint8_t *a = col_src + r.x;
          ok[u] = r.z;
          w0[u] = w1[u] = 0u;
          if (ok[u])
          {
            const uint32_t *al = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(a) & ~(uintptr_t)3);
            w0[u] = al[0], w1[u] = al[1];
          }
          sh[u] = (uint32_t)reinterpret_cast<uintptr_t>(a) << 3; // funnel shifts take the amount modulo 32
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (ok[u]) dst[u * kWordRows * (kSrcPitch / 4)] = __funnelshift_r(w0[u], w1[u], sh[u]);
      }
      else
      {
        constexpr int NW = kBpp + 1; // aligned words that cover a window of kBpp words at any alignment
        uint32_t w[U][NW], sh[U], ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
        {
          const uint4 r = rp[u * kWordRows];
          const uint8_t *a = col_src + r.x;
          ok[u] = r.z;
#pragma unroll
          for (int k = 0; k < NW; ++k) w[u][k] = 0u;
          if (ok[u])
          {
            const uint32_t *al = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(a) & ~(uintptr_t)3);
#pragma unroll
            for (int k = 0; k < NW; ++k) w[u][k] = al[k];
          }
          sh[u] = (uint32_t)reinterpret_cast<uintptr_t>(a) << 3;
        }
        const uint32_t w01 = p.cvt_w01, w2 = p.cvt_w2;
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (ok[u])
          {
            uint32_t b[kBpp];
#pragma unroll
            for (int k = 0; k < kBpp; ++k) b[k] = __funnelshift_r(w[u][k], w[u][k + 1], sh[u]);
            dst[u * kWordRows * (kSrcPitch / 4)] = gray4<kBpp>(b, w01, w2);
          }
      }
    }
  }
  {
    auto gather_word = [&](int ty, int j) { // REFLECT_101 per pixel; columns beyond the level + halo are zero
      const uint8_t *rowp = src + (size_t)sm.row[ty].x;
      const int rx = t.x0 - 4 + 4 * j;
      uint32_t v = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (rx + k < lw + kHalo) v |= gray_at<kBpp>(rowp + refl101(rx + k, lw) * kBpp, p) << (8 * k);
      reinterpret_cast<uint32_t *>(sm.src)[ty * (kSrcPitch / 4) + kSrcWord0 + j] = v;
    };
    // border word columns [0, jl) and (jh, kSrcWords), all rows
    const int n_slow = jl + (kSrcWords - 1 - jh);
    for (int i = tid; i < rows * n_slow; i += kPyrThreads)
    {
      const int ty = i / n_slow, k = i - ty * n_slow;
      gather_word(ty, k < jl ? k : jh + 1 + (k - jl));
    }
    // image rows 0 and lh - 1 (at most one tile row each), inner word columns
    const int ty_first = kHalo - t.y0, ty_last = lh - 1 + kHalo - t.y0;
    for (int i = tid; i < 2 * kSrcWords; i += kPyrThreads)
    {
      const int ty = i < kSrcWords ? ty_first : ty_last, j = i < kSrcWords ? i : i - kSrcWords;
      if (ty >= 0 && ty < rows && j >= jl && j <= jh && (i < kSrcWords || ty_last != ty_first)) gather_word(ty, j);
    }
  }
  __syncthreads();

  pyr_store_level(sm, t, lh, pitch, p.pyr + (size_t)img * p.pyr_img_stride + L.pyr_off);
  pyr_blur_rows(sm, rows);
  __syncthreads();
  pyr_blur_cols(sm, t, lh, pitch, p.blur + (size_t)img * p.pyr_img_stride + L.pyr_off);
}

template <bool kSharedWindow, bool kBox, class S> __device__ __forceinline__ void resize_rows(S &sm, const uint8_t *__restrict__ l0, uint32_t box_u32, int rows, int q, int grp,
                                                                           uint32_t base_a, uint32_t base_b, uint32_t sel_a, uint32_t sel_b,
                                                                           uint32_t coef_a, uint32_t coef_b)
{
  // No clamps, no store predicate: the row table is valid for all kSrcH entries (rows beyond `rows` repeat row 0) and a
  // pass may write up to kPairRows * (U - 1) rows past `rows` -- still inside the tile buffer, never consumed.
  uint16_t *dst = reinterpret_cast<uint16_t *>(sm.src) + (kSrcWord0 * 2 + q) + grp * (kSrcPitch / 2);
  const uint4 *rp = sm.row + grp;
  const uint8_t *pa = l0 + base_a, *pb = l0 + base_b;
  // keep the two window pointers in register pairs: a row address is then ONE IMAD.WIDE.U32 (pointer + 32-bit row offset)
  // instead of a chain of 3-input adds that rebuilds the image base from its uniform parts
  asm volatile("" : "+l"(pa), "+l"(pb));
  constexpr int U = 2; // rows per batch: 8 (16) word loads in flight per thread
  static_assert(kSrcH % (U * kPairRows) == 0, "the row passes tile the buffer exactly");
  for (int ty0 = grp; ty0 < rows; ty0 += U * kPairRows, rp += U * kPairRows, dst += U * kPairRows * (kSrcPitch / 2))
  {
    uint32_t a0[U], a1[U], a2[U], a3[U], b0[U], b1[U], b2[U], b3[U], bz[U], bw[U];
#pragma unroll
    for (int u = 0; u < U; ++u)
    {
      const uint4 r = rp[u * kPairRows];
      if (kBox)
      { // the source rectangle is in shared memory (TMA box): row offsets and window offsets are relative to the box
        const uint32_t q0 = box_u32 + base_a + r.x, q1 = box_u32 + base_a + r.y;
        a0[u] = lds_u32(q0), a1[u] = lds_u32(q0 + 4u), a2[u] = lds_u32(q1), a3[u] = lds_u32(q1 + 4u);
        if (!kSharedWindow)
        {
          const uint32_t s0 = box_u32 + base_b + r.x, s1 = box_u32 + base_b + r.y;
          b0[u] = lds_u32(s0), b1[u] = lds_u32(s0 + 4u), b2[u] = lds_u32(s1), b3[u] = lds_u32(s1 + 4u);
        }
      }
      else
      {
        const uint32_t *q0 = reinterpret_cast<const uint32_t *>(pa + r.x), *q1 = reinterpret_cast<const uint32_t *>(pa + r.y);
        a0[u] = q0[0], a1[u] = q0[1], a2[u] = q1[0], a3[u] = q1[1];
        if (!kSharedWindow)
        {
          const uint32_t *s0 = reinterpret_cast<const uint32_t *>(pb + r.x), *s1 = reinterpret_cast<const uint32_t *>(pb + r.y);
          b0[u] = s0[0], b1[u] = s0[1], b2[u] = s1[0], b3[u] = s1[1];
        }
      }
      if (kSharedWindow) b0[u] = a0[u], b1[u] = a1[u], b2[u] = a2[u], b3[u] = a3[u];
      bz[u] = r.z, bw[u] = r.w;
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
    {
      const uint32_t ha0 = __dp2a_lo(coef_a, __byte_perm(a0[u], a1[u], sel_a), 0u), ha1 = __dp2a_lo(coef_a, __byte_perm(a2[u], a3[u], sel_a), 0u);
      const uint32_t hb0 = __dp2a_lo(coef_b, __byte_perm(b0[u], b1[u], sel_b), 0u), hb1 = __dp2a_lo(coef_b, __byte_perm(b2[u], b3[u], sel_b), 0u);
      // (((bx * (h0 >> 4)) >> 16) + ((by * (h1 >> 4)) >> 16) + 2) >> 2; at most 255 because bx + by == 2048
      const uint32_t va = (__umulhi(bz[u], ha0 >> 4) + __umulhi(bw[u], ha1 >> 4) + 2u) >> 2;
      const uint32_t vb = (__umulhi(bz[u], hb0 >> 4) + __umulhi(bw[u], hb1 >> 4) + 2u) >> 2;
      dst[u * kPairRows * (kSrcPitch / 2)] = (uint16_t)(va | (vb << 8));
    }
  }
}

__global__ void __launch_bounds__(kPyrThreads) pyramid_levels_kernel(const Params p, const __grid_constant__ LevelMaps src_maps)
{
  __shared__ PyrSharedBox sm;
  __shared__ __align__(8) uint64_t s_bar;
  const Tile t = p.tiles[p.n_tiles0 + blockIdx.x];
  const int img = blockIdx.y;
  const Level &L = p.levels[t.level];
  const int lw = L.w, lh = L.h, pitch = L.pitch;
  const int H = p.height;
  const int area2x = L.area2x;
  const int tid = threadIdx.x;
  const int rows = tile_rows(t, lh);
  // level 0 of this image inside the pyramid buffer (written by pyramid_level0_kernel, same stream)
  const uint8_t *__restrict__ l0 = p.pyr + (size_t)img * p.pyr_img_stride + p.levels[0].pyr_off;
  // Levels whose per-tile source rectangle fits (scale < 2 at the usual 1.2 pyramid: most of the resized pixels) stage it in
  // shared memory through ONE TMA box load from the aligned level-0 copy: box origin (sx0, sy0) from the tile record (sx0 a
  // multiple of 16), box size per level.  The other levels gather their taps from global memory (L2) with the same arithmetic.
  const int box_w = L.src_box_w, box_h = L.src_box_h;
  const bool boxed = box_w != 0;
  const int sx0 = t.src & 0xffff, sy0 = t.src >> 16;
  if (boxed && tid == 0)
  {
    mbar_init(&s_bar, 1);
    mbar_expect_tx(&s_bar, (uint32_t)(box_w * box_h));
    tma_load_3d(sm.hbuf, &src_maps.m[t.level], sx0, sy0, p.img0 + img, &s_bar);
  }
  const uint32_t row_pitch = boxed ? (uint32_t)box_w : (uint32_t)p.levels[0].pitch;
  const int row_org = boxed ? sy0 : 0;

  if (tid < rows)
  {
    const int gy = refl101(t.y0 + tid - kHalo, lh);
    uint32_t o0, o1, z = 0, w = 0;
    if (area2x)
    {
      o0 = (uint32_t)(2 * gy) * row_pitch;
      o1 = o0 + row_pitch;
    }
    else
    {
      const int sy = p.tab_ofs[L.tab_y + gy];
      const short2 b = p.tab_coef[L.tab_y + gy];
      o0 = (uint32_t)(min(max(sy, 0), H - 1) - row_org) * row_pitch; // rows are clamped, not re-weighted (cv::resize)
      o1 = (uint32_t)(min(max(sy + 1, 0), H - 1) - row_org) * row_pitch;
      z = (uint32_t)b.x << 16, w = (uint32_t)b.y << 16; // coefficients are in [0, 2048]
    }
    sm.row[tid] = make_uint4(o0, o1, z, w);
  }
  else if (tid < kSrcH)
    sm.row[tid] = make_uint4(0u, 0u, 0u, 0u); // rows beyond the level: any valid source row, weights 0 (never consumed)
  __syncthreads(); // also orders thread 0's mbarrier init before everybody's wait
  if (boxed) mbar_wait(&s_bar, 0);

  // stage A: the tile plus a 3-pixel halo of the resized level image, REFLECT_101 at the level's borders.
  if (area2x)
  {
    // exact 2x decimation: cv::resize re-routes INTER_LINEAR to INTER_AREA = rounded 2x2 means
    for (int i = tid; i < rows * kSrcW; i += kPyrThreads)
    {
      const int ty = i / kSrcW, col = i - ty * kSrcW;
      const int rx = t.x0 + col - kHalo;
      uint32_t v = 0;
      if (rx < lw + kHalo)
      {
        const uint4 r = sm.row[ty];
        const uint8_t *q0 = l0 + r.x + 2 * refl101(rx, lw), *q1 = l0 + r.y + 2 * refl101(rx, lw);
        v = (q0[0] + q0[1] + q1[0] + q1[1] + 2) >> 2;
      }
      sm.src[ty * kSrcPitch + kSrcCol0 + col] = (uint8_t)v;
    }
  }
  else
  {
    const int q = tid % kPairs, grp = tid / kPairs;
    if (grp < kPairRows)
    {
      // columns rx = x0 - 4 + 2 q and rx + 1 (x0 - 4 and x0 + 67 are not used by anybody): their taps come from the level's
      // pair table (built on the host next to the resize tables): window offsets into a level-0 row, PRMT selectors of the two
      // tap pairs, packed coefficients ax | ay << 16 (0 for columns beyond the level + halo: value 0)
      const uint4 e = p.tab_pair[L.tab_pair + (t.x0 >> 1) + q];
      const uint32_t box_u32 = smem_u32(sm.hbuf) - (uint32_t)sx0; // window offsets are level-0 columns
      if (boxed)
      {
        if (L.pair_window)
          resize_rows<true, true>(sm, l0, box_u32, rows, q, grp, e.x & 0xffffu, e.x & 0xffffu, e.x >> 16, e.y >> 16, e.z, e.w);
        else
          resize_rows<false, true>(sm, l0, box_u32, rows, q, grp, e.x & 0xffffu, e.y & 0xffffu, e.x >> 16, e.y >> 16, e.z, e.w);
      }
      else if (L.pair_window)
        resize_rows<true, false>(sm, l0, 0u, rows, q, grp, e.x & 0xffffu, e.x & 0xffffu, e.x >> 16, e.y >> 16, e.z, e.w);
      else
        resize_rows<false, false>(sm, l0, 0u, rows, q, grp, e.x & 0xffffu, e.y & 0xffffu, e.x >> 16, e.y >> 16, e.z, e.w);
    }
  }
  __syncthreads();

  pyr_store_level(sm, t, lh, pitch, p.pyr + (size_t)img * p.pyr_img_stride + L.pyr_off);
  pyr_blur_rows(sm, rows);
  __syncthreads();
  pyr_blur_cols(sm, t, lh, pitch, p.blur + (size_t)img * p.pyr_img_stride + L.pyr_off);
}

const void *pyramid_kernel_symbol(int bpp)
{
  return bpp == 4 ? reinterpret_cast<const void *>(&pyramid_level0_kernel<4>)
                  : (bpp == 3 ? reinterpret_cast<const void *>(&pyramid_level0_kernel<3>) : reinterpret_cast<const void *>(&pyramid_level0_kernel<1>));
}

// two launches: level 0 (reads the caller's images), then the resized levels (read level 0 from the pyramid buffer)
void launch_pyramid_level0(const Params &p, int n_images, cudaStream_t s)
{
  const dim3 grid(p.n_tiles0, n_images);
  if (p.in_bpp == 4)
    pyramid_level0_kernel<4><<<grid, kPyrThreads, 0, s>>>(p);
  else if (p.in_bpp == 3)
    pyramid_level0_kernel<3><<<grid, kPyrThreads, 0, s>>>(p);
  else
    pyramid_level0_kernel<1><<<grid, kPyrThreads, 0, s>>>(p);
}

void launch_pyramid_levels(const Params &p, const LevelMaps &src_maps, int n_images, cudaStream_t s)
{
  if (p.n_tiles > p.n_tiles0) pyramid_levels_kernel<<<dim3(p.n_tiles - p.n_tiles0, n_images), kPyrThreads, 0, s>>>(p, src_maps);
}

// ------------------------------------------------------------------------------------------------------------------
// K2: FAST-9/16 with non-max suppression per 30-px cell and the iniTh -> minTh fallback.  One warp per cell.
//   arc value m(p) = max over the 16 arcs of 9 contiguous ring pixels of min(+-(I(p) - I(ring)));
//   corner at threshold t  <=>  m > t;  cv score = m - 1;  keep iff score > all 8 neighbours' scores (strict), where a
//   neighbour that is not a corner at t, or lies outside the cell's detection zone, scores 0.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kPatPitch = 80;                 // bytes = width of the TMA box: (x0 & 15) + patch width (<= 65)
constexpr int kZoneMax = 64;                  // detection zone edge (patch edge - 6); one 64-bit mask per zone row

__device__ __forceinline__ int fast_arc_value(const uint8_t *c)
{
  // m = max over the 16 arcs of 9 contiguous ring pixels of min(v - r) ("ring darker") and of min(r - v) ("ring brighter").
  // Both chains run in ONE register per ring pixel, as two signed 16-bit halves on the packed min/max unit
  // (VIMNMX(3).S16x2).  With G = 2 (r - v) + 1 (odd, so its sign is never ambiguous) one multiply-add packs
  //   x = G * 0xFFFF = (G << 16) - G :  low half = -G = 2 (v - r) - 1,  high half = G - [G > 0]   (borrow of the low half)
  // and both halves are strictly monotone in v - r / r - v, so min / max commute with the packing; the two transforms
  // are undone once, on the result.  (Plain int chains: twice the instructions, and nvcc 12.9 for sm_100a mis-folds
  // "max(best, max(mn9, -mx9))" into a 3-input VIMNMX3 that drops the negation.)
  constexpr int P = kPatPitch;
  const unsigned C = (unsigned)(1 - 2 * (int)c[0]) * 0xFFFFu;
  unsigned x[16];
  x[0] = c[3 * P] * 0x1FFFEu + C;
  x[1] = c[3 * P + 1] * 0x1FFFEu + C;
  x[2] = c[2 * P + 2] * 0x1FFFEu + C;
  x[3] = c[P + 3] * 0x1FFFEu + C;
  x[4] = c[3] * 0x1FFFEu + C;
  x[5] = c[-P + 3] * 0x1FFFEu + C;
  x[6] = c[-2 * P + 2] * 0x1FFFEu + C;
  x[7] = c[-3 * P + 1] * 0x1FFFEu + C;
  x[8] = c[-3 * P] * 0x1FFFEu + C;
  x[9] = c[-3 * P - 1] * 0x1FFFEu + C;
  x[10] = c[-2 * P - 2] * 0x1FFFEu + C;
  x[11] = c[-P - 3] * 0x1FFFEu + C;
  x[12] = c[-3] * 0x1FFFEu + C;
  x[13] = c[P - 3] * 0x1FFFEu + C;
  x[14] = c[2 * P - 2] * 0x1FFFEu + C;
  x[15] = c[3 * P - 1] * 0x1FFFEu + C;
  unsigned a3[16]; // min over ring pixels k .. k + 2
#pragma unroll
  for (int k = 0; k < 16; ++k) a3[k] = __vmins2(__vmins2(x[k], x[(k + 1) & 15]), x[(k + 2) & 15]);
  unsigned best = 0x80008000u;
#pragma unroll
  for (int k = 0; k < 16; ++k) best = __vmaxs2(best, __vmins2(__vmins2(a3[k], a3[(k + 3) & 15]), a3[(k + 6) & 15])); // k .. k + 8
  const int lo = (int)(short)(best & 0xffffu), hi = (int)best >> 16;
  const int darker = (lo + 1) >> 1;                      // lo = 2 m - 1
  const int brighter = (hi + (hi >= 0 ? 1 : 0) - 1) >> 1; // hi = G - [G > 0], G = 2 m + 1
  return max(darker, brighter);
}

constexpr int kFastWarps = kFastThreads / 32;

// Stage-1 test on two pixels at once (16-bit halves of a register, VIMNMX.U16x2): "two ADJACENT compass ring pixels are
// brighter (darker) than the centre by more than t".  The operands carry each pixel in the HIGH byte of its half (the low
// byte is whatever neighbour came along): an unsigned 16-bit max / min is decided by the high bytes, so the high bytes of
// hi2 / lo2 are exact and only v, hi2 and lo2 need unpacking.  c1 = 0x80008000 - (t + 1) * 0x00010001: bit 15 of a half of
// hi2 - v + c1 is set iff hi2 - v > t (every half stays inside [0, 65535], so the 32-bit add never carries between halves).
__device__ __forceinline__ uint32_t fast_pretest2(uint32_t v, uint32_t dn, uint32_t rt, uint32_t up, uint32_t lf, uint32_t c1, uint32_t mask)
{
  const uint32_t hi2 = __byte_perm(__vminu2(__vmaxu2(dn, up), __vmaxu2(rt, lf)), 0u, 0x4341);
  const uint32_t lo2 = __byte_perm(__vmaxu2(__vminu2(dn, up), __vminu2(rt, lf)), 0u, 0x4341);
  const uint32_t vc = __byte_perm(v, 0u, 0x4341);
  return ((hi2 - vc + c1) | (vc - lo2 + c1)) & mask;
}

// One WARP per cell: a 30 x 30-px cell is too small for a thread block -- its serial phases (map zeroing, suppression over
// ~40 corners, the output scan) would run on all warps for a handful of active lanes, and every phase boundary would be a
// block barrier.  A CTA is kFastWarps independent cells (ONE since the cells differ in length: a cell that needs the minThFAST
// pass would hold its neighbours' slots); each warp owns a slice of the dynamic shared memory:
//   patch (TMA box) | mbarrier | score map | candidate list | keep masks | flag-bit -> code table
__global__ void __launch_bounds__(kFastThreads) fast_cells_kernel(const Params p, const __grid_constant__ LevelMaps maps)
{
  extern __shared__ __align__(128) uint8_t fast_smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int cell = blockIdx.x * kFastWarps + wid;
  if (cell >= p.n_cells) return;
  const int img = blockIdx.y;
  uint8_t *const wbase = fast_smem + (size_t)wid * p.fast_warp_bytes;
  uint8_t *const s_pat = wbase;
  uint64_t *const s_bar = reinterpret_cast<uint64_t *>(wbase + p.fast_off_bar);
  uint8_t *const s_map = wbase + p.fast_off_map;
  unsigned long long *const s_keep = reinterpret_cast<unsigned long long *>(wbase + p.fast_off_mask);
  const uint32_t cand_u32 = smem_u32(wbase + p.fast_off_cand);
  // flag bit -> candidate code offset (rows 8 s + e, pixel 2 (b >> 4)): a 32-entry table instead of four ALU operations per candidate
  const uint32_t lut_u32 = smem_u32(wbase + p.fast_off_lut);
  sts_u16_if(lut_u32 + 2u * (uint32_t)(threadIdx.x & 31), (uint32_t)(((threadIdx.x & 7) * 8 + ((threadIdx.x >> 3) & 1)) * kZoneMax + ((threadIdx.x >> 4) & 1) * 2), true);
  const int mp = p.fast_map_pitch;

  const Cell c = p.cells[cell];
  const int pw = c.pw, ph = c.ph;
  const int zw = pw - 6, zh = ph - 6; // detection zone: FAST looks at [3, w-3) x [3, h-3) of the patch
  if (zw <= 0 || zh <= 0)
  {
    if (lane == 0) p.cell_cnt[(size_t)img * p.n_cells + cell] = 0;
    return;
  }

  // The patch (plus whatever lies right of / below it up to the box size; out-of-range bytes are zero-filled) arrives
  // through one TMA box load issued by lane 0; the map zeroing of the first threshold pass overlaps it.
  if (lane == 0)
  {
    mbar_init(s_bar, 1);
    mbar_expect_tx(s_bar, (uint32_t)(kPatPitch * c.box_h));
    tma_load_3d(s_pat, &maps.m[c.level], c.x0 & ~15, c.y0, p.img0 + img, s_bar); // TMA needs 16-byte aligned row starts
  }
  __syncwarp();
  const int a0 = 3 + (c.x0 & 15);                    // byte of zone column 0 inside a patch row; 15 + 65 <= the 80-byte box
  const uint8_t *pat0 = s_pat + 3 * kPatPitch + a0;  // zone pixel (0,0)
  const uint32_t pat_u32 = smem_u32(s_pat);

  // stage 1: lane <-> 4 adjacent zone pixels, 8 lanes per row, 4 rows per step; zones wider than 32 px take two column passes
  const int n_xp = zw > 32 ? 2 : 1;
  const int xi = lane & 7, yq = lane >> 3;
  // A step works on the four rows r0 + 2 yq (yq = 0..3): two rows apart, because the 80-byte patch pitch puts rows y and
  // y + 2 exactly 8 banks apart (40 words), so the 4 x 8 words of one load instruction fall into 32 different banks
  // (consecutive rows, 20 words apart, collide two-way).  Steps come in pairs: rows 8 s + 2 yq, then rows 8 s + 1 + 2 yq.
  const int n_steps2 = (zh + 7) >> 3;                                 // <= 8
  // flag bit of (pair s, row parity e) = 8 e + s; the bits whose row 8 s + e + 2 yq lies inside the zone (both halves):
  const int ne = max(0, (zh - 2 * yq + 7) >> 3), no = max(0, (zh - 2 * yq - 1 + 7) >> 3);
  const uint32_t step_ok = (((1u << ne) - 1u) | (((1u << no) - 1u) << 8)) * 0x00010001u;

  bool patch_ready = false;
  unsigned long long keep0 = 0ull, keep1 = 0ull;

  // cv::FAST(cell, iniThFAST); only if its post-NMS list is empty, cv::FAST(cell, minThFAST) (src/ORBExtractor.cc:365-367).
  // Running the thresholds one after the other (instead of computing everything at the lower one) keeps the second,
  // far more expensive pass to the few cells that need it.
  for (int pass = 0; pass < 2; ++pass)
  {
    const int t = pass == 0 ? p.ini_th : p.min_th;
    {
      uint4 *m128 = reinterpret_cast<uint4 *>(s_map);
      for (int i = lane; i < ((zh + 2) * mp + 15) / 16; i += 32) m128[i] = make_uint4(0u, 0u, 0u, 0u);
      for (int i = lane; i < zh; i += 32) s_keep[i] = 0ull;
    }
    __syncwarp();
    if (!patch_ready)
    {
      mbar_wait(s_bar, 0);
      patch_ready = true;
    }

    // Stage 1 (every zone pixel): two adjacent compass ring pixels are brighter (darker) than the centre by more than t
    // -- a necessary condition for a 9-arc: 9 contiguous ring pixels always contain two ADJACENT compass pixels, i.e. one
    // of {0, 8} and one of {4, 12}; brighter arc => min(max(r0, r8), max(r4, r12)) > v + t, darker arc =>
    // max(min(r0, r8), min(r4, r12)) < v - t.  Four pixels per lane from aligned words, two per register half.
    // The flags stay in the lane: bit 8 e + s of the low / high half of acc_a = pixels 0 / 2 of the lane's item in row
    // 8 s + e + 2 yq, acc_b likewise pixels 1 / 3.  Then the lanes expand their bits into the dense candidate list (exclusive scan
    // of the counts), so that the next stage runs on dense lanes.
    int n_cand = 0;
    {
      const uint32_t c1 = 0x80008000u - (uint32_t)(t + 1) * 0x00010001u;
      for (int xp = 0; xp < n_xp; ++xp)
      {
        const int zx0 = 32 * xp + 4 * xi, n_valid = zw - zx0;
        const uint32_t vm = n_valid >= 4 ? 0xFu : (n_valid <= 0 ? 0u : (1u << n_valid) - 1u);
        // flag masks of the lane's valid pixels: pixels (0, 2) live in bits 15 / 31 of one register, (1, 3) of another
        const uint32_t ma = ((vm & 1u) ? 0x8000u : 0u) | ((vm & 4u) ? 0x80000000u : 0u), mb = ((vm & 2u) ? 0x8000u : 0u) | ((vm & 8u) ? 0x80000000u : 0u);
        const uint32_t bv = (uint32_t)(a0 + min(zx0, (zw - 1) & ~3)); // first byte of the item in its patch row (idle lanes stay inside the row)
        const uint32_t row0 = pat_u32 + (uint32_t)(2 * yq + 3) * kPatPitch;
        // aligned word + funnel shift: the 4 pixels, their left (x - 3) and right (x + 3) compass neighbours
        uint32_t pv = row0 + (bv & ~3u), pl = row0 + ((bv - 3u) & ~3u), pr = row0 + ((bv + 3u) & ~3u);
        const uint32_t sv = (bv & 3u) * 8u, sl = ((bv - 3u) & 3u) * 8u, sr = ((bv + 3u) & 3u) * 8u;
        uint32_t acc_a = 0u, acc_b = 0u;
        // rows past the zone read whatever follows the patch inside the warp's slice; their flags are dropped by step_ok
        auto pretest_rows = [&](uint32_t o, int bit, uint32_t &fa, uint32_t &fb) {
          const uint32_t v = __funnelshift_r(lds_u32(pv + o), lds_u32(pv + o + 4u), sv);
          const uint32_t lf = __funnelshift_r(lds_u32(pl + o), lds_u32(pl + o + 4u), sl);
          const uint32_t rt = __funnelshift_r(lds_u32(pr + o), lds_u32(pr + o + 4u), sr);
          const uint32_t up = __funnelshift_r(lds_u32(pv + o - 3 * kPatPitch), lds_u32(pv + o - 3 * kPatPitch + 4u), sv);
          const uint32_t dn = __funnelshift_r(lds_u32(pv + o + 3 * kPatPitch), lds_u32(pv + o + 3 * kPatPitch + 4u), sv);
          // pixels (1, 3) sit in the high bytes of the halves as loaded, pixels (0, 2) after a shift by one byte
          fb |= fast_pretest2(v, dn, rt, up, lf, c1, mb) >> (15 - bit);
          fa |= fast_pretest2(v << 8, dn << 8, rt << 8, up << 8, lf << 8, c1, ma) >> (15 - bit);
        };
        for (int s2 = 0; s2 < n_steps2; ++s2, pv += 8 * kPatPitch, pl += 8 * kPatPitch, pr += 8 * kPatPitch)
        {
          pretest_rows(0u, s2, acc_a, acc_b);
          pretest_rows((uint32_t)kPatPitch, 8 + s2, acc_a, acc_b);
        }
        acc_a &= step_ok;
        acc_b &= step_ok;
        const int cnt = __popc(acc_a) + __popc(acc_b);
        const int inc = warp_inclusive_scan(cnt, lane);
        uint32_t wa = cand_u32 + 2u * (uint32_t)(n_cand + inc - cnt);
        n_cand += __shfl_sync(kFullMask, inc, 31);
        const uint32_t code0 = (uint32_t)(2 * yq * kZoneMax + zx0);
#pragma unroll
        for (int h = 0; h < 2; ++h)
        {
          uint32_t w = h == 0 ? acc_a : acc_b;
          while (w)
          {
            const uint32_t b = (uint32_t)__ffs((int)w) - 1u; // pair s = b & 7, row parity e = (b >> 3) & 1, pixel = 2 (b >> 4) + h
            w &= w - 1u;
            sts_u16_if(wa, code0 + lds_u16(lut_u32 + 2u * b) + (uint32_t)h, true);
            wa += 2u;
          }
        }
      }
    }
    __syncwarp();

    // Stage 2 (stage-1 survivors, dense lanes): the arc value m decides (corner at t <=> m > t) and is the score the
    // non-max suppression needs, so it goes straight into the map.  The list is compacted in place to the corners
    // (every chunk is read before it is overwritten).
    const unsigned lt_mask = (1u << lane) - 1u;
    uint32_t cend = cand_u32;
    for (int k0 = 0; k0 < n_cand; k0 += 32)
    {
      const int k = k0 + lane;
      bool corner = false;
      uint32_t i = 0;
      if (k < n_cand)
      {
        i = lds_u16(cand_u32 + 2u * k);
        const int zy = i >> 6, zx = i & (kZoneMax - 1);
        const int m = fast_arc_value(pat0 + zy * kPatPitch + zx);
        corner = m > t;
        if (corner) s_map[(zy + 1) * mp + zx + 1] = (uint8_t)m;
      }
      __syncwarp();
      const unsigned m = __ballot_sync(kFullMask, corner);
      sts_u16_if(cend + 2u * __popc(m & lt_mask), i, corner);
      cend += 2u * __popc(m);
    }
    const int n_corners = (int)(cend - cand_u32) >> 1;
    __syncwarp();

    // Non-max suppression: keep  <=>  score m - 1 > the scores of all 8 neighbours (strict), where a neighbour that is not
    // a corner at this threshold (map 0) scores 0; the map q -> (q ? q - 1 : 0) is monotone, so only the largest neighbour
    // matters.
    for (int k = lane; k < n_corners; k += 32)
    {
      const int i = (int)lds_u16(cand_u32 + 2u * (uint32_t)k);
      const int zy = i >> 6, zx = i & (kZoneMax - 1);
      const uint8_t *mq = &s_map[(zy + 1) * mp + zx + 1];
      const int m = mq[0];
      const int q = max(max(max((int)mq[-1], (int)mq[1]), max((int)mq[-mp - 1], (int)mq[-mp])),
                        max(max((int)mq[-mp + 1], (int)mq[mp - 1]), max((int)mq[mp], (int)mq[mp + 1])));
      if (m - 1 > (q ? q - 1 : 0)) atomicOr(&s_keep[zy], 1ull << zx);
    }
    __syncwarp();
    keep0 = lane < zh ? s_keep[lane] : 0ull;
    keep1 = lane + 32 < zh ? s_keep[lane + 32] : 0ull;
    if (__any_sync(kFullMask, (keep0 | keep1) != 0ull)) break; // fallback iff the post-NMS list is empty (:366)
  }

  // lane <-> zone rows lane and lane + 32, row-major output order: exclusive scans of the rows' corner counts
  static_assert(kZoneMax <= 64, "the output scan covers two rows per lane");
  const int cnt0 = __popcll(keep0), cnt1 = __popcll(keep1);
  const int inc0 = warp_inclusive_scan(cnt0, lane), inc1 = warp_inclusive_scan(cnt1, lane);
  const int tot0 = __shfl_sync(kFullMask, inc0, 31), total = tot0 + __shfl_sync(kFullMask, inc1, 31);
  uint32_t *slot = p.cell_list + (size_t)img * p.cell_entries + c.slot;
#pragma unroll
  for (int h = 0; h < 2; ++h)
  {
    unsigned long long keep = h == 0 ? keep0 : keep1;
    int off = h == 0 ? inc0 - cnt0 : tot0 + inc1 - cnt1;
    const int zy = lane + 32 * h;
    const uint32_t y = (uint32_t)(c.y0 - kEdge + 3 + zy); // ROI coordinates (:368-372)
    while (keep)
    {
      const int zx = __ffsll((long long)keep) - 1;
      keep &= keep - 1;
      const uint32_t score = (uint32_t)s_map[(zy + 1) * mp + zx + 1] - 1u;
      const uint32_t x = (uint32_t)(c.x0 - kEdge + 3 + zx);
      if (off < c.cap) slot[off] = x | (y << 12) | (score << 24);
      ++off;
    }
  }
  if (lane == 0) p.cell_cnt[(size_t)img * p.n_cells + cell] = min(total, c.cap);
}

int fast_configure(const Params &p)
{
  static SmemOptIn state;
  return raise_dynamic_smem(fast_cells_kernel, state, (size_t)kFastWarps * p.fast_warp_bytes);
}

void launch_fast(const Params &p, const LevelMaps &maps, int n_images, cudaStream_t s)
{
  dim3 grid((p.n_cells + kFastWarps - 1) / kFastWarps, n_images);
  fast_cells_kernel<<<grid, kFastThreads, (size_t)kFastWarps * p.fast_warp_bytes, s>>>(p, maps);
}

// ------------------------------------------------------------------------------------------------------------------
// K3: quadtree keypoint distribution.  One CTA per (level, image).
//   Phase A/B  concatenate the level's cell lists in cell-row-major order (the reference's levelKps order) into the
//              level's corner list (global scratch) and give every corner its DESCENT KEY: the root strip it falls in
//              and its quadrant at each of the next 9 subdivision depths (or "on a split line").  The sequence of nodes
//              that contain a corner is fixed by geometry alone (midlines are (a+b)/2 in double, exactly as :60-72), so
//              the keys can be computed for all corners in parallel, before any pop order is known.
//   Phase B'   the root split (initSplit :81-96) is done by the whole block: a stable partition of the corners by strip.
//   Phase C    warp 0 replays Quadtree::split(): the multimap<count, node, greater> becomes FIFO buckets indexed by
//              count with a descending cursor (a child never holds more corners than its parent, so the pop key is
//              monotone).  Counts >= 256 (a handful of early nodes) live in a small unsorted list ordered by
//              (count, insertion sequence); counts < 256 in 256 linked FIFO buckets.  A node's corner list is a range of
//              an index array, split by a stable 4-way warp partition (key digit -> ballot + popc) between two
//              ping-pong arrays; nodes deeper than the key covers fall back to the double-precision geometry test.
//   Phase D    nodes2kpoints(): best response per surviving node, ascending index order, shift by the 16-px margin.
// Index arrays / keys live in shared memory when the level has at most qt_smem_cap corners, otherwise in the global
// scratch; node pool, buckets and the big-node list are always in shared memory.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kQtBuckets = 256;  // small buckets hold counts 0..255
constexpr int kQtMaxBinStrips = 8; // up to this many root strips the block pre-sorts kQtPresort subdivision depths
constexpr int kQtPresort = 3;      // depths 1..3 (5 slots each: quadrants 0-3, "on a split line")
constexpr int kQtBinsPerStrip = 125;
constexpr int kNodeBytes = 8 + 4 + 3 * 2 + 1;  // shared memory per node: rec {lo, cnt|depth|buf} | seq | next prev free | state
constexpr int kKeyLevels = 9;    // subdivision depths encoded in a key (3 bits each) below the 5-bit strip id
constexpr int kKeyStripShift = 27;
constexpr uint32_t kKeyNoStrip = 31u;
constexpr uint32_t kDigitDrop = 7u;
// Node bounds are dyadic rationals: the strip bounds are float-rounded values below 4096 (at most 23 fractional bits) and
// every split halves an interval, adding one bit.  Up to depth 17 they are exact both in double ((a+b)/2 has at most
// 12 + 23 + 17 = 52 significant bits) and in 24.40 fixed point, so the integer computation below is bit-identical to the
// reference's double arithmetic (src/ORBExtractor.cc:60-72) -- and it keeps FP64 latency out of the single-warp loop.
// Deeper nodes (reachable only through single-corner nodes) continue in double exactly like the reference.
constexpr int kFixShift = 40;
constexpr int kFixDepth = 17; // nodes up to this depth store fixed-point bounds; nodes up to depth 16 split in fixed point

struct QtNodePool
{
  long long *r0, *r1, *c0, *c1; // bounds: 24.40 fixed point up to depth kFixDepth, IEEE double bit patterns below
  uint2 *rec;    // x = first index of the node's range, y = count (24 bits) | depth << 24 (7 bits, saturating) | buffer << 31
  uint32_t *seq;
  uint16_t *next, *prev, *free_ids;
  uint8_t *state; // 0 dead, 1 live, 2 live but beyond the first `need` entries
};

__device__ __forceinline__ uint2 qt_rec(uint32_t lo, uint32_t cnt, int depth, int buf)
{
  return make_uint2(lo, cnt | ((uint32_t)min(depth, 127) << 24) | ((uint32_t)buf << 31));
}
__device__ __forceinline__ uint32_t qt_rec_cnt(uint2 r) { return r.y & 0xffffffu; }
__device__ __forceinline__ int qt_rec_depth(uint2 r) { return (int)((r.y >> 24) & 127u); }
__device__ __forceinline__ int qt_rec_buf(uint2 r) { return (int)(r.y >> 31); }

__host__ __device__ inline size_t qt_align16(size_t b) { return (b + 15) & ~(size_t)15; }

// shared memory: node pool | bucket heads+tails | big-node list | (smem path) ia, ib (u16), key (u32)
// node-pool region: the sequential path's node pool / the loop-free path's records
static_assert(kNodeBytes <= 22, "the node-pool region is sized for 22 bytes per node");
__host__ __device__ inline size_t qt_pool_bytes(int node_cap)
{
  return qt_align16((size_t)node_cap * 22 + 16); // 19 B per node (sequential path) / 22 B per record (loop-free path)
}

// The two formulations never run at the same time, so their private tables share one region:
//   sequential loop   bucket heads + tails (1 KB) | list of the nodes of 256+ corners
//   loop-free path    2 KB of histogram / bucket tables | 8 B per leaf | best-response corner of every (strip, d1, d2, d3) bin
__host__ __device__ inline size_t qt_union_bytes(int node_cap, int big_cap)
{
  const size_t seq = qt_align16((size_t)2 * kQtBuckets * sizeof(uint16_t)) + qt_align16((size_t)big_cap * sizeof(uint16_t));
  const size_t fast = 2048 + qt_align16((size_t)node_cap * 8) + qt_align16((size_t)kQtMaxBinStrips * kQtBinsPerStrip * sizeof(uint16_t));
  return seq > fast ? seq : fast;
}

// shared memory: node pool / records | per-cell offsets | the union above | keys u32, ia u16, ib u16, responses u8 per list slot
size_t quadtree_smem_bytes(int list_cap, int node_cap, int big_cap, int max_level_cells)
{
  size_t b = qt_pool_bytes(node_cap);
  b += qt_align16((size_t)max_level_cells * sizeof(int));
  b += qt_union_bytes(node_cap, big_cap);
  b += qt_align16((size_t)list_cap * 9);
  return b + 64;
}

struct QtState
{
  QtNodePool np;
  uint16_t *bhead, *btail, *big;
  int nbig;
  uint32_t seq_ctr;
};

__device__ __forceinline__ void qt_push(QtState &q, uint32_t id, uint32_t count, int lane)
{
  // warp-uniform call; lane 0 performs the stores
  if (count >= (uint32_t)kQtBuckets)
  {
    if (lane == 0)
    {
      q.big[q.nbig] = (uint16_t)id;
      q.np.seq[id] = q.seq_ctr;
      q.np.state[id] = 1;
    }
    ++q.nbig;
    ++q.seq_ctr;
    return;
  }
  if (lane == 0)
  {
    const uint32_t t = q.btail[count];
    q.np.next[id] = (uint16_t)kNil;
    q.np.prev[id] = (uint16_t)t;
    if (t == kNil)
      q.bhead[count] = (uint16_t)id;
    else
      q.np.next[t] = (uint16_t)id;
    q.btail[count] = (uint16_t)id;
    q.np.state[id] = 1;
  }
}

// position in the big list of the first (want_max) or last (!want_max) node in multimap order (count desc, FIFO)
__device__ __forceinline__ int qt_big_extreme(const QtState &q, int lane, bool want_max)
{
  unsigned long long best = want_max ? 0ull : ~0ull;
  int best_pos = -1;
  for (int j = lane; j < q.nbig; j += 32)
  {
    const uint32_t id = q.big[j];
    const unsigned long long key = ((unsigned long long)qt_rec_cnt(q.np.rec[id]) << 32) | (unsigned long long)(0xffffffffu - q.np.seq[id]);
    if (want_max ? key >= best : key <= best)
    {
      best = key;
      best_pos = j;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
  {
    const unsigned long long ok = __shfl_xor_sync(kFullMask, best, o);
    const int op = __shfl_xor_sync(kFullMask, best_pos, o);
    const bool take = op >= 0 && (best_pos < 0 || (want_max ? ok > best : ok < best));
    if (take)
    {
      best = ok;
      best_pos = op;
    }
  }
  return best_pos; // keys are unique (seq), so all lanes agree
}

// quadrant of (x, y) inside a node with midlines (mr, mc): 0..3 in the reference's child order, or kDigitDrop on a midline
template <typename T> __device__ __forceinline__ uint32_t qt_quadrant(T x, T y, T mr, T mc)
{
  const int jx = x < mc ? 0 : (x > mc ? 1 : -1);
  const int iy = y < mr ? 0 : (y > mr ? 1 : -1);
  return (jx >= 0 && iy >= 0) ? (uint32_t)(iy * 2 + jx) : kDigitDrop;
}

// Descent key of one corner (strip id + kKeyLevels quadrant digits); cols = strip bounds in 24.40 fixed point.
// Inside a strip [c0, c0 + W) x [0, H) the depth-j nodes are the 2^j x 2^j grid of equal dyadic sub-intervals, so the
// column of the depth-j node holding x is floor((x - c0) * 2^j / W), its low bit is the left/right choice at depth j, and x
// lies on a depth-j midline iff (x - c0) * 2^j / W is an integer: one division per axis replaces the level-by-level descent.
__device__ __forceinline__ uint32_t qt_make_key(uint32_t e, const long long *cols, int K, int roi_h)
{
  const uint32_t xi = e & 0xfffu, yi = (e >> 12) & 0xfffu;
  const long long x = (long long)xi << kFixShift;
  int strip = -1;
  if (yi > 0u && yi < (uint32_t)roi_h)
    for (int k = 0; k < K; ++k)
      if (x > cols[k] && x < cols[k + 1])
      {
        strip = k;
        break;
      }
  if (strip < 0) return kKeyNoStrip << kKeyStripShift;
  const unsigned long long ux = (unsigned long long)(x - cols[strip]) << kKeyLevels, wx = (unsigned long long)(cols[strip + 1] - cols[strip]);
  // floor(ux / wx) < 2^kKeyLevels because the corner lies inside the strip: a float quotient is off by less than one, and one
  // exact 64-bit correction step in either direction replaces the (emulated, ~100-instruction) 64-bit division
  uint32_t qx = (uint32_t)__fdividef((float)ux, (float)wx);
  long long rem = (long long)(ux - (unsigned long long)qx * wx);
  if (rem < 0) --qx, rem += (long long)wx;
  if (rem >= (long long)wx) ++qx, rem -= (long long)wx;
  const bool x_exact = rem == 0;
  const uint32_t uy = yi << kKeyLevels, qy = uy / (uint32_t)roi_h;
  const bool y_exact = qy * (uint32_t)roi_h == uy;
  // first depth at which the corner sits on a midline (kKeyLevels + 1: none within the key)
  const int jdx = x_exact ? kKeyLevels - (__ffs((int)qx) - 1) : kKeyLevels + 1;
  const int jdy = y_exact ? kKeyLevels - (__ffs((int)qy) - 1) : kKeyLevels + 1;
  const int jd = max(1, min(jdx, jdy));
  uint32_t key = (uint32_t)strip << kKeyStripShift;
#pragma unroll
  for (int j = 1; j <= kKeyLevels; ++j)
  {
    const uint32_t d = (((qy >> (kKeyLevels - j)) & 1u) << 1) | ((qx >> (kKeyLevels - j)) & 1u);
    key |= (j < jd ? d : (j == jd ? kDigitDrop : 0u)) << (kKeyStripShift - 3 * j);
  }
  return key;
}

// bounds (24.40 fixed point) of the depth-kKeyLevels node a key leads to
__device__ __forceinline__ void qt_bounds_from_key(uint32_t key, const long long *cols, long long roi_h_fx, long long &r0, long long &r1, long long &c0, long long &c1)
{
  const int strip = (int)(key >> kKeyStripShift);
  r0 = 0;
  r1 = roi_h_fx;
  c0 = cols[strip];
  c1 = cols[strip + 1];
#pragma unroll 1
  for (int j = 1; j <= kKeyLevels; ++j)
  {
    const uint32_t d = (key >> (kKeyStripShift - 3 * j)) & 7u;
    const long long mr = (r0 + r1) >> 1, mc = (c0 + c1) >> 1;
    if (d & 2u)
      r0 = mr;
    else
      r1 = mr;
    if (d & 1u)
      c0 = mc;
    else
      c1 = mc;
  }
}

template <typename IdxT>
__device__ void qt_simulate(const Params &p, const Level &L, QtState &q, const uint32_t *kp, const uint32_t *keys, bool use_keys, const int *bin_start,
                            IdxT *ia, IdxT *ib, int n, int need, int node_cap, int lane, int live, int n_alloc, bool root_pending, int &out_n_alloc,
                            int &out_take)
{
  const unsigned lt_mask = (1u << lane) - 1u;
  QtNodePool &np = q.np;
  int n_free = 0;
  int cursor = kQtBuckets - 1;
  // `live` == the reference's mnNodes: every live node sits in the multimap
  while (live < need && live > 0)
  {
    uint32_t id;
    if (q.nbig > 0)
    {
      const int pos = qt_big_extreme(q, lane, true);
      id = q.big[pos];
      __syncwarp();
      if (lane == 0)
      {
        q.big[pos] = q.big[q.nbig - 1];
        np.state[id] = 0;
      }
      --q.nbig;
    }
    else
    {
      // highest non-empty small bucket at or below the cursor
      for (;;)
      {
        const int b = cursor - lane;
        const bool hit = (b >= 0) && (q.bhead[b] != (uint16_t)kNil);
        const unsigned m = __ballot_sync(kFullMask, hit);
        if (m)
        {
          cursor -= __ffs(m) - 1;
          break;
        }
        cursor -= 32;
        if (cursor < 0) break;
      }
      if (cursor < 0) break; // cannot happen while live > 0
      if (cursor == 1 && !root_pending)
      {
        // Every live node holds exactly one corner and we are still short of `need`: a one-corner node yields at most one
        // one-corner child, so the node count can never grow again and the reference keeps splitting until each corner
        // lands exactly on a midline and vanishes -- the multimap drains and the level returns no keypoints (:151).
        for (int i = lane; i < node_cap; i += 32) np.state[i] = 0;
        live = 0;
        break;
      }
      id = q.bhead[cursor];
      __syncwarp();
      if (lane == 0)
      {
        const uint32_t nx = np.next[id];
        q.bhead[cursor] = (uint16_t)nx;
        if (nx == kNil)
          q.btail[cursor] = (uint16_t)kNil;
        else
          np.prev[nx] = (uint16_t)kNil;
        np.state[id] = 0;
      }
    }
    const uint2 rec = np.rec[id];
    const uint32_t lo = rec.x, cnt = qt_rec_cnt(rec);
    const int buf = qt_rec_buf(rec), depth = qt_rec_depth(rec);
    --live;
    const IdxT *src = buf ? ib : ia;
    IdxT *dst = buf ? ia : ib;
    // Bounds are only needed where the keys end: nodes above depth kKeyLevels never store or load them, a node AT that depth
    // rebuilds them from the key of any of its corners, deeper nodes (and key-less configurations) keep them in the pool.
    const bool keyed = use_keys && depth < kKeyLevels && !root_pending;
    long long r0 = 0, r1 = 0, c0 = 0, c1 = 0;
    if (!keyed)
    {
      if (use_keys && depth == kKeyLevels && cnt > 0)
        qt_bounds_from_key(keys[src[lo]], p.strips_fx + L.strip_off, (long long)L.roi_h << kFixShift, r0, r1, c0, c1);
      else
      {
        r0 = np.r0[id];
        r1 = np.r1[id];
        c0 = np.c0[id];
        c1 = np.c1[id];
      }
    }

    if (root_pending)
    {
      // initSplit (:81-96) for configurations the keys cannot express (more than 31 strips): generic K-way passes
      root_pending = false;
      const int K = L.n_ini;
      const long long *cols = p.strips_fx + L.strip_off;
      uint32_t base = lo;
      for (int k = 0; k < K; ++k)
      {
        uint32_t run = 0;
        for (uint32_t i0 = 0; i0 < cnt; i0 += 32)
        {
          const uint32_t i = i0 + lane;
          bool f = false;
          uint32_t idx = 0;
          if (i < cnt)
          {
            idx = src[lo + i];
            const uint32_t e = kp[idx];
            const long long x = (long long)(e & 0xfffu) << kFixShift, y = (long long)((e >> 12) & 0xfffu) << kFixShift;
            f = x > cols[k] && x < cols[k + 1] && y > r0 && y < r1;
          }
          const unsigned m = __ballot_sync(kFullMask, f);
          if (f) dst[base + run + __popc(m & lt_mask)] = (IdxT)idx;
          run += __popc(m);
        }
        if (run > 0)
        {
          uint32_t cid;
          if (n_free > 0)
            cid = np.free_ids[--n_free];
          else
            cid = n_alloc++;
          if (lane == 0)
          {
            np.r0[cid] = r0;
            np.r1[cid] = r1;
            np.c0[cid] = cols[k];
            np.c1[cid] = cols[k + 1];
            np.rec[cid] = qt_rec(base, run, 0, buf ^ 1);
          }
          qt_push(q, cid, run, lane);
          ++live;
          base += run;
        }
        __syncwarp();
      }
    }
    else
    {
      // split (:60-72): midlines in double, children (row0,col0) (row0,col1) (row1,col0) (row1,col1); corners on a
      // midline belong to no child (strict isIn, ORBExtractor.h:55-62)
      const bool fixed = depth < kFixDepth; // this node splits in fixed point; its children (depth <= kFixDepth) store fixed bounds
      long long mr = 0, mc = 0;             // midlines in the representation of the CHILDREN
      double mr_d = 0.0, mc_d = 0.0;
      if (!keyed)
      {
        if (fixed)
        {
          mr = (r0 + r1) >> 1;
          mc = (c0 + c1) >> 1;
        }
        else
        {
          // depth == kFixDepth holds fixed-point bounds (exactly convertible), deeper nodes hold double bit patterns
          const double scale = 1.0 / (double)(1ll << kFixShift);
          const double dr0 = depth == kFixDepth ? __dmul_rn((double)r0, scale) : __longlong_as_double(r0);
          const double dr1 = depth == kFixDepth ? __dmul_rn((double)r1, scale) : __longlong_as_double(r1);
          const double dc0 = depth == kFixDepth ? __dmul_rn((double)c0, scale) : __longlong_as_double(c0);
          const double dc1 = depth == kFixDepth ? __dmul_rn((double)c1, scale) : __longlong_as_double(c1);
          mr_d = __dmul_rn(__dadd_rn(dr0, dr1), 0.5);
          mc_d = __dmul_rn(__dadd_rn(dc0, dc1), 0.5);
          mr = __double_as_longlong(mr_d);
          mc = __double_as_longlong(mc_d);
        }
      }
      const int shift = kKeyStripShift - 3 * (depth + 1);
      uint32_t t0 = 0, t1 = 0, t2 = 0, t3 = 0;
      auto digit_of = [&](uint32_t idx) -> uint32_t {
        if (keyed) return (keys[idx] >> shift) & 7u;
        const uint32_t e = kp[idx];
        if (fixed) return qt_quadrant((long long)(e & 0xfffu) << kFixShift, (long long)((e >> 12) & 0xfffu) << kFixShift, mr, mc);
        return qt_quadrant((double)(e & 0xfffu), (double)((e >> 12) & 0xfffu), mr_d, mc_d);
      };
      // The block sorted the corners by (strip, digits of depths 1..3) up front: the children of nodes above depth 3 are
      // contiguous sub-ranges of the parent's range, their sizes come from the bin table, nothing moves.
      const bool presorted = bin_start != nullptr && keyed && depth < kQtPresort;
      if (presorted)
      {
        // base-5 prefix of the node (strip, digits 1..depth) from the key of any of its corners
        const uint32_t key0 = keys[src[lo]];
        int prefix = (int)(key0 >> kKeyStripShift);
        for (int j = 1; j <= depth; ++j) prefix = prefix * 5 + (int)((key0 >> (kKeyStripShift - 3 * j)) & 7u);
        int span = 1; // bins below one child: 5^(kQtPresort - 1 - depth)
        for (int j = depth + 1; j < kQtPresort; ++j) span *= 5;
        const int b = prefix * 5 * span;
        t0 = (uint32_t)(bin_start[b + span] - bin_start[b]);
        t1 = (uint32_t)(bin_start[b + 2 * span] - bin_start[b + span]);
        t2 = (uint32_t)(bin_start[b + 3 * span] - bin_start[b + 2 * span]);
        t3 = (uint32_t)(bin_start[b + 4 * span] - bin_start[b + 3 * span]);
      }
      else if (cnt <= 32)
      {
        // the common case: the whole node fits one warp pass
        uint32_t d = kDigitDrop, idx = 0;
        if ((uint32_t)lane < cnt)
        {
          idx = src[lo + lane];
          d = digit_of(idx);
        }
        const unsigned m0 = __ballot_sync(kFullMask, d == 0), m1 = __ballot_sync(kFullMask, d == 1);
        const unsigned m2 = __ballot_sync(kFullMask, d == 2), m3 = __ballot_sync(kFullMask, d == 3);
        t0 = __popc(m0);
        t1 = __popc(m1);
        t2 = __popc(m2);
        t3 = __popc(m3);
        const unsigned mm = d == 0 ? m0 : (d == 1 ? m1 : (d == 2 ? m2 : m3));
        const uint32_t bb = d == 0 ? 0u : (d == 1 ? t0 : (d == 2 ? t0 + t1 : t0 + t1 + t2));
        if (d != kDigitDrop) dst[lo + bb + __popc(mm & lt_mask)] = (IdxT)idx;
      }
      else
      {
        // four chunks of 32 per iteration: the (index -> key) load chains of the chunks are independent, which is what
        // hides the shared-memory latency on this single warp
        for (uint32_t i0 = 0; i0 < cnt; i0 += 128)
        {
          uint32_t d[4];
#pragma unroll
          for (int u = 0; u < 4; ++u)
          {
            const uint32_t i = i0 + 32 * u + lane;
            d[u] = i < cnt ? digit_of(src[lo + i]) : kDigitDrop;
          }
#pragma unroll
          for (int u = 0; u < 4; ++u)
          {
            t0 += __popc(__ballot_sync(kFullMask, d[u] == 0));
            t1 += __popc(__ballot_sync(kFullMask, d[u] == 1));
            t2 += __popc(__ballot_sync(kFullMask, d[u] == 2));
            t3 += __popc(__ballot_sync(kFullMask, d[u] == 3));
          }
        }
        const uint32_t b0 = lo, b1 = b0 + t0, b2 = b1 + t1, b3 = b2 + t2;
        uint32_t q0 = 0, q1 = 0, q2 = 0, q3 = 0;
        for (uint32_t i0 = 0; i0 < cnt; i0 += 128)
        {
          uint32_t d[4];
          IdxT idx[4];
#pragma unroll
          for (int u = 0; u < 4; ++u)
          {
            const uint32_t i = i0 + 32 * u + lane;
            d[u] = kDigitDrop;
            idx[u] = 0;
            if (i < cnt)
            {
              idx[u] = src[lo + i];
              d[u] = digit_of(idx[u]);
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u)
          {
            const unsigned m0 = __ballot_sync(kFullMask, d[u] == 0), m1 = __ballot_sync(kFullMask, d[u] == 1);
            const unsigned m2 = __ballot_sync(kFullMask, d[u] == 2), m3 = __ballot_sync(kFullMask, d[u] == 3);
            if (d[u] == 0) dst[b0 + q0 + __popc(m0 & lt_mask)] = idx[u];
            if (d[u] == 1) dst[b1 + q1 + __popc(m1 & lt_mask)] = idx[u];
            if (d[u] == 2) dst[b2 + q2 + __popc(m2 & lt_mask)] = idx[u];
            if (d[u] == 3) dst[b3 + q3 + __popc(m3 & lt_mask)] = idx[u];
            q0 += __popc(m0);
            q1 += __popc(m1);
            q2 += __popc(m2);
            q3 += __popc(m3);
          }
        }
      }
      // children: lane k < 4 fills the record of child k; ids come from the free stack first, then fresh slots
      const uint32_t tc[4] = {t0, t1, t2, t3};
      const uint32_t bs[4] = {lo, lo + t0, lo + t0 + t1, lo + t0 + t1 + t2};
      const int ne[4] = {t0 > 0, t1 > 0, t2 > 0, t3 > 0};
      const int rk[4] = {0, ne[0], ne[0] + ne[1], ne[0] + ne[1] + ne[2]};
      const int n_new = rk[3] + ne[3];
      uint32_t cid[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) cid[k] = rk[k] < n_free ? (uint32_t)np.free_ids[n_free - 1 - rk[k]] : (uint32_t)(n_alloc + rk[k] - n_free);
      {
        const int k = lane & 3;
        const uint32_t my_t = k == 0 ? tc[0] : (k == 1 ? tc[1] : (k == 2 ? tc[2] : tc[3]));
        const uint32_t my_b = k == 0 ? bs[0] : (k == 1 ? bs[1] : (k == 2 ? bs[2] : bs[3]));
        const uint32_t c = k == 0 ? cid[0] : (k == 1 ? cid[1] : (k == 2 ? cid[2] : cid[3]));
        if (lane < 4 && my_t > 0)
        {
          if (!keyed)
          {
            long long pr0 = r0, pr1 = r1, pc0 = c0, pc1 = c1; // parent bounds in the children's representation
            if (depth == kFixDepth)
            {
              const double scale = 1.0 / (double)(1ll << kFixShift);
              pr0 = __double_as_longlong(__dmul_rn((double)r0, scale));
              pr1 = __double_as_longlong(__dmul_rn((double)r1, scale));
              pc0 = __double_as_longlong(__dmul_rn((double)c0, scale));
              pc1 = __double_as_longlong(__dmul_rn((double)c1, scale));
            }
            np.r0[c] = (k & 2) ? mr : pr0;
            np.r1[c] = (k & 2) ? pr1 : mr;
            np.c0[c] = (k & 1) ? mc : pc0;
            np.c1[c] = (k & 1) ? pc1 : mc;
          }
          np.rec[c] = qt_rec(my_b, my_t, depth + 1, presorted ? buf : buf ^ 1);
        }
      }
      const int from_free = min(n_free, n_new);
      n_alloc += n_new - from_free;
      n_free -= from_free;
      __syncwarp();
      // multimap insertion order == child order; it only matters between children of EQUAL count (same bucket), so when
      // the non-empty children have pairwise distinct counts below 256 the four pushes go to four different buckets and
      // lanes 0..3 do them concurrently
      const bool distinct = (t0 != t1 || t0 == 0) && (t0 != t2 || t0 == 0) && (t0 != t3 || t0 == 0) && (t1 != t2 || t1 == 0) && (t1 != t3 || t1 == 0) &&
                            (t2 != t3 || t2 == 0) && max(max(t0, t1), max(t2, t3)) < (uint32_t)kQtBuckets;
      if (distinct)
      {
        const int k = lane & 3;
        const uint32_t my_t = k == 0 ? t0 : (k == 1 ? t1 : (k == 2 ? t2 : t3));
        const uint32_t c = k == 0 ? cid[0] : (k == 1 ? cid[1] : (k == 2 ? cid[2] : cid[3]));
        if (lane < 4 && my_t > 0)
        {
          const uint32_t tl = q.btail[my_t];
          np.next[c] = (uint16_t)kNil;
          np.prev[c] = (uint16_t)tl;
          if (tl == kNil)
            q.bhead[my_t] = (uint16_t)c;
          else
            np.next[tl] = (uint16_t)c;
          q.btail[my_t] = (uint16_t)c;
          np.state[c] = 1;
        }
        live += n_new;
      }
      else
      {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (tc[k] > 0)
          {
            qt_push(q, cid[k], tc[k], lane);
            ++live;
          }
      }
    }
    // the popped node's slot can be reused
    if (lane == 0) np.free_ids[n_free] = (uint16_t)id;
    ++n_free;
    __syncwarp();
  }

  // nodes2kpoints (:182-192): only the first min(need, |M|) entries in (count desc, FIFO) order are used; the surplus
  // sits at the tails of the lowest buckets (and, if those run out, at the low end of the big-node list)
  const int take = min(need, live);
  int excl = live - take;
  int b = 0;
  while (excl > 0 && b < kQtBuckets)
  {
    const uint32_t t = q.btail[b];
    if (t == kNil)
    {
      ++b;
      continue;
    }
    __syncwarp();
    if (lane == 0)
    {
      np.state[t] = 2;
      const uint32_t pv = np.prev[t];
      q.btail[b] = (uint16_t)pv;
      if (pv == kNil) q.bhead[b] = (uint16_t)kNil;
    }
    --excl;
    __syncwarp();
  }
  while (excl > 0 && q.nbig > 0)
  {
    const int pos = qt_big_extreme(q, lane, false);
    __syncwarp();
    if (lane == 0)
    {
      np.state[q.big[pos]] = 2;
      q.big[pos] = q.big[q.nbig - 1];
    }
    --q.nbig;
    --excl;
    __syncwarp();
  }
  out_n_alloc = n_alloc;
  out_take = take;
}

template <typename IdxT>
__device__ void qt_select(const QtNodePool &np, const uint32_t *kp, const IdxT *ia, const IdxT *ib, uint32_t *flag, int n, int n_slots, int tid)
{
  // best response per surviving node (getFeature :103-117: strict '>' over the node's list, whose order is ascending
  // detection index, i.e. the lowest index among the maxima wins; default index 0 when no response is positive)
  for (int s = tid; s < n_slots; s += kQtThreads)
  {
    if (np.state[s] != 1) continue;
    const uint2 rec = np.rec[s];
    const IdxT *arr = qt_rec_buf(rec) ? ib : ia;
    const uint32_t lo = rec.x, cnt = qt_rec_cnt(rec);
    uint32_t best = 0, best_i = 0;
    for (uint32_t i = 0; i < cnt; ++i)
    {
      const uint32_t idx = arr[lo + i];
      const uint32_t r = kp[idx] >> 24;
      if (r > best || (r == best && r > 0 && idx < best_i))
      {
        best = r;
        best_i = idx;
      }
    }
    if ((int)best_i < n) flag[best_i] = 1u;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// K3 fast path: Quadtree::split() without the priority loop.
//   A child never holds more corners than its parent, so the multimap's pop sequence is the list of ALL tree nodes ordered
//   by (count desc, pop position of the parent, child index), cut at the first prefix whose running node count reaches
//   `need`; unrolled, two nodes of equal count compare by the counts of their ancestors (parent first, +inf for the root),
//   then by their path.  With D[c] = sum over the nodes of c corners of (non-empty children - 1), the loop stops inside the
//   bucket c* = the largest c whose suffix sum lifts the node count to `need`, and it pops every node above c* plus a prefix of
//   bucket c* in that order.  So the block builds the tree level by level instead of pop by pop, and only where it can matter:
//     V1  nodes of depths 0..2 straight from the bin table of the presort (counts of every (strip, d1, d2, d3) prefix)
//     V2  level-synchronous descent from depth 3: a node is split (a thread partitions its corners by the next key digit)
//         only if its count reaches the running LOWER BOUND of c* (the crossing computed from the deltas known so far: an
//         unsplit node is smaller than the bound, so the suffix sums at and above the bound are already exact)
//     V3  exact c*; pop rank of every record of count >= c* (bucket lists + ancestor-count chains) -> how much of bucket c* pops
//     V4  leaves = children of popped records that did not pop; best response per leaf; the surplus beyond `need` (at most 3)
//         leaves from the END of the (count desc, insertion) order
//   It bails out (returns false: the sequential loop runs instead) exactly where the keys do not decide: a node at the key depth
//   that would have to be split, a popped node whose corners all sit on split lines (negative delta: the running count is not
//   monotone), c* >= 255, record capacity.  scripts/devtests/quadtree_parallel_model.py is the CPU model of this formulation.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kFpWarps = kQtThreads / 32;
constexpr int kFpSmall = 8;        // node counts below this are accumulated in per-warp counters (the hot histogram bins)
constexpr int kFpRecBytes = 22;    // shared memory per record
static_assert(kFpRecBytes == 22, "qt_pool_bytes");
constexpr uint32_t kFpNone = 0xffffu;
constexpr uint8_t kFpActive = 1, kFpPopped = 2, kFpKidsBuf = 0x80;

// warp-aggregated slot allocation: the lanes that execute this together take consecutive indices with ONE shared-memory atomic
__device__ __forceinline__ int fp_alloc(int *counter)
{
  const unsigned act = __activemask();
  const int lane = threadIdx.x & 31, leader = __ffs(act) - 1;
  int base = 0;
  if (lane == leader) base = atomicAdd(counter, __popc(act));
  base = __shfl_sync(act, base, leader);
  return base + __popc(act & ((1u << lane) - 1u));
}

// views into the CTA's shared memory (derived from a few numbers; a by-value table of pointers would live in local memory)
struct QtFast
{
  uint8_t *pool;   // records: u16 lo cnt par rank best t0 t1 t2 t3 [nc] | u8 kidrec meta delta state [nc]      (22 B per record)
  uint8_t *lists;  // keys u32[cap] | ia u16[cap] | ib u16[cap] | resp u8[cap]
  int *scr;        // 2 KB: D[256] during the descent, start[256] + cursor[256] during the ranking
  uint8_t *lf;     // leaves: I u32[nc] | best u16[nc] | cnt u16[nc]   (the ranking keeps its bucket list and deltas here before)
  uint16_t *bin_best; // best-response corner of every (strip, d1, d2, d3) bin (kFpNone: empty)
  int cap, nc;
  __device__ __forceinline__ uint32_t *keys() const { return (uint32_t *)lists; }
  __device__ __forceinline__ uint16_t *arr(int buf) const { return (uint16_t *)(lists + (4 + 2 * (size_t)buf) * cap); }
  __device__ __forceinline__ const uint8_t *resp() const { return lists + 8 * (size_t)cap; } // response (FAST score) by corner
  // layout: kidrec u8[nc rounded up to 16] (first: it takes 32-bit atomics) | nine u16 arrays | three u8 arrays
  __device__ __forceinline__ size_t pad() const { return ((size_t)nc + 15) & ~(size_t)15; }
  __device__ __forceinline__ uint16_t *u16(int k) const { return (uint16_t *)(pool + pad()) + (size_t)k * nc; }
  __device__ __forceinline__ uint16_t *r_lo() const { return u16(0); }   // first position of its corners (table records: first bin)
  __device__ __forceinline__ uint16_t *r_cnt() const { return u16(1); }
  __device__ __forceinline__ uint16_t *r_par() const { return u16(2); }
  __device__ __forceinline__ uint16_t *r_rank() const { return u16(3); }
  __device__ __forceinline__ uint16_t *r_best() const { return u16(4); } // best-response corner, taken while its list was intact
  __device__ __forceinline__ uint16_t *r_t(int k) const { return u16(5 + k); }
  __device__ __forceinline__ uint8_t *r_kidrec() const { return pool; } // children that have a record of their own
  __device__ __forceinline__ uint8_t *r_meta() const { return pool + pad() + 18 * (size_t)nc; }   // depth << 4 | child << 1 | buffer of its corners
  __device__ __forceinline__ int8_t *r_delta() const { return (int8_t *)(pool + pad() + 19 * (size_t)nc); }
  __device__ __forceinline__ uint8_t *r_state() const { return pool + pad() + 20 * (size_t)nc; }
  __device__ __forceinline__ uint32_t *lf_I() const { return (uint32_t *)lf; }
  __device__ __forceinline__ uint16_t *lf_best() const { return (uint16_t *)(lf + 4 * (size_t)nc); }
  __device__ __forceinline__ uint16_t *lf_cnt() const { return (uint16_t *)(lf + 6 * (size_t)nc); }
};

// a child announces its record to the parent (several threads may do so for one parent: atomic on the containing word)
__device__ __forceinline__ void fp_mark_kid(const QtFast &f, uint32_t par, uint32_t child)
{
  atomicOr((unsigned int *)(f.r_kidrec() + (par & ~3u)), 1u << (8u * (par & 3u) + child));
}

// best response over the bins [b0, b1): lowest corner index among the maxima (getFeature :103-117; bins hold their own best)
__device__ __forceinline__ uint32_t fp_best_of_bins(const QtFast &f, int b0, int b1)
{
  const uint8_t *resp = f.resp();
  uint32_t best = 0, best_i = 0;
  for (int b = b0; b < b1; ++b)
  {
    const uint32_t idx = f.bin_best[b];
    if (idx == kFpNone) continue;
    const uint32_t r = resp[idx];
    if (r > best || (r == best && r > 0 && idx < best_i)) best = r, best_i = idx;
  }
  return best_i;
}

// equal counts: does record u pop before record v?  (ancestor counts, parent first; the root -- record 0 -- counts as +inf;
// then the child index below the first common ancestor)
__device__ __forceinline__ bool fp_chain_before(const QtFast &f, uint32_t u, uint32_t v)
{
  uint32_t a = u, b = v;
  for (;;)
  {
    const uint32_t pa = a, pb = b;
    a = f.r_par()[a];
    b = f.r_par()[b];
    if (a == b) return ((f.r_meta()[pa] >> 1) & 7u) < ((f.r_meta()[pb] >> 1) & 7u);
    const uint32_t ca = a == 0 ? 0x10000u : f.r_cnt()[a], cb = b == 0 ? 0x10000u : f.r_cnt()[b];
    if (ca != cb) return ca > cb;
  }
}

// block barrier of the loop-free path: thread-dependent branches (one thread publishing a result, lanes with and without work)
// precede most of them, so the warp is explicitly reconverged before the aligned barrier
__device__ __forceinline__ void fp_sync()
{
  __syncwarp();
  __syncthreads();
}

__device__ __noinline__ bool qt_fast_path(uint8_t *pool, uint8_t *lists, int *scr, uint8_t *lf, uint16_t *bin_best, const int *bin_start, int cap, int nc, int K,
                                          int n, int need, int *s_warp, unsigned long long *stats)
{
  __shared__ int s_live0, s_dbig, s_neg, s_deep, s_cstar, s_before, s_first, s_nrec, s_f1, s_k, s_nleaf, s_over;
  __shared__ int s_small[kFpWarps][kFpSmall];
  __shared__ uint16_t s_tab[kQtMaxBinStrips * 31]; // record of every depth 0..2 prefix (kFpNone: no node)
  __shared__ unsigned long long s_amax;
  QtFast f;
  f.pool = pool, f.lists = lists, f.scr = scr, f.lf = lf, f.bin_best = bin_best, f.cap = cap, f.nc = nc;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  enum { kRun = 0, kEmpty = 1, kNoPop = 2, kBail = 3 };
  int *D = f.scr;
  long long t_prev = clock64();
  auto tick = [&](int phase) {
    if (tid == 0 && stats)
    {
      const long long t = clock64();
      atomicAdd(&stats[2 + phase], (unsigned long long)(t - t_prev));
      t_prev = t;
    }
  };
  auto add_delta = [&](int cnt, int delta) {
    if (delta < 0) atomicMax(&s_neg, cnt);
    if (delta == 0) return;
    if (cnt < kFpSmall)
      atomicAdd(&s_small[wid][cnt], delta);
    else if (cnt < 256)
      atomicAdd(&D[cnt], delta);
    else
      atomicAdd(&s_dbig, delta);
  };
  // The crossing of the node count over `need` in the deltas known so far: thread t <-> count c = 255 - t,
  // after(c) = live0 + sum of the deltas of all nodes of >= c corners.  s_first = 255 - c* (0x7fffffff: none), s_before = after(c* + 1).
  auto find_cross = [&]() {
    const int c = 255 - tid;
    int d = 0;
    if (c >= kFpSmall)
      d = D[c];
    else if (c >= 2)
      for (int w = 0; w < kFpWarps; ++w) d += s_small[w][c];
    const int inc = warp_inclusive_scan(d, lane);
    if (tid == 0) s_first = 0x7fffffff;
    if (lane == 31) s_warp[wid] = inc;
    fp_sync();
    int base = 0;
    for (int w = 0; w < wid; ++w) base += s_warp[w];
    const int after = s_live0 + s_dbig + base + inc;
    if (c >= 2 && after >= need) atomicMin(&s_first, tid);
    fp_sync();
    if (tid == s_first)
    {
      s_cstar = c;
      s_before = after - d;
    }
    if (tid == 0 && s_first == 0x7fffffff) s_cstar = 0;
    fp_sync();
  };

  // ---- V0: accumulators, the root record, the strips
  for (int i = tid; i < 256; i += kQtThreads) D[i] = 0;
  if (tid < kFpWarps * kFpSmall) (&s_small[0][0])[tid] = 0;
  for (int i = tid; i < kQtMaxBinStrips * 31; i += kQtThreads) s_tab[i] = (uint16_t)kFpNone;
  if (tid == 0)
  {
    s_live0 = 0, s_dbig = 0, s_neg = 0, s_deep = 0, s_cstar = 0, s_before = 0, s_nrec = 1, s_k = 0, s_nleaf = 0, s_over = 0;
    s_amax = 0ull;
    f.r_cnt()[0] = 0xffffu;
    f.r_par()[0] = (uint16_t)kFpNone;
    f.r_meta()[0] = 0;
    f.r_state()[0] = kFpActive | kFpPopped; // the loop always pops the root first (need >= 2)
    f.r_rank()[0] = 0;
  }
  for (int i = tid; i < nc; i += kQtThreads) f.r_kidrec()[i] = 0;
  fp_sync();
  if (tid < K) atomicAdd(&s_live0, bin_start[(tid + 1) * kQtBinsPerStrip] > bin_start[tid * kQtBinsPerStrip] ? 1 : 0);
  fp_sync();
  const int live0 = s_live0;
  int mode = live0 == 0 ? kEmpty : (live0 >= need ? kNoPop : kRun);
  int cstar = 0;

  // ---- V0b: every (strip, d1, d2, d3) bin once: its best-response corner (leaves are read off these: a node's own list may be
  // overwritten by its grandchildren later), and -- the bin being a depth-3 node when it holds >= 2 corners -- the number of its
  // children (the fourth key digits present), i.e. the deltas one level below the table
  {
    const uint32_t *keys = f.keys();
    const uint8_t *resp = f.resp();
    for (int j = tid; j < K * kQtBinsPerStrip; j += kQtThreads)
    {
      const int lo = bin_start[j], cnt = bin_start[j + 1] - lo;
      const uint16_t *src = f.arr(0) + lo;
      uint32_t mask = 0, best = 0, best_i = 0;
      for (int i = 0; i < cnt; ++i)
      {
        const uint32_t idx = src[i], r = resp[idx];
        mask |= 1u << ((keys[idx] >> (kKeyStripShift - 12)) & 7u);
        if (r > best || (r == best && r > 0 && idx < best_i)) best = r, best_i = idx;
      }
      f.bin_best[j] = best > 0 ? (uint16_t)best_i : (uint16_t)kFpNone; // no positive response: getFeature's default (index 0) applies

      const bool node = !(j % 5 == 4 || (j / 5) % 5 == 4 || (j / 25) % 5 == 4) && cnt >= 2;
      if (node && mode == kRun) add_delta(cnt, __popc(mask & 15u) - 1);
    }
  }
  fp_sync();

  if (mode == kRun)
  {
    // ---- V1: the nodes of depths 0..2 from the bin table (thread <-> prefix; depth by depth: a record links to its parent's)
    int tab0 = 0, pow5 = 1; // first table slot of the depth, 5^depth
    for (int d = 0; d <= 2; ++d)
    {
      const int span = d == 0 ? 125 : (d == 1 ? 25 : 5), w = span / 5;
      for (int j = tid; j < K * pow5; j += kQtThreads)
      {
        const int g_last = j % 5, g_prev = (j / 5) % 5; // a prefix through a "split line" digit (4) is not a node
        if (d >= 1 && g_last == 4) continue;
        if (d >= 2 && g_prev == 4) continue;
        const int B = j * span, lo = bin_start[B], cnt = bin_start[B + span] - lo;
        if (cnt < 2) continue;
        int t[4], ne = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
        {
          t[k] = bin_start[B + (k + 1) * w] - bin_start[B + k * w];
          ne += t[k] > 0;
        }
        const int idx = fp_alloc(&s_nrec);
        if (idx >= nc)
        {
          s_over = 1;
          continue;
        }
        const uint32_t par = d == 0 ? 0u : (uint32_t)s_tab[tab0 - pow5 / 5 * K + j / 5], child = (uint32_t)(d == 0 ? j : g_last);
        f.r_lo()[idx] = (uint16_t)B; // table records keep their first bin (their corners are the bins [B, B + span))
        f.r_cnt()[idx] = (uint16_t)cnt;
        f.r_par()[idx] = (uint16_t)par;
        f.r_meta()[idx] = (uint8_t)((d << 4) | (child << 1));
        f.r_delta()[idx] = (int8_t)(ne - 1);
        f.r_state()[idx] = kFpActive; // (its best response, should it end up as a leaf, is read off the bins then)
        fp_mark_kid(f, par, child);
#pragma unroll
        for (int k = 0; k < 4; ++k) f.r_t(k)[idx] = (uint16_t)t[k];
        s_tab[tab0 + j] = (uint16_t)idx;
        add_delta(cnt, ne - 1);
      }
      fp_sync();
      tab0 += K * pow5;
      pow5 *= 5;
    }
    tick(0);

    // ---- V2: descent from depth 3, level by level.  The deltas are always known ONE level below the records (a cheap count-only
    // look at the next key digit of every child), so the bound that decides which children get a record -- and will be split --
    // already includes them: bound = the crossing computed from all nodes down to that level, a lower bound of c*.
    const uint32_t *keys = f.keys();
    const uint8_t *resp = f.resp();
    int f0 = s_nrec; // first depth-3 record: read by every thread BEFORE the barriers of find_cross, i.e. before anybody allocates again
    find_cross();
    int bound = max(2, s_cstar); // no crossing yet: every node of >= 2 corners may matter
    for (int j = tid; j < K * kQtBinsPerStrip; j += kQtThreads)
    {
      if (j % 5 == 4 || (j / 5) % 5 == 4 || (j / 25) % 5 == 4) continue;
      const int lo = bin_start[j], cnt = bin_start[j + 1] - lo;
      if (cnt < bound) continue;
      const int idx = fp_alloc(&s_nrec);
      if (idx >= nc)
      {
        s_over = 1;
        continue;
      }
      const uint32_t par = s_tab[6 * K + j / 5]; // the depth-2 prefix
      f.r_lo()[idx] = (uint16_t)lo;
      f.r_cnt()[idx] = (uint16_t)cnt;
      f.r_par()[idx] = (uint16_t)par;
      f.r_meta()[idx] = (uint8_t)((3 << 4) | ((j % 5) << 1));
      f.r_state()[idx] = 0;
      f.r_best()[idx] = f.bin_best[j] == kFpNone ? (uint16_t)0 : f.bin_best[j];
      fp_mark_kid(f, par, (uint32_t)(j % 5));
    }
    fp_sync();
    if (tid == 0) s_f1 = s_nrec;
    fp_sync();
    for (int level = 3; level <= 8; ++level)
    {
      const int f1 = min(s_f1, nc);
      if (f1 <= f0 || s_over) break; // uniform
      // pass A: split every record of this level (stable 4-way partition by the next digit into the other index array) and
      // look one digit further into its children
      const int shift = kKeyStripShift - 3 * (level + 1);
      for (int v = f0 + tid; v < f1; v += kQtThreads)
      {
        const int cnt = f.r_cnt()[v], lo = f.r_lo()[v], buf = f.r_meta()[v] & 1;
        const uint16_t *src = f.arr(buf) + lo;
        uint16_t *dst = f.arr(buf ^ 1);
        int c0 = 0, c1 = 0, c2 = 0, c3 = 0;
        for (int i = 0; i < cnt; ++i)
        {
          const uint32_t dg = (keys[src[i]] >> shift) & 7u;
          c0 += dg == 0, c1 += dg == 1, c2 += dg == 2, c3 += dg == 3;
        }
        int o0 = lo, o1 = o0 + c0, o2 = o1 + c1, o3 = o2 + c2;
        uint32_t m0 = 0, m1 = 0, m2 = 0, m3 = 0; // digits (level + 2) present in each child
        uint32_t best = 0, best_i = 0;
        for (int i = 0; i < cnt; ++i)
        {
          const uint32_t idx = src[i], key = keys[idx], dg = (key >> shift) & 7u;
          if (level > 3)
          { // its own best response, while the list is intact (depth-3 records took theirs from the bin)
            const uint32_t r = resp[idx];
            if (r > best || (r == best && r > 0 && idx < best_i)) best = r, best_i = idx;
          }
          const uint32_t nx = level < 8 ? 1u << ((key >> (shift - 3)) & 7u) : 0u;
          if (dg == 0) dst[o0++] = (uint16_t)idx, m0 |= nx;
          if (dg == 1) dst[o1++] = (uint16_t)idx, m1 |= nx;
          if (dg == 2) dst[o2++] = (uint16_t)idx, m2 |= nx;
          if (dg == 3) dst[o3++] = (uint16_t)idx, m3 |= nx;
        }
        const int ne = (c0 > 0) + (c1 > 0) + (c2 > 0) + (c3 > 0);
        f.r_t(0)[v] = (uint16_t)c0, f.r_t(1)[v] = (uint16_t)c1, f.r_t(2)[v] = (uint16_t)c2, f.r_t(3)[v] = (uint16_t)c3;
        f.r_delta()[v] = (int8_t)(ne - 1);
        f.r_state()[v] = (uint8_t)(kFpActive | ((buf ^ 1) ? kFpKidsBuf : 0));
        if (level > 3) f.r_best()[v] = (uint16_t)best_i;
        const int t[4] = {c0, c1, c2, c3};
        const uint32_t mk[4] = {m0, m1, m2, m3};
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (t[k] >= 2)
          {
            if (level == 8)
              atomicMax(&s_deep, t[k]); // a node AT the key depth with >= 2 corners: the keys cannot split it
            else
              add_delta(t[k], __popc(mk[k] & 15u) - 1);
          }
      }
      fp_sync();
      if (level == 8) break; // uniform
      find_cross();
      bound = max(bound, max(2, s_cstar));
      // pass B: records for the children that may still pop
      for (int v = f0 + tid; v < f1; v += kQtThreads)
      {
        const int buf = f.r_meta()[v] & 1;
        int base = f.r_lo()[v];
#pragma unroll
        for (int k = 0; k < 4; ++k)
        {
          const int tk = f.r_t(k)[v];
          if (tk >= bound)
          {
            const int idx = fp_alloc(&s_nrec);
            if (idx >= nc)
              s_over = 1;
            else
            {
              f.r_lo()[idx] = (uint16_t)base;
              f.r_cnt()[idx] = (uint16_t)tk;
              f.r_par()[idx] = (uint16_t)v;
              f.r_meta()[idx] = (uint8_t)(((level + 1) << 4) | (k << 1) | (buf ^ 1));
              f.r_state()[idx] = 0;
              f.r_kidrec()[v] |= (uint8_t)(1u << k);
            }
          }
          base += tk;
        }
      }
      fp_sync();
      f0 = f1;
      if (tid == 0) s_f1 = s_nrec;
      fp_sync();
    }
    if (s_over || s_nrec > nc) return false; // uniform: more records than the pool holds
    tick(1);

    // ---- V3: exact c*
    find_cross();
    cstar = s_cstar;
    {
      const int hard = max(s_neg, s_deep);
      if (live0 + s_dbig >= need)
        mode = kBail; // the loop stops among the nodes of 256+ corners
      else if (cstar == 0)
        mode = hard >= 2 ? kBail : kEmpty; // starved: the multimap drains (src/ORBExtractor.cc:151), 0 keypoints
      else if (cstar <= hard || cstar >= 255 || cstar < bound)
        mode = kBail;
    }
    if (mode == kBail) return false; // uniform (shared values)
    tick(2);
  }

  const int nrec = mode == kRun ? s_nrec : 1;

  if (mode == kRun)
  {
    // ---- V3b: pop rank of every record of >= c* corners = records in higher buckets + position inside its own bucket.
    // start[b] = records in buckets above b (thread t <-> bucket 255 - t); list = those records grouped by bucket.
    int *start = f.scr, *cursor = f.scr + 256; // D is dead
    uint16_t *list = (uint16_t *)f.lf;          // [<= nrec]
    uint16_t *dlt = list + nc;                  // [bucket c*] deltas in pop order
    fp_sync();
    for (int i = tid; i < 512; i += kQtThreads) f.scr[i] = 0;
    fp_sync();
    auto in_S = [&](int v) { return (f.r_state()[v] & kFpActive) && (int)f.r_cnt()[v] >= cstar; };
    for (int v = 1 + tid; v < nrec; v += kQtThreads)
      if (in_S(v)) atomicAdd(&cursor[min((int)f.r_cnt()[v], 255)], 1); // cursor = bucket sizes for now
    fp_sync();
    {
      const int b = 255 - tid;
      const int h = cursor[b];
      const int inc = warp_inclusive_scan(h, lane);
      if (lane == 31) s_warp[wid] = inc;
      fp_sync();
      int base = 0;
      for (int w = 0; w < wid; ++w) base += s_warp[w];
      start[b] = base + inc - h;
      fp_sync();
      cursor[b] = base + inc - h;
    }
    fp_sync();
    for (int v = 1 + tid; v < nrec; v += kQtThreads)
      if (in_S(v)) list[atomicAdd(&cursor[min((int)f.r_cnt()[v], 255)], 1)] = (uint16_t)v;
    fp_sync();
    const int R0 = start[cstar], mb = cursor[cstar] - R0; // cursor[b] = end of bucket b now
    for (int v = 1 + tid; v < nrec; v += kQtThreads)
    {
      if (!in_S(v)) continue;
      const uint32_t cv = f.r_cnt()[v];
      const int b = min((int)cv, 255);
      const int j0 = start[b], j1 = cursor[b];
      int r = j0;
      for (int j = j0; j < j1; ++j)
      {
        const uint32_t u = list[j];
        if (u == (uint32_t)v) continue;
        const uint32_t cu = f.r_cnt()[u]; // differs only inside the 255+ bucket
        r += cu != cv ? (cu > cv) : fp_chain_before(f, u, (uint32_t)v);
      }
      f.r_rank()[v] = (uint16_t)(r + 1); // the root popped first
      if ((int)cv == cstar) dlt[r - R0] = (uint16_t)f.r_delta()[v]; // all >= 0 here (c* lies above every negative delta)
    }
    fp_sync();
    if (wid == 0)
    {
      int run = s_before, k = 0;
      for (int j0 = 0; j0 < mb; j0 += 32)
      {
        const int j = j0 + lane;
        const int val = j < mb ? (int)dlt[j] : 0;
        const int inc = warp_inclusive_scan(val, lane);
        const bool pops = j < mb && run + inc - val < need; // the loop tests the node count BEFORE every pop
        const unsigned pm = __ballot_sync(kFullMask, pops);
        k += __popc(pm);
        run += __shfl_sync(kFullMask, inc, 31);
        if (pm != kFullMask) break;
      }
      if (lane == 0) s_k = k;
    }
    fp_sync();
    const int k = s_k;
    for (int v = 1 + tid; v < nrec; v += kQtThreads)
    {
      if (!in_S(v)) continue;
      if ((int)f.r_cnt()[v] > cstar || (int)f.r_rank()[v] - 1 - R0 < k)
      {
        f.r_state()[v] |= kFpPopped; // its children stand in for it
      }
    }
    fp_sync();
    tick(3);
  }

  // ---- V4: leaves = the children of popped records (the root included) that did not pop.  A child WITH a record announces itself
  // (its best response was taken while its list was intact); children without one -- single corners, nodes below the bound -- are
  // read by the parent: from the bins under a table record, from the (never overwritten) list of an unsplit child otherwise.
  if (mode != kEmpty)
  {
    const uint8_t *resp = f.resp();
    auto emit = [&](uint32_t best_i, int cnt, uint32_t key) {
      const int li = fp_alloc(&s_nleaf);
      if (li < nc)
      {
        f.lf_best()[li] = (uint16_t)best_i;
        f.lf_cnt()[li] = (uint16_t)cnt;
        f.lf_I()[li] = key;
      }
    };
    for (int v = tid; v < nrec; v += kQtThreads)
    {
      const uint8_t st = f.r_state()[v];
      const uint32_t meta = f.r_meta()[v];
      if (!(st & kFpPopped))
      {
        const uint32_t par = f.r_par()[v];
        if (v > 0 && (f.r_state()[par] & kFpPopped))
        {
          const int depth = (int)(meta >> 4);
          const int B = f.r_lo()[v], span = depth == 0 ? 125 : (depth == 1 ? 25 : 5); // (table records only)
          const uint32_t best_i = depth <= 2 ? fp_best_of_bins(f, B, B + span) : (uint32_t)f.r_best()[v];
          emit(best_i, f.r_cnt()[v], ((uint32_t)f.r_rank()[par] << 3) | ((meta >> 1) & 7u));
        }
        continue;
      }
      const uint32_t kidrec = f.r_kidrec()[v];
      const uint32_t prank = (uint32_t)f.r_rank()[v]; // 0 for the root
      const int depth = v == 0 ? -1 : (int)(meta >> 4);
      if (depth <= 2)
      {
        // children = bin ranges: strips under the root, five times finer under every table record
        const int span = depth < 0 ? kQtBinsPerStrip : (depth == 0 ? 25 : (depth == 1 ? 5 : 1));
        const int B = depth < 0 ? 0 : (int)f.r_lo()[v], nk = depth < 0 ? K : 4;
        for (int k = 0; k < nk; ++k)
        {
          const int b0 = B + k * span, tk = bin_start[b0 + span] - bin_start[b0];
          if (tk > 0 && !((kidrec >> k) & 1u)) emit(fp_best_of_bins(f, b0, b0 + span), tk, (prank << 3) | (uint32_t)k);
        }
      }
      else
      {
        const uint16_t *arr = f.arr((st & kFpKidsBuf) ? 1 : 0);
        int base = f.r_lo()[v];
        for (int k = 0; k < 4; ++k)
        {
          const int tk = f.r_t(k)[v];
          if (tk > 0 && !((kidrec >> k) & 1u))
          {
            uint32_t best = 0, best_i = 0;
            for (int pos = base; pos < base + tk; ++pos)
            {
              const uint32_t idx = arr[pos], r = resp[idx];
              if (r > best || (r == best && r > 0 && idx < best_i)) best = r, best_i = idx;
            }
            emit(best_i, tk, (prank << 3) | (uint32_t)k);
          }
          base += tk;
        }
      }
    }
  }
  fp_sync();
  const int nleaf = s_nleaf;
  if (nleaf > nc) return false; // uniform
  tick(4);
  // nodes2kpoints (:182-192): the first min(need, |M|) entries in (count desc, insertion order); drop the rest from the end
  const int surplus = nleaf - min(need, nleaf);
  for (int it = 0; it < surplus; ++it)
  {
    for (int li = tid; li < nleaf; li += kQtThreads)
      if (f.lf_cnt()[li] != 0xffffu)
        atomicMax(&s_amax, ((unsigned long long)(0xffffu - f.lf_cnt()[li]) << 32) | (unsigned long long)(f.lf_I()[li] + 1u));
    fp_sync();
    const unsigned long long top = s_amax;
    for (int li = tid; li < nleaf; li += kQtThreads)
      if (f.lf_cnt()[li] != 0xffffu && (((unsigned long long)(0xffffu - f.lf_cnt()[li]) << 32) | (unsigned long long)(f.lf_I()[li] + 1u)) == top)
        f.lf_cnt()[li] = 0xffffu;
    fp_sync();
    if (tid == 0) s_amax = 0ull;
    fp_sync();
  }
  // flags (the key array is dead by now)
  uint32_t *flag = f.keys();
  for (int i = tid; i < n; i += kQtThreads) flag[i] = 0u;
  fp_sync();
  for (int li = tid; li < nleaf; li += kQtThreads)
    if (f.lf_cnt()[li] != 0xffffu && (int)f.lf_best()[li] < n) flag[f.lf_best()[li]] = 1u;
  fp_sync();
  tick(5);
  return true;
}

__global__ void __launch_bounds__(kQtThreads, 4) quadtree_kernel(const Params p)
{
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ int s_warp[kQtThreads / 32];
  __shared__ int s_n, s_take;
  __shared__ int s_strip_cnt[32];
  __shared__ int s_bin_start[kQtMaxBinStrips * kQtBinsPerStrip + 1];

  // grid = (images, levels): CTAs are dispatched x-fastest, so every image's level 0 (the longest chain) starts first
  // and the short high levels fill the tail
  const long long t_kernel0 = clock64();
  const int level = blockIdx.y, img = blockIdx.x;
  const Level &L = p.levels[level];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int need = L.quota;
  const int ncell = L.n_level_cells;
  const int *ccnt = p.cell_cnt + (size_t)img * p.n_cells + L.cell_base;
  const Cell *cells = p.cells + L.cell_base;
  int *sel_cnt = p.sel_cnt + (size_t)img * p.n_levels + level;
  uint32_t *sel_out = p.sel + (size_t)img * p.sel_entries + L.sel_off;

  // ---- Phase A: per-cell offsets (exclusive scan of the cell counts) and the total number of corners on the level
  int *cell_off = (int *)(smem + qt_pool_bytes(p.qt_node_cap));
  const int per_c = (ncell + kQtThreads - 1) / kQtThreads;
  const int c0i = min(tid * per_c, ncell), c1i = min(c0i + per_c, ncell);
  int mysum = 0;
  for (int c = c0i; c < c1i; ++c) mysum += ccnt[c];
  int n;
  {
    int off = block_exclusive_scan<kQtThreads>(mysum, n, s_warp);
    for (int c = c0i; c < c1i; ++c)
    {
      cell_off[c] = off;
      off += ccnt[c];
    }
    if (tid == 0) cell_off[ncell] = n;
  }

  // carve shared memory
  const int node_cap = p.qt_node_cap;
  QtState q;
  uint8_t *lists, *fast_tables;
  {
    uint8_t *w = smem;
    // node bounds: global scratch behind the level's lists (only nodes below the key depth ever read or write them)
    q.np.r0 = (long long *)(p.qt_scratch + (size_t)img * p.qt_scratch_img_stride + L.scratch_off + 4 * (size_t)L.list_cap + 8);
    q.np.r1 = q.np.r0 + node_cap;
    q.np.c0 = q.np.r1 + node_cap;
    q.np.c1 = q.np.c0 + node_cap;
    q.np.rec = (uint2 *)w;
    q.np.seq = (uint32_t *)(q.np.rec + node_cap);
    q.np.next = (uint16_t *)(q.np.seq + node_cap);
    q.np.prev = q.np.next + node_cap;
    q.np.free_ids = q.np.prev + node_cap;
    q.np.state = (uint8_t *)(q.np.free_ids + node_cap);
    w = smem + qt_pool_bytes(node_cap) + qt_align16((size_t)p.qt_cell_cap * sizeof(int));
    q.bhead = (uint16_t *)w;
    q.btail = q.bhead + kQtBuckets;
    q.big = (uint16_t *)(w + qt_align16((size_t)2 * kQtBuckets * sizeof(uint16_t)));
    fast_tables = w; // the loop-free path's tables share this region with the two above
    w += qt_union_bytes(node_cap, p.qt_big_cap);
    lists = w;
    q.nbig = 0;
    q.seq_ctr = 0;
  }
  // the level's corner list always lives in the global scratch; index arrays / keys there only for dense levels
  uint32_t *kp = p.qt_scratch + (size_t)img * p.qt_scratch_img_stride + L.scratch_off;
  const bool in_smem = n <= p.qt_smem_cap;
  uint32_t *keys = in_smem ? (uint32_t *)lists : kp + L.list_cap;
  uint16_t *ia16 = (uint16_t *)(lists + (size_t)p.qt_smem_cap * sizeof(uint32_t)), *ib16 = ia16 + p.qt_smem_cap;
  uint32_t *ia32 = kp + 2 * (size_t)L.list_cap, *ib32 = ia32 + L.list_cap;
  const int K = L.n_ini;
  const bool use_keys = K <= 31;
  // the strip bounds are read several times per corner (strip search, key division): one copy in shared memory instead of
  // dependent global loads (kMaxStrips + 1 entries would be 2 KB; the key path needs at most 32 of them)
  __shared__ long long s_cols[33];
  const bool cols_in_smem = K <= 32;
  if (cols_in_smem && tid <= K) s_cols[tid] = p.strips_fx[L.strip_off + tid];
  const long long *cols = cols_in_smem ? s_cols : p.strips_fx + L.strip_off;
  const long long roi_h_fx = (long long)L.roi_h << kFixShift, roi_w_fx = (long long)L.roi_w << kFixShift;

  // ---- Phase B: gather the cell lists (cell-row-major, row-major inside a cell == the reference's detection order),
  // one thread per corner: binary search of the corner's cell in the offsets, then load + key
  __syncthreads();
  uint8_t *resp8 = lists + 8 * (size_t)p.qt_smem_cap; // FAST score by corner (loop-free path)
  auto gather = [&]() {
    const uint32_t *cl = p.cell_list + (size_t)img * p.cell_entries;
    // where cell c's list starts in the cell-list buffer, relative to its offset in the level's list: corner i of cell c is
    // cl[i + delta[c]].  Kept in the (still unused) second index array so that the corner's load does not wait for a global load
    // of the cell record first.
    int *cell_delta = (int *)ib16;
    const bool delta_ok = (size_t)ncell * sizeof(int) <= (size_t)p.qt_smem_cap * sizeof(uint16_t);
    if (delta_ok)
      for (int c = tid; c < ncell; c += kQtThreads) cell_delta[c] = cells[c].slot - cell_off[c];
    __syncthreads();
    int n_steps = 0; // binary search steps: the same for every corner
    while ((1 << n_steps) < ncell) ++n_steps;
    constexpr int G = 4; // corners per thread in flight: the searches and the loads of a batch are independent
    for (int i0 = tid; i0 < n; i0 += G * kQtThreads)
    {
      int idx[G], lo_c[G], hi_c[G];
#pragma unroll
      for (int g = 0; g < G; ++g) idx[g] = min(i0 + g * kQtThreads, n - 1), lo_c[g] = 0, hi_c[g] = ncell; // largest c with cell_off[c] <= i
      for (int st = 0; st < n_steps; ++st)
      {
#pragma unroll
        for (int g = 0; g < G; ++g)
          if (hi_c[g] - lo_c[g] > 1)
          {
            const int mid = (lo_c[g] + hi_c[g]) >> 1;
            if (cell_off[mid] <= idx[g])
              lo_c[g] = mid;
            else
              hi_c[g] = mid;
          }
      }
      uint32_t e[G];
#pragma unroll
      for (int g = 0; g < G; ++g) e[g] = delta_ok ? cl[idx[g] + cell_delta[lo_c[g]]] : cl[cells[lo_c[g]].slot + (idx[g] - cell_off[lo_c[g]])];
#pragma unroll
      for (int g = 0; g < G; ++g)
        if (i0 + g * kQtThreads < n)
        {
          const int i = idx[g];
          kp[i] = e[g];
          if (use_keys) keys[i] = qt_make_key(e[g], cols, K, L.roi_h);
          if (in_smem) resp8[i] = (uint8_t)(e[g] >> 24);
        }
    }
  };

  // ---- Phase B': root.  With need <= 1 the reference never pops the root (:151); otherwise its first pop is the root,
  // whose children are the strips: partition the corners by strip with the whole block (stable: K ordered scans).
  gather();
  const bool split_root_here = use_keys && need > 1;
  const bool presort = split_root_here && K <= kQtMaxBinStrips;
  auto root_partition = [&]() {
    if (tid < 32) s_strip_cnt[tid] = 0;
    __syncthreads();
    if (presort)
    {
      // counting sort by (strip, depth-1 digit, depth-2 digit), "on a split line" (7) last; order inside a bin is arbitrary
      // (nothing downstream depends on the order of a node's list: the best-response pick breaks ties by lowest index)
      const int nb = K * kQtBinsPerStrip;
      int *s_bin_cur = in_smem ? (int *)ib16 : (int *)ib32; // scatter cursors: the second index array is still unused here
      auto bin_of = [&](uint32_t key) -> int {
        const uint32_t sidx = key >> kKeyStripShift;
        if (sidx == kKeyNoStrip) return -1;
        uint32_t b = sidx;
#pragma unroll
        for (int j = 1; j <= kQtPresort; ++j) b = b * 5u + min((key >> (kKeyStripShift - 3 * j)) & 7u, 4u);
        return (int)b;
      };
      for (int i = tid; i <= nb; i += kQtThreads) s_bin_start[i] = 0;
      __syncthreads();
      for (int i = tid; i < n; i += kQtThreads)
      {
        const int b = bin_of(keys[i]);
        if (b >= 0) atomicAdd(&s_bin_start[b + 1], 1);
      }
      __syncthreads();
      {
        // exclusive scan over the bins: a contiguous run of bins per thread
        const int per = (nb + kQtThreads - 1) / kQtThreads;
        const int b0 = min(tid * per, nb), b1 = min(b0 + per, nb);
        int mine = 0;
        for (int b = b0; b < b1; ++b) mine += s_bin_start[b + 1];
        int total;
        int off = block_exclusive_scan<kQtThreads>(mine, total, s_warp);
        for (int b = b0; b < b1; ++b)
        {
          const int c = s_bin_start[b + 1];
          s_bin_cur[b] = off;
          off += c;
        }
        __syncthreads();
        for (int b = b0; b < b1; ++b) s_bin_start[b] = s_bin_cur[b];
        if (tid == 0) s_bin_start[nb] = total;
      }
      __syncthreads();
      for (int i = tid; i < n; i += kQtThreads)
      {
        const int b = bin_of(keys[i]);
        if (b >= 0)
        {
          const int pos = atomicAdd(&s_bin_cur[b], 1);
          if (in_smem)
            ia16[pos] = (uint16_t)i;
          else
            ia32[pos] = (uint32_t)i;
        }
      }
      if (tid < K) s_strip_cnt[tid] = s_bin_start[(tid + 1) * kQtBinsPerStrip] - s_bin_start[tid * kQtBinsPerStrip];
    }
    else if (split_root_here)
    {
      const int per = (n + kQtThreads - 1) / kQtThreads;
      const int i0 = min(tid * per, n), i1 = min(i0 + per, n);
      int base = 0;
      for (int k = 0; k < K; ++k)
      {
        int mine = 0;
        for (int i = i0; i < i1; ++i) mine += (keys[i] >> kKeyStripShift) == (uint32_t)k;
        int total;
        int off = base + block_exclusive_scan<kQtThreads>(mine, total, s_warp);
        for (int i = i0; i < i1; ++i)
          if ((keys[i] >> kKeyStripShift) == (uint32_t)k)
          {
            if (in_smem)
              ia16[off] = (uint16_t)i;
            else
              ia32[off] = (uint32_t)i;
            ++off;
          }
        if (tid == 0) s_strip_cnt[k] = total;
        base += total;
      }
    }
    else
    {
      if (in_smem)
        for (int i = tid; i < n; i += kQtThreads) ia16[i] = (uint16_t)i; // root holds every corner (:26-27)
      else
        for (int i = tid; i < n; i += kQtThreads) ia32[i] = (uint32_t)i;
    }

    __syncthreads();
  };
  root_partition();

  // ---- loop-free path (see qt_fast_path): the usual case -- the keys decide everything -- needs no sequential loop at all.
  // It works on the presorted corners (index array grouped by (strip, d1, d2, d3) bin + the bin table); if it has to give up
  // after it has started to partition nodes, the presort is simply redone for the sequential loop.
  bool done = false;
  if (tid == 0 && p.qt_stats) atomicAdd(&p.qt_stats[2 + 6], (unsigned long long)(clock64() - t_kernel0)); // phases A, B, B'
  if (p.qt_fast && presort && in_smem)
  {
    uint8_t *lf = fast_tables + 2048;
    done = qt_fast_path(smem, lists, (int *)fast_tables, lf, (uint16_t *)(lf + qt_align16((size_t)node_cap * 8)), s_bin_start, p.qt_smem_cap, node_cap, K, n, need,
                        s_warp, p.qt_stats);
    if (!done)
    { // start over for the sequential loop (the loop-free path reuses the key / index arrays)
      gather();
      root_partition();
    }
  }
  uint32_t *flag = keys; // the key array doubles as the "selected" flag array at the end
  if (tid == 0 && p.qt_stats) atomicAdd(&p.qt_stats[done ? 0 : 1], 1ull);
  const long long t_post0 = clock64();
  if (!done)
  {
  for (int i = tid; i < 2 * kQtBuckets; i += kQtThreads) q.bhead[i] = (uint16_t)kNil; // heads and tails are contiguous
  for (int i = tid; i < node_cap; i += kQtThreads) q.np.state[i] = 0;
  __syncthreads();

  // ---- Phase C: the priority loop, warp 0 only
  if (wid == 0)
  {
    int n_alloc = 0, live = 0, take = 0;
    bool root_pending;
    if (split_root_here)
    {
      // state right after the reference's first iteration: root popped, its non-empty strips inserted in order
      uint32_t base = 0;
      for (int k = 0; k < K; ++k)
      {
        const uint32_t cnt = (uint32_t)s_strip_cnt[k];
        if (cnt == 0) continue;
        const uint32_t cid = (uint32_t)n_alloc++;
        if (lane == 0)
        {
          q.np.r0[cid] = 0;
          q.np.r1[cid] = roi_h_fx;
          q.np.c0[cid] = cols[k];
          q.np.c1[cid] = cols[k + 1];
          q.np.rec[cid] = qt_rec(base, cnt, 0, 0);
        }
        qt_push(q, cid, cnt, lane);
        ++live;
        base += cnt;
      }
      root_pending = false;
    }
    else
    {
      if (lane == 0)
      {
        q.np.r0[0] = 0;
        q.np.r1[0] = roi_h_fx;
        q.np.c0[0] = 0;
        q.np.c1[0] = roi_w_fx;
        q.np.rec[0] = qt_rec(0, (uint32_t)n, 0, 0);
      }
      qt_push(q, 0, (uint32_t)n, lane);
      n_alloc = 1;
      live = 1;
      root_pending = true;
    }
    __syncwarp();
    if (in_smem)
      qt_simulate<uint16_t>(p, L, q, kp, keys, use_keys, presort ? s_bin_start : nullptr, ia16, ib16, n, need, node_cap, lane, live, n_alloc, root_pending,
                            n_alloc, take);
    else
      qt_simulate<uint32_t>(p, L, q, kp, keys, use_keys, presort ? s_bin_start : nullptr, ia32, ib32, n, need, node_cap, lane, live, n_alloc, root_pending,
                            n_alloc, take);
    if (lane == 0)
    {
      s_n = n_alloc; // node slots ever used
      s_take = take;
    }
  }
  // the key array doubles as the "selected" flag array from here on
  __syncthreads();
  for (int i = tid; i < n; i += kQtThreads) flag[i] = 0u;
  __syncthreads();

  // ---- Phase D
  if (s_take > 0)
  {
    if (in_smem)
      qt_select<uint16_t>(q.np, kp, ia16, ib16, flag, n, s_n, tid);
    else
      qt_select<uint32_t>(q.np, kp, ia32, ib32, flag, n, s_n, tid);
  }
  __syncthreads();
  } // !done
  {
    const int per = (n + kQtThreads - 1) / kQtThreads;
    const int i0 = min(tid * per, n), i1 = min(i0 + per, n);
    int mine = 0;
    for (int i = i0; i < i1; ++i) mine += (int)flag[i];
    int total;
    int off = block_exclusive_scan<kQtThreads>(mine, total, s_warp);
    for (int i = i0; i < i1; ++i)
      if (flag[i])
      {
        const uint32_t e = kp[i];
        // back to level coordinates (:382-383)
        if (off < need) sel_out[off] = ((e & 0xfffu) + kEdge) | ((((e >> 12) & 0xfffu) + kEdge) << 12) | (e & 0xff000000u);
        ++off;
      }
    if (tid == 0) *sel_cnt = min(total, need);
  }
  if (tid == 0 && p.qt_stats && done) atomicAdd(&p.qt_stats[2 + 7], (unsigned long long)(clock64() - t_post0)); // ordered emit
}

int quadtree_configure(size_t smem_bytes)
{
  static SmemOptIn state;
  return raise_dynamic_smem(quadtree_kernel, state, smem_bytes);
}

void launch_quadtree(const Params &p, int n_images, size_t smem_bytes, cudaStream_t s)
{
  dim3 grid(n_images, p.n_levels);
  quadtree_kernel<<<grid, kQtThreads, smem_bytes, s>>>(p);
}

// ------------------------------------------------------------------------------------------------------------------
// K4: intensity-centroid orientation + rotated BRIEF.  One warp per keypoint.
// ------------------------------------------------------------------------------------------------------------------
__constant__ int c_umax[16] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3}; // initMaxU (:217-236), radius 15

constexpr int kBriefWarps = 8;
constexpr int kBriefReach = 18;                          // cvRound of the largest rotated pattern radius, |(13, 13)| = 18.38
constexpr int kBriefPatchRows = 2 * kBriefReach + 1;     // 37
constexpr uint32_t kBriefPatchPitch = 64;                // bytes = width of the TMA box: up to 15 bytes of alignment shift + 37
constexpr int kBriefPatchBytes = 2432;                   // 37 rows x 64 bytes, rounded up to the 128-byte alignment of a TMA destination

__device__ __forceinline__ void undistort_point(const Params &p, float u, float v, float &uo, float &vo)
{
  // cv::undistortPoints(pts, pts, K, D, noArray(), K) (src/Camera.cc:36): 5 fixed-point iterations in double
  const double fx = p.fx, fy = p.fy, cx = p.cx, cy = p.cy;
  const double k1 = p.dist[0], k2 = p.dist[1], p1 = p.dist[2], p2 = p.dist[3], k3 = p.dist[4];
  const double ifx = __ddiv_rn(1.0, fx), ify = __ddiv_rn(1.0, fy);
  double x = __dmul_rn(__dsub_rn((double)u, cx), ifx), y = __dmul_rn(__dsub_rn((double)v, cy), ify);
  const double x0 = x, y0 = y;
#pragma unroll 1
  for (int it = 0; it < 5; ++it)
  {
    const double xx = __dmul_rn(x, x), yy = __dmul_rn(y, y);
    const double r2 = __dadd_rn(xx, yy);
    double poly = __dadd_rn(__dmul_rn(k3, r2), k2);
    poly = __dadd_rn(__dmul_rn(poly, r2), k1);
    poly = __dadd_rn(1.0, __dmul_rn(poly, r2));
    const double icdist = __ddiv_rn(1.0, poly);
    const double dx = __dadd_rn(__dmul_rn(__dmul_rn(__dmul_rn(2.0, p1), x), y), __dmul_rn(p2, __dadd_rn(r2, __dmul_rn(2.0, xx))));
    const double dy = __dadd_rn(__dmul_rn(p1, __dadd_rn(r2, __dmul_rn(2.0, yy))), __dmul_rn(__dmul_rn(__dmul_rn(2.0, p2), x), y));
    x = __dmul_rn(__dsub_rn(x0, dx), icdist);
    y = __dmul_rn(__dsub_rn(y0, dy), icdist);
  }
  uo = __double2float_rn(__dadd_rn(__dmul_rn(x, fx), cx));
  vo = __double2float_rn(__dadd_rn(__dmul_rn(y, fy), cy));
}

__device__ __forceinline__ int dp4a_u8_s8(uint32_t a_u8x4, uint32_t b_s8x4, int c)
{
  int d;
  asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a_u8x4), "r"(b_s8x4), "r"(c));
  return d;
}

// kBriefGroup keypoints per warp: lane j < kBriefGroup evaluates atan2 / sincos of keypoint j (once, not 32 times).  Large
// batches use 8 (throughput), a handful of images 2 (shorter warps: single-frame latency).
template <int kBriefGroup> __global__ void __launch_bounds__(kBriefWarps * 32, 5) orient_brief_kernel(const Params p, const __grid_constant__ LevelMaps blur_maps)
{
  // Per-lane DP4A weights of the radius-15 disc for the moment pass below (lane <-> word wk of row 3 i + rg, see there):
  // byte b of s_wx[i][lane] = dx of that byte if it lies inside the disc (|dx| <= umax[|dy|]), else 0; s_wy: dy likewise.
  __shared__ uint32_t s_wx[11][32], s_wy[11][32];
  for (int t = threadIdx.x; t < 11 * 32; t += kBriefWarps * 32)
  {
    const int i = t >> 5, ln = t & 31, g = ln / 9, k = ln - 9 * g, r = 3 * i + g, dy = r - 15;
    uint32_t wx = 0, wy = 0;
    if (g < 3 && k < 8 && r < 31)
    {
#pragma unroll
      for (int b = 0; b < 4; ++b)
      {
        const int dx = 4 * k + b - 15; // byte 31 of the 32-byte row (dx = 16) is never part of the disc
        if (dx <= 15 && abs(dx) <= c_umax[abs(dy)]) wx |= (uint32_t)(dx & 0xff) << (8 * b), wy |= (uint32_t)(dy & 0xff) << (8 * b);
      }
    }
    s_wx[i][ln] = wx;
    s_wy[i][ln] = wy;
  }
  // BRIEF pattern, one word (x1, y1, x2, y2 as signed bytes) per pair: bit b = lane * 8 + k at [k][lane]
  __shared__ uint32_t s_pat8[8][32];
  {
    const int b = threadIdx.x;
    static_assert(kBriefWarps * 32 == 256, "one thread per pattern pair");
    const char4 q = p.pattern[b];
    s_pat8[b & 7][b >> 3] = ((uint32_t)(uint8_t)q.x | ((uint32_t)(uint8_t)q.y << 8) | ((uint32_t)(uint8_t)q.z << 16) | ((uint32_t)(uint8_t)q.w << 24));
  }
  __syncthreads();

  const int img = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int slot0 = (blockIdx.x * kBriefWarps + (threadIdx.x >> 5)) * kBriefGroup;

  // which level does an output slot belong to? (level-major concatenation, src/ORBExtractor.cc:501-506)
  const int *sel_cnt = p.sel_cnt + (size_t)img * p.n_levels;
  const int my = lane < p.n_levels ? sel_cnt[lane] : 0;
  const int inc = warp_inclusive_scan(my, lane);
  const int total = __shfl_sync(kFullMask, inc, 31);
  if (slot0 == 0 && lane == 0) p.n_kps[img] = total;
  if (slot0 >= total) return;
  const int n_here = min(kBriefGroup, total - slot0);
  const uint8_t *__restrict__ pyr_img = p.pyr + (size_t)img * p.pyr_img_stride;

  // Pass 1, keypoint by keypoint: getGrayCentroid (:465-487), moments over the radius-15 disc of the un-blurred level.
  // The disc's 31 rows are fetched as aligned words, 3 rows x 9 words per warp request (3 cache lines); a lane takes its
  // word and the next one (from the neighbour lane), shifts them to the row start and takes both moments with DP4A against
  // the lane's signed weights (dx resp. dy inside the disc, 0 outside; tables above).  Every level pitch is a multiple of
  // 4, so the shift is the same for all rows.  Lane j keeps keypoint j's entry and moments.
  uint32_t my_e = 0;
  int my_level = 0, my_m10 = 0, my_m01 = 0;
  const int rg = lane / 9, wk = lane - 9 * rg; // lanes 27..31: rg == 3, idle (zero weights)
#pragma unroll 1
  for (int j = 0; j < n_here; ++j)
  {
    const int slot = slot0 + j;
    const unsigned above = __ballot_sync(kFullMask, inc > slot); // first lane whose inclusive sum exceeds the slot
    const int level = __ffs(above) - 1;
    const int level_start = __shfl_sync(kFullMask, inc - my, level);
    const Level &L = p.levels[level];
    const uint32_t e = p.sel[(size_t)img * p.sel_entries + L.sel_off + (slot - level_start)];
    const int x = (int)(e & 0xfffu), y = (int)((e >> 12) & 0xfffu);
    const int pitch = L.pitch;
    const uint8_t *row0 = pyr_img + L.pyr_off + (size_t)(y - 15) * pitch + (x - 15);
    const uint32_t mis = (uint32_t)(size_t)row0 & 3u, sh = mis * 8u;
    // idle lanes re-read rows 0..2
    const uint8_t *wp = row0 - mis + 4 * wk + (size_t)min(rg, 2) * pitch;
    const uint32_t pitch3 = 3u * (uint32_t)pitch;
    uint32_t a[11];
#pragma unroll
    for (int i = 0; i < 10; ++i) a[i] = __ldg(reinterpret_cast<const uint32_t *>(wp + (uint64_t)pitch3 * (uint32_t)i)); // one IMAD.WIDE per address
    a[10] = __ldg(reinterpret_cast<const uint32_t *>(row0 - mis + 4 * wk + 30 * (size_t)pitch)); // row 30: only the rg == 0 lanes carry weights
    int m10 = 0, m01 = 0;
#pragma unroll
    for (int i = 0; i < 11; ++i)
    {
      const uint32_t nxt = __shfl_down_sync(kFullMask, a[i], 1);
      const uint32_t v = __funnelshift_r(a[i], nxt, sh);
      m10 = dp4a_u8_s8(v, s_wx[i][lane], m10);
      m01 = dp4a_u8_s8(v, s_wy[i][lane], m01);
    }
    m10 = __reduce_add_sync(kFullMask, m10);
    m01 = __reduce_add_sync(kFullMask, m01);
    if (lane == j) my_e = e, my_level = level, my_m10 = m10, my_m01 = m01;
  }

  // Pass 2, keypoint by keypoint: computeBRIEF (:427-456) with rotateTemplate (:534-540): double products, float result,
  // float add, round-half-even; lane <-> descriptor byte.
  // The rotated pattern stays within 18 px of the keypoint (|(13, 13)| = 18.4): the 37 x 37 blurred patch around it arrives in
  // shared memory through ONE TMA box load (cp.async.bulk.tensor.3d from the level's {pitch, rows, images} byte tensor over
  // `blur`; box = 64 bytes x 37 rows, its first column aligned down to 16 bytes as TMA requires), so that the 512 scattered
  // byte gathers of the descriptor hit shared-memory banks instead of 512 different L1 sectors.  Two buffers per warp: the
  // patch of keypoint j + 1 is in flight while keypoint j is evaluated; the first one is requested before atan2 / sincos.
  // Keypoints keep 19 px from the border (mnBorderSize), so rows y - 18 .. y + 18 exist; whatever the box covers beyond the
  // level's pitch is zero-filled and never read.
  __shared__ __align__(128) uint8_t s_patch[kBriefWarps][2][kBriefPatchBytes];
  __shared__ __align__(8) uint64_t s_bar[kBriefWarps][2];
  const int wid = threadIdx.x >> 5;
  if (lane == 0)
  {
    mbar_init(&s_bar[wid][0], 1);
    mbar_init(&s_bar[wid][1], 1);
  }
  __syncwarp();
  auto request_patch = [&](int j) { // all lanes call; lane 0 issues the load of keypoint j's patch into buffer j & 1
    const uint32_t e = __shfl_sync(kFullMask, my_e, j);
    const int level = __shfl_sync(kFullMask, my_level, j);
    if (lane == 0)
    {
      const int kx_i = (int)(e & 0xfffu), ky_i = (int)((e >> 12) & 0xfffu);
      mbar_expect_tx(&s_bar[wid][j & 1], kBriefPatchRows * kBriefPatchPitch);
      tma_load_3d(s_patch[wid][j & 1], &blur_maps.m[level], (kx_i - kBriefReach) & ~15, ky_i - kBriefReach, p.img0 + img, &s_bar[wid][j & 1]);
    }
  };
  request_patch(0);

  // orientation of keypoint `lane` (lanes >= n_here compute on zeros and are ignored)
  const double theta = atan2((double)my_m01, (double)my_m10);
  double sn, cs;
  sincos(theta, &sn, &cs);

#pragma unroll 1
  for (int j = 0; j < n_here; ++j)
  {
    const uint32_t e = __shfl_sync(kFullMask, my_e, j);
    const double sj = __shfl_sync(kFullMask, sn, j), cj = __shfl_sync(kFullMask, cs, j);
    const float fx = (float)(e & 0xfffu), fy = (float)((e >> 12) & 0xfffu);
    const int kx_i = (int)(e & 0xfffu), ky_i = (int)((e >> 12) & 0xfffu);
    __syncwarp(); // keypoint j - 1's gathers from the other buffer are done
    if (j + 1 < n_here) request_patch(j + 1);
    mbar_wait(&s_bar[wid][j & 1], (uint32_t)((j >> 1) & 1));
    const uint32_t mis = (uint32_t)(kx_i - kBriefReach) & 15u; // column of the patch origin inside the box
    const uint32_t *my_patch = reinterpret_cast<const uint32_t *>(s_patch[wid][j & 1]);
    // cvRound without the conversion unit (below) leaves 0x4B400000 in both coordinates; that, the patch origin and the
    // alignment shift fold into one constant (modulo 2^32), so one 32-bit multiply-add gives the byte index into the patch
    uint32_t kofs = mis - 0x4B400000u * (kBriefPatchPitch + 1u) - (uint32_t)(ky_i - kBriefReach) * kBriefPatchPitch - (uint32_t)(kx_i - kBriefReach);
    asm volatile("" : "+r"(kofs)); // opaque: stays one register instead of being re-materialised per access
    const uint8_t *patch_b = reinterpret_cast<const uint8_t *>(my_patch);
    uint32_t byte = 0;
#pragma unroll 4
    for (int k = 0; k < 8; ++k)
    {
      // bit b = lane * 8 + k lands in byte b >> 3 == lane, position b & 7 == k.  The pair's four integer coordinates come as
      // one packed word; int8 -> double is one conversion each (I2F.F64.S8 with a byte selector), exact
      const uint32_t w = s_pat8[k][lane];
      const double x1 = (double)(signed char)(w & 0xffu), y1 = (double)(signed char)((w >> 8) & 0xffu);
      const double x2 = (double)(signed char)((w >> 16) & 0xffu), y2 = (double)(signed char)(w >> 24);
      const float p1x = __double2float_rn(__dsub_rn(__dmul_rn(x1, cj), __dmul_rn(y1, sj)));
      const float p1y = __double2float_rn(__dadd_rn(__dmul_rn(x1, sj), __dmul_rn(y1, cj)));
      const float p2x = __double2float_rn(__dsub_rn(__dmul_rn(x2, cj), __dmul_rn(y2, sj)));
      const float p2y = __double2float_rn(__dadd_rn(__dmul_rn(x2, sj), __dmul_rn(y2, cj)));
      // cvRound without the conversion unit: float_as_uint(v + 1.5 * 2^23) == 0x4B400000 + round_half_even(v) for 0 <= v < 2^22
      const uint32_t r1y = __float_as_uint(__fadd_rn(__fadd_rn(fy, p1y), 12582912.f)), r1x = __float_as_uint(__fadd_rn(__fadd_rn(fx, p1x), 12582912.f));
      const uint32_t r2y = __float_as_uint(__fadd_rn(__fadd_rn(fy, p2y), 12582912.f)), r2x = __float_as_uint(__fadd_rn(__fadd_rn(fx, p2x), 12582912.f));
      const int v1 = patch_b[r1y * kBriefPatchPitch + kofs + r1x];
      const int v2 = patch_b[r2y * kBriefPatchPitch + kofs + r2x];
      byte = __funnelshift_l((uint32_t)(v1 - v2), byte, 1); // shifts in the sign: 1 iff v1 < v2; bit k ends at position 7 - k
    }
    p.desc[((size_t)img * p.n_features + slot0 + j) * 32 + lane] = (uint8_t)(__brev(byte) >> 24);
  }

  // keypoint record (:407-409) + the row band used by the stereo search (createRowIndexDB, src/ORBMatcher.cc:915-932):
  // lane j writes keypoint j
  if (lane < n_here)
  {
    const size_t o = (size_t)img * p.n_features + slot0 + lane;
    const float sf = p.levels[my_level].sf;
    const float kx = __fmul_rn((float)(my_e & 0xfffu), sf), ky = __fmul_rn((float)((my_e >> 12) & 0xfffu), sf);
    orbx_keypoint kpt;
    kpt.x = kx;
    kpt.y = ky;
    kpt.size = 7.f;
    kpt.angle = __double2float_rn(__dmul_rn(__ddiv_rn(theta, 3.14159265358979323846), 180.0));
    kpt.response = (float)(my_e >> 24);
    kpt.octave = my_level;
    kpt.class_id = -1;
    p.kps[o] = kpt;
    if (p.undistort) undistort_point(p, kx, ky, kpt.x, kpt.y); // Camera::undistortPoints (src/Camera.cc:29-39)
    p.kps_und[o] = kpt;
    const float r = __double2float_rn(__dmul_rn(2.0, (double)sf));
    const unsigned row = (unsigned)__float2int_rn(ky);
    RTab rt;
    rt.x = kx;
    rt.max_row = (short)min(p.height, __float2int_rn(__fadd_rn(__fadd_rn((float)row, r), 1.0f)));
    rt.min_row = (short)max(0, __float2int_rn(__fsub_rn((float)row, r)));
    p.rtab[o] = rt;
  }
}

void launch_orient_brief(const Params &p, const LevelMaps &blur_maps, int n_images, cudaStream_t s)
{
  if (n_images > 4)
  {
    dim3 grid((p.n_features + kBriefWarps * 8 - 1) / (kBriefWarps * 8), n_images);
    orient_brief_kernel<8><<<grid, kBriefWarps * 32, 0, s>>>(p, blur_maps);
  }
  else
  {
    dim3 grid((p.n_features + kBriefWarps * 2 - 1) / (kBriefWarps * 2), n_images);
    orient_brief_kernel<2><<<grid, kBriefWarps * 32, 0, s>>>(p, blur_maps);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// K5a: createRowIndexDB (src/ORBMatcher.cc:915-932) as a CSR: for every image row the right keypoints whose band
// [minRow, maxRow) covers it.  One CTA per frame: shared-memory histogram, block scan, fill.  (Order inside a row does not
// matter: the search takes the lexicographic minimum of (distance, index), which equals the reference's first minimum
// over ascending indices.)
// ------------------------------------------------------------------------------------------------------------------
constexpr int kRowThreads = 1024;

__device__ __forceinline__ void rowindex_body(const Params &p, int frame, int *s_cnt /* [height + 1] */, int *s_warp)
{
  const int tid = threadIdx.x;
  const int H = p.height;
  const int imgR = 2 * frame + 1;
  const int nR = p.n_kps[imgR];
  const RTab *rt = p.rtab + (size_t)imgR * p.n_features;
  int *row_start = p.row_start + (size_t)frame * (H + 1);
  uint16_t *entries = p.row_entries + (size_t)frame * p.row_cap;
  for (int i = tid; i <= H; i += kRowThreads) s_cnt[i] = 0;
  __syncthreads();
  // four band records per thread are in flight before the first one is used (the loop is latency-bound: one CTA per frame)
  constexpr int U = 4;
  for (int j0 = tid; j0 < nR; j0 += U * kRowThreads)
  {
    RTab t[U];
#pragma unroll
    for (int u = 0; u < U; ++u) t[u] = rt[min(j0 + u * kRowThreads, nR - 1)];
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (j0 + u * kRowThreads < nR)
        for (int r = t[u].min_row; r < t[u].max_row; ++r) atomicAdd(&s_cnt[r], 1);
  }
  __syncthreads();
  const int per = (H + kRowThreads - 1) / kRowThreads;
  const int r0 = min(tid * per, H), r1 = min(r0 + per, H);
  int mine = 0;
  for (int r = r0; r < r1; ++r) mine += s_cnt[r];
  int total;
  int off = block_exclusive_scan<kRowThreads>(mine, total, s_warp);
  for (int r = r0; r < r1; ++r)
  {
    const int c = s_cnt[r];
    s_cnt[r] = off;
    row_start[r] = off;
    off += c;
  }
  if (tid == 0) row_start[H] = total;
  __syncthreads();
  for (int j0 = tid; j0 < nR; j0 += U * kRowThreads)
  {
    RTab t[U];
#pragma unroll
    for (int u = 0; u < U; ++u) t[u] = rt[min(j0 + u * kRowThreads, nR - 1)];
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (j0 + u * kRowThreads < nR)
        for (int r = t[u].min_row; r < t[u].max_row; ++r)
        {
          const int pos = atomicAdd(&s_cnt[r], 1);
          if (pos < p.row_cap) entries[pos] = (uint16_t)(j0 + u * kRowThreads);
        }
  }
}

// (launched together with the grid of the left keypoints: frame_index_kernel below)

// ------------------------------------------------------------------------------------------------------------------
// K5: stereo association.  One warp per left keypoint: row-band + x-range scan over the right keypoints, Hamming argmin
// (first minimum == lexicographic min of (distance, index)), 11 SADs over an 11x11 window, parabola refinement.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kStereoWarps = 8;

constexpr int kWinPitch = 24;

__global__ void __launch_bounds__(kStereoWarps * 32, 8) stereo_kernel(const Params p)
{
  __shared__ uint8_t s_win[kStereoWarps][11 * kWinPitch];
  const int frame = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int li = blockIdx.x * kStereoWarps + (threadIdx.x >> 5);
  const int imgL = 2 * frame, imgR = 2 * frame + 1;
  const int nL = p.n_kps[imgL];
  if (li >= p.n_features) return;
  const size_t oL = (size_t)imgL * p.n_features, oR = (size_t)imgR * p.n_features;
  double *ur_out = p.u_right + (size_t)frame * p.n_features + li;
  double *dp_out = p.depth + (size_t)frame * p.n_features + li;
  if (lane == 0)
  {
    *ur_out = -1.0; // :22-25
    *dp_out = -1.0;
  }
  if (li >= nL) return;

  const orbx_keypoint lk = p.kps_und[oL + li]; // the left keypoints are undistorted before matching (src/Frame.cc:106)
  const float maxU = lk.x;
  const float minU = fmaxf(0.f, __fsub_rn(lk.x, p.fx));
  const int row = __float2int_rn(lk.y);
  const uint4 *dl4 = reinterpret_cast<const uint4 *>(p.desc + (oL + li) * 32);
  const uint4 a0 = dl4[0], a1 = dl4[1];

  // getBestMatch over rowIdxDB[row] filtered by minU < x < maxU (:38-52, :967-990)
  unsigned best = 0xffffffffu;
  const RTab *rt = p.rtab + oR;
  if (row >= 0 && row < p.height) // rows outside the image index the reference's rowIdxDB out of range
  {
    const int *rs = p.row_start + (size_t)frame * (p.height + 1) + row;
    const int e0 = rs[0], e1 = min(rs[1], p.row_cap);
    const uint16_t *entries = p.row_entries + (size_t)frame * p.row_cap;
    for (int e = e0 + lane; e < e1; e += 32)
    {
      const int j = entries[e];
      const float xr = rt[j].x;
      if (xr < maxU && xr > minU)
      {
        const uint4 *dr4 = reinterpret_cast<const uint4 *>(p.desc + (oR + j) * 32);
        const uint4 b0 = dr4[0], b1 = dr4[1];
        const int d = hamming256(a0, a1, b0, b1);
        best = min(best, ((unsigned)d << 20) | (unsigned)j);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(kFullMask, best, o));
  if (best == 0xffffffffu) return;          // no candidates (:49-50)
  if ((int)(best >> 20) > 75) return;       // mnMeanThreshold (:53)
  const int rj = (int)(best & 0xfffffu);
  const orbx_keypoint rk = p.kps[oR + rj];
  if (lk.octave > rk.octave + 1 || lk.octave < rk.octave - 1) return; // :57

  // pixelSADMatch (:841-881) on the un-blurred pyramid levels of each keypoint's own octave
  const Level &LL = p.levels[lk.octave];
  const Level &LR = p.levels[rk.octave];
  const uint8_t *il = p.pyr + (size_t)imgL * p.pyr_img_stride + LL.pyr_off;
  const uint8_t *ir = p.pyr + (size_t)imgR * p.pyr_img_stride + LR.pyr_off;
  const int lx = __float2int_rd(__fdiv_rn(lk.x, LL.sf)), ly = __float2int_rd(__fdiv_rn(lk.y, LL.sf)); // getPitch (:1002-1011)
  const int rx = __float2int_rd(__fdiv_rn(rk.x, LR.sf)), ry = __float2int_rd(__fdiv_rn(rk.y, LR.sf));
  // Out-of-image windows can only arise with undistorted left coordinates; the reference would throw cv::Exception there.
  if (lx - 5 < 0 || ly - 5 < 0 || lx + 5 >= LL.w || ly + 5 >= LL.h || rx - 10 < 0 || ry - 5 < 0 || rx + 10 >= LR.w || ry + 5 >= LR.h) return;

  // 11 SADs of 11x11 centre-subtracted patches (:841-881).  The right window (11 rows x 21 columns) is staged in shared
  // memory; lane i handles the left-patch positions i, i + 32, i + 64, i + 96 (< 121) for all 11 shifts:
  // |(L - lc) - (R - rc_s)| = |(L - lc + rc_s) - R| is one add and one sad per term, and the 11 sums leave through REDUX.
  uint8_t *win = s_win[threadIdx.x >> 5];
  {
    uint8_t tmp[8];
#pragma unroll
    for (int k = 0; k < 8; ++k)
    {
      const int i = min(lane + 32 * k, 230), r = i / 21, c = i - 21 * r;
      tmp[k] = ir[(size_t)(ry - 5 + r) * LR.pitch + rx - 10 + c];
    }
#pragma unroll
    for (int k = 0; k < 8; ++k)
    {
      const int i = lane + 32 * k, r = i / 21, c = i - 21 * r;
      if (i < 231) win[r * kWinPitch + c] = tmp[k];
    }
  }
  const int lc = il[(size_t)ly * LL.pitch + lx];
  int lv[4];
#pragma unroll
  for (int k = 0; k < 4; ++k)
  {
    const int i = min(lane + 32 * k, 120), r = i / 11, c = i - 11 * r;
    lv[k] = (int)il[(size_t)(ly - 5 + r) * LL.pitch + lx - 5 + c] - lc;
  }
  __syncwarp();
  int rc[11], acc[11];
#pragma unroll
  for (int s = 0; s < 11; ++s)
  {
    rc[s] = win[5 * kWinPitch + 5 + s];
    acc[s] = 0;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k)
  {
    const int i = lane + 32 * k, r = min(i, 120) / 11, c = min(i, 120) - 11 * r;
    if (i < 121)
    {
      const uint8_t *w = win + r * kWinPitch + c;
#pragma unroll
      for (int s = 0; s < 11; ++s) acc[s] = __sad(lv[k] + rc[s], (int)w[s], acc[s]);
    }
  }
  int sad[11];
#pragma unroll
  for (int s = 0; s < 11; ++s) sad[s] = __reduce_add_sync(kFullMask, acc[s]);
  if (lane != 0) return;
  int bi = 0;
#pragma unroll
  for (int s = 1; s < 11; ++s)
    if (sad[s] < sad[bi]) bi = s; // first minimum (:862-866)
  float delta = 0.f;
  if (bi > 0 && bi < 10)
  {
    float s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
    for (int s = 1; s < 10; ++s)
      if (s == bi)
      {
        s1 = (float)sad[s - 1];
        s2 = (float)sad[s];
        s3 = (float)sad[s + 1];
      }
    const float num = __fsub_rn(s1, s3);
    const float den = __fsub_rn(__fadd_rn(s1, s3), __fmul_rn(2.f, s2));
    delta = __double2float_rn(__ddiv_rn(__dmul_rn(0.5, (double)num), (double)den));
    if (delta < 1.f && delta > -1.f)
      delta = __fmul_rn(delta, LR.sf);
    else
      delta = 0.f;
  }
  float uR = __fadd_rn(rk.x, delta);
  uR = fmaxf(0.f, uR);
  uR = fminf(uR, __fsub_rn((float)p.width, 1.f));
  float disp = __fsub_rn(lk.x, uR);
  if (disp <= 0.f)
  {
    uR = rk.x;
    disp = __fsub_rn(lk.x, uR);
    if (disp <= 0.f) return;
  }
  *ur_out = (double)uR;
  *dp_out = (double)__fdiv_rn(p.bf, __fsub_rn(lk.x, uR));
  atomicAdd(p.n_matches + frame, 1);
}

void launch_stereo(const Params &p, int n_frames, cudaStream_t s)
{
  dim3 grid((p.n_features + kStereoWarps - 1) / kStereoWarps, n_frames);
  stereo_kernel<<<grid, kStereoWarps * 32, 0, s>>>(p);
}

// ------------------------------------------------------------------------------------------------------------------
// K6: RGB-D depth association (src/Frame.cc:125-159): d = depth(int(y), int(x)) on the RAW keypoint, uRight from the
// undistorted x.  The whole-image convertTo / divide of the reference is folded into the per-keypoint gather.
// ------------------------------------------------------------------------------------------------------------------
__global__ void rgbd_kernel(const Params p)
{
  const int frame = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n_features) return;
  const size_t o = (size_t)frame * p.n_features + i;
  double ur = -1.0, dp = -1.0;
  if (i < p.n_kps[frame])
  {
    const orbx_keypoint k = p.kps[o];
    const int yy = (int)k.y, xx = (int)k.x; // Mat::at<float>(float, float): truncation
    const uint8_t *base = (const uint8_t *)p.depth_img + (size_t)frame * p.depth_frame_stride + (size_t)yy * p.depth_stride;
    const float raw = p.depth_type == ORBX_DEPTH_F32 ? ((const float *)base)[xx] : (float)((const uint16_t *)base)[xx];
    const float d = __fmul_rn(raw, p.depth_scale_inv);
    if (d > 0.f)
    {
      dp = (double)d;
      ur = (double)__fsub_rn(p.kps_und[o].x, __fdiv_rn(p.bf, d));
      atomicAdd(p.n_matches + frame, 1);
    }
  }
  p.u_right[o] = ur;
  p.depth[o] = dp;
}

void launch_rgbd(const Params &p, int n_frames, cudaStream_t s)
{
  dim3 grid((p.n_features + 127) / 128, n_frames);
  rgbd_kernel<<<grid, 128, 0, s>>>(p);
}

// ------------------------------------------------------------------------------------------------------------------
// K7: VirtualFrame::initGrid (src/Frame.cc:53-69): bucket the frame's (undistorted) left keypoints into 64x48-px cells,
// rowIdx = cvFloor(pt.y / 48), colIdx = cvFloor(pt.x / 64) in float; a cell lists its keypoints in ascending index order
// (the reference push_backs them in keypoint order).  One CTA per frame: histogram, scan, fill, per-cell sort.
// ------------------------------------------------------------------------------------------------------------------
constexpr int kGridThreads = 1024;

__device__ __forceinline__ void grid_body(const Params &p, int frame, int image_stride, int *s_cell /* [n_cells + 1] */, uint16_t *s_ent /* [n_features] */,
                                          int *s_warp)
{
  const int tid = threadIdx.x;
  const int img = frame * image_stride;
  const int nc = p.grid_rows * p.grid_cols;
  const int n = p.n_kps[img];
  const orbx_keypoint *kps = p.kps_und + (size_t)img * p.n_features;
  int *start = p.grid_start + (size_t)frame * (nc + 1);
  uint16_t *entries = p.grid_entries + (size_t)frame * p.n_features;
  auto cell_of = [&](int i) -> int {
    const int r = __float2int_rd(__fdiv_rn(kps[i].y, 48.f)), c = __float2int_rd(__fdiv_rn(kps[i].x, 64.f));
    return (r >= 0 && r < p.grid_rows && c >= 0 && c < p.grid_cols) ? r * p.grid_cols + c : -1; // outside: UB in the reference
  };
  for (int i = tid; i <= nc; i += kGridThreads) s_cell[i] = 0;
  __syncthreads();
  constexpr int U = 4; // keypoints per thread in flight (their coordinates come from global memory in every pass)
  for (int i0 = tid; i0 < n; i0 += U * kGridThreads)
  {
    int c[U];
#pragma unroll
    for (int u = 0; u < U; ++u) c[u] = cell_of(min(i0 + u * kGridThreads, n - 1));
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (i0 + u * kGridThreads < n && c[u] >= 0) atomicAdd(&s_cell[c[u]], 1);
  }
  __syncthreads();
  const int per = (nc + kGridThreads - 1) / kGridThreads;
  const int c0 = min(tid * per, nc), c1 = min(c0 + per, nc);
  int mine = 0;
  for (int c = c0; c < c1; ++c) mine += s_cell[c];
  int total;
  int off = block_exclusive_scan<kGridThreads>(mine, total, s_warp);
  for (int c = c0; c < c1; ++c)
  {
    const int k = s_cell[c];
    s_cell[c] = off;
    start[c] = off;
    off += k;
  }
  if (tid == 0) start[nc] = total;
  __syncthreads();
  for (int i0 = tid; i0 < n; i0 += U * kGridThreads)
  {
    int c[U];
#pragma unroll
    for (int u = 0; u < U; ++u) c[u] = cell_of(min(i0 + u * kGridThreads, n - 1));
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (i0 + u * kGridThreads < n && c[u] >= 0) s_ent[atomicAdd(&s_cell[c[u]], 1)] = (uint16_t)(i0 + u * kGridThreads);
  }
  __syncthreads();
  // ascending index order inside every cell (the reference's push_back order), by rank: keypoint i goes to the cell's start +
  // the number of cell members with a smaller index.  One thread per keypoint scans its cell (a few dozen entries, independent
  // shared-memory reads) instead of one thread per cell running a dependent insertion sort; the ranks are distinct, so the
  // entries go straight to global memory.  After the scatter s_cell[c] is the END of cell c, i.e. the start of cell c + 1.
  for (int i0 = tid; i0 < n; i0 += U * kGridThreads)
  {
    int c[U];
#pragma unroll
    for (int u = 0; u < U; ++u) c[u] = cell_of(min(i0 + u * kGridThreads, n - 1));
#pragma unroll
    for (int u = 0; u < U; ++u)
    {
      const int i = i0 + u * kGridThreads;
      if (i >= n || c[u] < 0) continue;
      const int b = c[u] == 0 ? 0 : s_cell[c[u] - 1], e = s_cell[c[u]];
      int rank = 0;
      for (int j = b; j < e; ++j) rank += (int)(s_ent[j] < (uint16_t)i);
      entries[b + rank] = (uint16_t)i;
    }
  }
}

// K5a + K7 in ONE launch: blocks [0, n_frames) build the row index of the right keypoints (stereo frames only), the next n_frames
// blocks the 64x48-px grid of the left keypoints.  Both are one-CTA-per-frame jobs; side by side they cost the longer of the two.
static_assert(kRowThreads == kGridThreads, "frame_index_kernel");
__global__ void __launch_bounds__(kGridThreads) frame_index_kernel(const Params p, int n_frames, int image_stride, int with_rowindex)
{
  extern __shared__ __align__(16) int s_dyn[];
  __shared__ int s_warp[kGridThreads / 32];
  const int b = blockIdx.x;
  if (with_rowindex && b < n_frames)
    rowindex_body(p, b, s_dyn, s_warp);
  else
  {
    const int frame = with_rowindex ? b - n_frames : b;
    const int nc = p.grid_rows * p.grid_cols;
    grid_body(p, frame, image_stride, s_dyn, reinterpret_cast<uint16_t *>(s_dyn + nc + 1), s_warp);
  }
}

static size_t frame_index_smem(const Params &p)
{
  const size_t row = (size_t)(p.height + 1) * sizeof(int);
  const size_t grid = (size_t)(p.grid_rows * p.grid_cols + 1) * sizeof(int) + (size_t)p.n_features * sizeof(uint16_t);
  return row > grid ? row : grid;
}

int frame_index_configure(const Params &p)
{
  static SmemOptIn state;
  const size_t bytes = frame_index_smem(p);
  return bytes > 48 * 1024 ? raise_dynamic_smem(frame_index_kernel, state, bytes) : 0;
}

// stereo frames: row index + grid; mono / RGB-D frames (image_stride 1): grid only
void launch_frame_index(const Params &p, int n_frames, int image_stride, bool with_rowindex, cudaStream_t s)
{
  frame_index_kernel<<<with_rowindex ? 2 * n_frames : n_frames, kGridThreads, frame_index_smem(p), s>>>(p, n_frames, image_stride, with_rowindex ? 1 : 0);
}

} // namespace orbx
