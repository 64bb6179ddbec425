// orbx_sequence.cu -- whole sequences sharded by frame over GPUs, behind the C ABI (include/orbx.h, "sequences").
//
// Replaces the dataset loop of the reference's examples (example/Stereo/KittiStereo.cc:28-37: for every frame
// Frame::createStereo, include/ORB_SLAM2/Frame.h:313-322) for offline map / vocabulary building, where frames are
// independent: rank r of R takes the contiguous block [r * ceil(F/R), min(F, (r + 1) * ceil(F/R))) (SURVEY.md section 8e),
// streams it through the context's device slots (H2D of one chunk, kernels of another, D2H of a third overlap on the
// pipeline streams) and leaves every frame's results as ONE fixed-stride record (orbx_record_layout), so that a chunk of
// frames leaves the device in a single copy.  The only exchange between ranks is the gather of the left descriptors
// (north_star: "only the descriptor gather is collected"), in one of two transports:
//   NCCL   piecewise grouped ncclSend/ncclRecv on a side stream while later chunks are still being computed
//   peer   the pack kernel that assembles the records stores the descriptors straight into every rank's gathered array
//          through peer pointers (same process: cudaDeviceEnablePeerAccess; other processes: CUDA IPC handles) -- the
//          gather is fused into the kernel that produces the data and rides NVLink as plain stores
// For an offline map export (orbx_sequence_stereo_keyframes) every chunk also runs, after its pack kernel, the
// bag-of-words descent and assembly and the serialiser on its own slots, so that each frame additionally leaves the
// device as the KeyFrameData record of a keyframe made from it; those records stay on their rank.
#include <dlfcn.h>

#include <algorithm>
#include <cstring>
#include <memory>
#include <mutex>

#include "orbx_internal.h"

using namespace orbx;

namespace
{

// ---- NCCL, resolved at run time (dlopen): a single-GPU host needs no NCCL installed -------------------------------
typedef struct ncclComm *nccl_comm_t;
struct NcclId
{
  char internal[ORBX_COMM_ID_BYTES];
};
struct NcclApi
{
  void *lib = nullptr;
  int (*GetUniqueId)(NcclId *) = nullptr;
  int (*CommInitRank)(nccl_comm_t *, int, NcclId, int) = nullptr;
  int (*CommDestroy)(nccl_comm_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  int (*Send)(const void *, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
  int (*Recv)(void *, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
  int (*AllGather)(const void *, void *, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
  int (*AllReduce)(const void *, void *, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
  bool ok = false;
};
constexpr int kNcclUint8 = 1, kNcclInt32 = 2, kNcclSum = 0; // ncclDataType_t / ncclRedOp_t values of nccl.h (stable since 2.0)

NcclApi &nccl()
{
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    // a process that already carries an NCCL (e.g. the one bundled with PyTorch) hands back that copy for the same soname
    for (const char *name : {"libnccl.so.2", "libnccl.so"})
      if ((api.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL))) break;
    if (!api.lib) return;
    auto sym = [&](const char *n) { return dlsym(api.lib, n); };
    api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
    api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
    api.Send = (decltype(api.Send))sym("ncclSend");
    api.Recv = (decltype(api.Recv))sym("ncclRecv");
    api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
    api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
    api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
    api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.GroupStart && api.GroupEnd && api.Send && api.Recv && api.AllGather &&
             api.AllReduce && api.GetErrorString;
  });
  return api;
}

#define ORBX_NCCL(ctx, expr)                                                                                                   \
  do                                                                                                                           \
  {                                                                                                                            \
    int r__ = (expr);                                                                                                          \
    if (r__ != 0) return orbx::fail((ctx), ORBX_ERR_COMM, std::string(#expr) + ": " + nccl().GetErrorString(r__));            \
  } while (0)

constexpr int kMaxRanks = 16;
constexpr int kPieceEvents = orbx_ctx::kPipeMax;

inline size_t up16(size_t v) { return (v + 15) & ~(size_t)15; }

// gathered arrays of one rank: [world * block][N][32] descriptors followed by [world * block] counts, ONE allocation so
// that one IPC handle covers both
struct Gathered
{
  uint8_t *base = nullptr;
  size_t desc_bytes = 0; // offset of the counts
  int64_t cap_frames = 0;
  uint8_t *desc() const { return base; }
  int32_t *n() const { return reinterpret_cast<int32_t *>(base + desc_bytes); }
};

} // namespace

struct orbx_comm
{
  orbx_ctx *ctx = nullptr;
  int rank = 0, world = 1;
  int transport = ORBX_TRANSPORT_NONE;
  int64_t max_frames = 0; // capacity in frames of the whole sequence (all ranks agree)
  Gathered g;             // this rank's gathered arrays
  // peer transport: every rank's gathered base as seen from this device (own entry = g.base)
  uint8_t *peer_base[kMaxRanks] = {};
  bool peer_opened[kMaxRanks] = {}; // mapped through cudaIpcOpenMemHandle (to be closed)
  // NCCL
  nccl_comm_t nccl_comm = nullptr;
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t piece_ev[kPieceEvents] = {};
  int32_t *d_flag = nullptr; // all-reduce scratch for the closing barrier
  int piece_frames = 64;
};

namespace
{

int gathered_alloc(orbx_ctx *c, Gathered &g, int64_t world, int64_t max_frames)
{
  const int64_t block = (max_frames + world - 1) / world;
  const int64_t cap = std::max<int64_t>(1, block * world);
  const size_t N = (size_t)c->cfg.n_features;
  g.desc_bytes = up16((size_t)cap * N * 32);
  const size_t total = g.desc_bytes + up16((size_t)cap * 4);
  ORBX_CUDA(c, cudaMalloc((void **)&g.base, total));
  ORBX_CUDA(c, cudaMemset(g.base, 0, total));
  g.cap_frames = cap;
  return ORBX_OK;
}

// ---- pack kernel -------------------------------------------------------------------------------------------------
// One frame's results leave the slot buffers (interleaved left/right images, orbx_device.cuh) as one record:
//   int32 n_left, n_right, n_matches, 0 | kps_left[N] (undistorted) | desc_left[N][32] | kps_right[N] | desc_right[N][32] |
//   u_right[N] f64 | depth[N] f64          (offsets: orbx_record_layout; entries beyond the counts are zero)
// and the left descriptors + count go to row `gframe` of the gathered arrays of every rank in `peers` (peer transport: all
// ranks, i.e. the descriptor gather is these stores; otherwise only this rank's own array, which NCCL then exchanges).
struct PackArgs
{
  uint8_t *rec;         // record of the launch's first frame (device), or null
  size_t rec_stride;
  orbx_record_layout lay;
  int64_t gframe0;      // global index of the launch's first frame
  int n_peers;
  uint8_t *peer_desc[kMaxRanks];
  int32_t *peer_n[kMaxRanks];
};

constexpr int kPackThreads = 256;
constexpr int kPackBlocksPerFrame = 8;

// copies `valid` bytes and zero-fills up to `total` (both multiples of 4; 16-byte vectors when everything is aligned)
__device__ __forceinline__ void copy_fill(uint8_t *__restrict__ dst, const uint8_t *__restrict__ src, size_t valid, size_t total, int t, int nt)
{
  if ((((size_t)dst | (size_t)src | valid | total) & 15) == 0)
  {
    uint4 *d = reinterpret_cast<uint4 *>(dst);
    const uint4 *s = reinterpret_cast<const uint4 *>(src);
    const size_t nv = valid >> 4, n = total >> 4;
    for (size_t i = t; i < n; i += nt) d[i] = i < nv ? s[i] : make_uint4(0u, 0u, 0u, 0u);
  }
  else
  {
    uint32_t *d = reinterpret_cast<uint32_t *>(dst);
    const uint32_t *s = reinterpret_cast<const uint32_t *>(src);
    const size_t nv = valid >> 2, n = total >> 2;
    for (size_t i = t; i < n; i += nt) d[i] = i < nv ? s[i] : 0u;
  }
}

__global__ void __launch_bounds__(kPackThreads) pack_records_kernel(const Params p, const PackArgs a)
{
  const int f = blockIdx.y; // frame of this launch (slot-relative: p is already offset to the slot)
  const int t = blockIdx.x * kPackThreads + threadIdx.x, nt = gridDim.x * kPackThreads;
  const size_t N = (size_t)p.n_features;
  const int nl = p.n_kps[2 * f], nr = p.n_kps[2 * f + 1];
  const uint8_t *kl = reinterpret_cast<const uint8_t *>(p.kps_und + (size_t)(2 * f) * N);
  const uint8_t *kr = reinterpret_cast<const uint8_t *>(p.kps + (size_t)(2 * f + 1) * N);
  const uint8_t *dl = p.desc + (size_t)(2 * f) * N * 32, *dr = p.desc + (size_t)(2 * f + 1) * N * 32;
  if (a.rec)
  {
    uint8_t *r = a.rec + (size_t)f * a.rec_stride;
    if (t == 0) *reinterpret_cast<int4 *>(r) = make_int4(nl, nr, p.n_matches[f], 0);
    copy_fill(r + a.lay.off_kps_left, kl, (size_t)nl * 28, N * 28, t, nt);
    copy_fill(r + a.lay.off_desc_left, dl, (size_t)nl * 32, N * 32, t, nt);
    copy_fill(r + a.lay.off_kps_right, kr, (size_t)nr * 28, N * 28, t, nt);
    copy_fill(r + a.lay.off_desc_right, dr, (size_t)nr * 32, N * 32, t, nt);
    copy_fill(r + a.lay.off_u_right, reinterpret_cast<const uint8_t *>(p.u_right + (size_t)f * N), (size_t)nl * 8, N * 8, t, nt);
    copy_fill(r + a.lay.off_depth, reinterpret_cast<const uint8_t *>(p.depth + (size_t)f * N), (size_t)nl * 8, N * 8, t, nt);
  }
  const size_t grow = (size_t)(a.gframe0 + f);
  for (int k = 0; k < a.n_peers; ++k)
  {
    copy_fill(a.peer_desc[k] + grow * N * 32, dl, (size_t)nl * 32, N * 32, t, nt);
    if (t == 0) a.peer_n[k][grow] = nl;
  }
}

// keyframe records of the chunk in device slots [d0, d0 + nf) = local frames [f0, f0 + nf), on the chunk's stream after its
// pack kernel: bag-of-words descent + assembly into the slots' BoW buffers (with a vocabulary), then the serialiser.  The
// slots hold stereo frames (image stride 2) whatever the context's previous call left resident.
int keyframe_chunk(orbx_ctx *c, const orbx_keyframe_io *kio, const Params &p, cudaStream_t s, size_t d0, int64_t f0, int nf, int64_t lo)
{
  const size_t ks = kio->stride;
  const bool host = !kio->on_device;
  // host outputs: per slot `ks` bytes of record, then per slot 12 floats of pose; the sizes of the whole block
  uint8_t *stage = host ? c->kf_staging.p + d0 * ks : nullptr;
  float *stage_pose = host ? reinterpret_cast<float *>(c->kf_staging.p + (size_t)c->cfg.max_batch * ks) + d0 * 12 : nullptr;
  const float *pose = nullptr;
  if (kio->pose_rt)
  {
    if (host) ORBX_CUDA(c, cudaMemcpyAsync(stage_pose, kio->pose_rt + (size_t)f0 * 12, (size_t)nf * 12 * sizeof(float), cudaMemcpyHostToDevice, s));
    pose = host ? stage_pose : kio->pose_rt + (size_t)f0 * 12;
  }
  SerArgs sa = ser_args(c, 2, host ? stage : kio->out + (size_t)f0 * ks, ks, (host ? reinterpret_cast<int64_t *>(c->kf_sizes.p) : kio->sizes) + f0,
                        kio->id0 + (uint64_t)(lo + f0), pose, kio->with_map_points);
  if (kio->vocab)
  {
    const BowArgs ba = bow_at(bow_args(c, kio->vocab, kio->levelsup, 2), d0, (size_t)c->cfg.n_features);
    launch_bow_descend(p, ba, nf, s);
    launch_bow_assemble(p, ba, nf, s);
    c->launches += 2;
    ser_bow_inputs(sa, ba);
  }
  launch_serialize(p, sa, nf, s);
  ++c->launches;
  ORBX_CUDA(c, cudaGetLastError());
  if (host) ORBX_CUDA(c, cudaMemcpyAsync(kio->out + (size_t)f0 * ks, stage, ks * nf, cudaMemcpyDeviceToHost, s));
  return ORBX_OK;
}

void comm_free(orbx_comm *m)
{
  if (!m) return;
  if (m->ctx) cudaSetDevice(m->ctx->device);
  if (m->comm_stream) cudaStreamSynchronize(m->comm_stream);
  for (int r = 0; r < kMaxRanks; ++r)
    if (m->peer_opened[r] && m->peer_base[r]) cudaIpcCloseMemHandle(m->peer_base[r]);
  if (m->nccl_comm && nccl().ok) nccl().CommDestroy(m->nccl_comm);
  for (auto &e : m->piece_ev)
    if (e) cudaEventDestroy(e);
  if (m->comm_stream) cudaStreamDestroy(m->comm_stream);
  if (m->d_flag) cudaFree(m->d_flag);
  if (m->g.base) cudaFree(m->g.base);
  delete m;
}

int comm_common_init(orbx_ctx *c, orbx_comm *m, int rank, int world, int64_t max_frames)
{
  m->ctx = c;
  m->rank = rank;
  m->world = world;
  m->max_frames = max_frames;
  ORBX_CUDA(c, cudaSetDevice(c->device));
  int rc = gathered_alloc(c, m->g, world, max_frames);
  if (rc) return rc;
  m->peer_base[rank] = m->g.base;
  if (const char *e = std::getenv("ORBX_PIECE")) m->piece_frames = std::max(1, std::atoi(e));
  return ORBX_OK;
}

} // namespace

extern "C"
{

  void orbx_frame_range(int64_t n_frames_total, int rank, int world, int64_t *lo, int64_t *hi)
  {
    const int64_t F = std::max<int64_t>(0, n_frames_total), R = std::max(1, world);
    const int64_t block = (F + R - 1) / R;
    if (lo) *lo = std::min(F, (int64_t)rank * block);
    if (hi) *hi = std::min(F, ((int64_t)rank + 1) * block);
  }

  int orbx_record_layout_get(const orbx_ctx *c, orbx_record_layout *out)
  {
    if (!c || !out) return ORBX_ERR_INVALID_ARG;
    const size_t N = (size_t)c->cfg.n_features;
    size_t o = 16;
    out->n_features = (int32_t)N;
    out->reserved = 0;
    out->off_kps_left = (int64_t)o, o = up16(o + N * 28);
    out->off_desc_left = (int64_t)o, o = up16(o + N * 32);
    out->off_kps_right = (int64_t)o, o = up16(o + N * 28);
    out->off_desc_right = (int64_t)o, o = up16(o + N * 32);
    out->off_u_right = (int64_t)o, o = up16(o + N * 8);
    out->off_depth = (int64_t)o, o = up16(o + N * 8);
    out->record_bytes = (int64_t)o;
    return ORBX_OK;
  }

  int orbx_comm_unique_id(uint8_t *id)
  {
    if (!id) return ORBX_ERR_INVALID_ARG;
    if (!nccl().ok) return ORBX_ERR_COMM;
    NcclId nid;
    if (nccl().GetUniqueId(&nid) != 0) return ORBX_ERR_COMM;
    std::memcpy(id, nid.internal, ORBX_COMM_ID_BYTES);
    return ORBX_OK;
  }

  int orbx_comm_create(orbx_ctx *c, int rank, int world, const uint8_t *id, int64_t max_frames_total, orbx_comm **out)
  {
    if (!c || !out || !id || world < 1 || world > kMaxRanks || rank < 0 || rank >= world || max_frames_total < 0) return ORBX_ERR_INVALID_ARG;
    *out = nullptr;
    if (!nccl().ok) return fail(c, ORBX_ERR_COMM, "libnccl.so.2 could not be loaded (dlopen) -- multi-process sequences need NCCL");
    orbx_comm *m = new orbx_comm();
    int rc = comm_common_init(c, m, rank, world, max_frames_total);
    if (rc)
    {
      comm_free(m);
      return rc;
    }
    m->transport = ORBX_TRANSPORT_NCCL;
    NcclId nid;
    std::memcpy(nid.internal, id, ORBX_COMM_ID_BYTES);
    auto bail = [&](int code, const std::string &msg) {
      comm_free(m);
      return fail(c, code, msg);
    };
    int r = nccl().CommInitRank(&m->nccl_comm, world, nid, rank);
    if (r != 0) return bail(ORBX_ERR_COMM, std::string("ncclCommInitRank: ") + nccl().GetErrorString(r));
    if (cudaStreamCreateWithFlags(&m->comm_stream, cudaStreamNonBlocking) != cudaSuccess) return bail(ORBX_ERR_CUDA, "cudaStreamCreate (comm)");
    for (auto &e : m->piece_ev)
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return bail(ORBX_ERR_CUDA, "cudaEventCreate (comm)");
    if (cudaMalloc((void **)&m->d_flag, 256) != cudaSuccess || cudaMemset(m->d_flag, 0, 256) != cudaSuccess) return bail(ORBX_ERR_CUDA, "cudaMalloc (comm flag)");
    *out = m;
    return ORBX_OK;
  }

  int orbx_comm_create_local(orbx_ctx *const *ctxs, int world, int64_t max_frames_total, orbx_comm **out)
  {
    if (!ctxs || !out || world < 1 || world > kMaxRanks || max_frames_total < 0) return ORBX_ERR_INVALID_ARG;
    for (int r = 0; r < world; ++r)
    {
      out[r] = nullptr;
      if (!ctxs[r]) return ORBX_ERR_INVALID_ARG;
      if (ctxs[r]->cfg.n_features != ctxs[0]->cfg.n_features) return fail(ctxs[r], ORBX_ERR_INVALID_ARG, "all ranks must share n_features");
    }
    int rc = ORBX_OK;
    for (int r = 0; r < world && rc == ORBX_OK; ++r)
    {
      out[r] = new orbx_comm();
      out[r]->transport = ORBX_TRANSPORT_PEER;
      rc = comm_common_init(ctxs[r], out[r], r, world, max_frames_total);
    }
    // every rank stores into every other rank's arrays: same device = same address space; another device needs peer access
    for (int r = 0; r < world && rc == ORBX_OK; ++r)
      for (int q = 0; q < world && rc == ORBX_OK; ++q)
      {
        out[r]->peer_base[q] = out[q]->g.base;
        const int dr = ctxs[r]->device, dq = ctxs[q]->device;
        if (dr == dq) continue;
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, dr, dq) != cudaSuccess || !can)
        {
          rc = fail(ctxs[r], ORBX_ERR_COMM, "devices of a local communicator cannot access each other's memory");
          break;
        }
        cudaSetDevice(dr);
        const cudaError_t e = cudaDeviceEnablePeerAccess(dq, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) rc = fail(ctxs[r], ORBX_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
        (void)cudaGetLastError();
      }
    if (rc != ORBX_OK)
      for (int r = 0; r < world; ++r)
      {
        comm_free(out[r]);
        out[r] = nullptr;
      }
    return rc;
  }

  int orbx_comm_ipc_handle(orbx_comm *m, uint8_t *handle)
  {
    if (!m || !handle) return ORBX_ERR_INVALID_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == ORBX_IPC_HANDLE_BYTES, "IPC handle size");
    ORBX_CUDA(m->ctx, cudaSetDevice(m->ctx->device));
    cudaIpcMemHandle_t h;
    ORBX_CUDA(m->ctx, cudaIpcGetMemHandle(&h, m->g.base));
    std::memcpy(handle, &h, sizeof(h));
    return ORBX_OK;
  }

  int orbx_comm_open_peers(orbx_comm *m, const uint8_t *handles)
  {
    if (!m || !handles) return ORBX_ERR_INVALID_ARG;
    if (m->transport != ORBX_TRANSPORT_NCCL) return fail(m->ctx, ORBX_ERR_STATE, "peer handles belong to a multi-process (NCCL) communicator");
    ORBX_CUDA(m->ctx, cudaSetDevice(m->ctx->device));
    for (int r = 0; r < m->world; ++r)
    {
      if (r == m->rank) continue;
      cudaIpcMemHandle_t h;
      std::memcpy(&h, handles + (size_t)r * ORBX_IPC_HANDLE_BYTES, sizeof(h));
      void *ptr = nullptr;
      ORBX_CUDA(m->ctx, cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
      m->peer_base[r] = (uint8_t *)ptr;
      m->peer_opened[r] = true;
    }
    m->transport = ORBX_TRANSPORT_PEER; // data path: stores through the peer pointers; NCCL stays for the closing barrier
    return ORBX_OK;
  }

  void orbx_comm_destroy(orbx_comm *m) { comm_free(m); }

  int orbx_comm_info(const orbx_comm *m, int32_t *rank, int32_t *world, int32_t *transport)
  {
    if (!m) return ORBX_ERR_INVALID_ARG;
    if (rank) *rank = m->rank;
    if (world) *world = m->world;
    if (transport) *transport = m->transport;
    return ORBX_OK;
  }

  int orbx_sequence_stereo(orbx_ctx *c, orbx_comm *m, int64_t n_frames_total, const orbx_sequence_io *io, orbx_sequence_result *res)
  {
    return orbx_sequence_stereo_keyframes(c, m, n_frames_total, io, nullptr, res);
  }

  int orbx_sequence_stereo_keyframes(orbx_ctx *c, orbx_comm *m, int64_t n_frames_total, const orbx_sequence_io *io, const orbx_keyframe_io *kio,
                                     orbx_sequence_result *res)
  {
    if (!c || !io || n_frames_total < 0 || !io->left || !io->right) return ORBX_ERR_INVALID_ARG;
    if (m && m->ctx != c) return fail(c, ORBX_ERR_INVALID_ARG, "communicator belongs to another context");
    if (kio && kio->vocab && kio->vocab->ctx != c) return fail(c, ORBX_ERR_INVALID_ARG, "vocabulary belongs to another context");
    ORBX_CUDA(c, cudaSetDevice(c->device));
    if (!m)
    { // single rank: the context keeps its own gathered arrays
      if (c->self_comm && c->self_comm->max_frames < n_frames_total)
      {
        ORBX_CUDA(c, cudaDeviceSynchronize());
        comm_free(c->self_comm);
        c->self_comm = nullptr;
      }
      if (!c->self_comm)
      {
        c->self_comm = new orbx_comm();
        int rc = comm_common_init(c, c->self_comm, 0, 1, n_frames_total);
        if (rc)
        {
          comm_free(c->self_comm);
          c->self_comm = nullptr;
          return rc;
        }
      }
      m = c->self_comm;
    }
    if (n_frames_total > m->max_frames) return fail(c, ORBX_ERR_CAPACITY, "sequence longer than the communicator's max_frames_total");
    const int R = m->world, me = m->rank;
    const int64_t F = n_frames_total, block = (F + R - 1) / R;
    int64_t lo, hi;
    orbx_frame_range(F, me, R, &lo, &hi);
    const int64_t n_local = hi - lo;
    orbx_record_layout lay;
    orbx_record_layout_get(c, &lay);
    const size_t rs = io->records ? io->record_stride : (size_t)lay.record_bytes;
    if (io->records && (rs < (size_t)lay.record_bytes || (rs & 15) || ((size_t)io->records & 15)))
      return fail(c, ORBX_ERR_INVALID_ARG, "records must be 16-byte aligned with a stride >= orbx_record_layout.record_bytes that is a multiple of 16");
    const bool rec_dev = io->records && io->records_on_device, rec_host = io->records && !io->records_on_device;
    if (rec_host)
    {
      int rc = c->rec_staging.reserve(c, (size_t)c->cfg.max_batch * rs);
      if (rc) return rc;
    }
    const size_t N = (size_t)c->cfg.n_features;
    const bool kf_bow = kio && kio->vocab, kf_host = kio && !kio->on_device;
    if (kio)
    {
      if (n_local > 0 && (!kio->out || !kio->sizes)) return fail(c, ORBX_ERR_INVALID_ARG, "keyframe io needs `out` and `sizes`");
      if ((kio->stride & 15) || ((size_t)kio->out & 15))
        return fail(c, ORBX_ERR_INVALID_ARG, "keyframe records must be 16-byte aligned with a stride that is a multiple of 16");
      if ((int64_t)kio->stride < (kf_bow ? orbx_serialized_capacity_bow(c) : orbx_serialized_capacity(c)))
        return fail(c, ORBX_ERR_CAPACITY, kf_bow ? "keyframe stride is smaller than orbx_serialized_capacity_bow()" : "keyframe stride is smaller than orbx_serialized_capacity()");
      int rc = kf_bow ? bow_buffers(c) : ORBX_OK;
      if (!rc && kf_host) rc = c->kf_staging.reserve(c, (size_t)c->cfg.max_batch * (kio->stride + 12 * sizeof(float)));
      if (!rc && kf_host) rc = c->kf_sizes.reserve(c, (size_t)std::max<int64_t>(1, n_local) * sizeof(int64_t));
      if (rc) return rc;
    }

    const bool use_nccl = m->transport == ORBX_TRANSPORT_NCCL && R > 1;
    // padding rows of this rank's block (ragged last block) carry a zero count; on the context's stream, so that the fork of
    // the pipeline streams orders everything after it
    if (n_local < block)
    {
      if (m->transport == ORBX_TRANSPORT_PEER)
      {
        for (int r = 0; r < R; ++r)
          ORBX_CUDA(c, cudaMemsetAsync(reinterpret_cast<int32_t *>(m->peer_base[r] + m->g.desc_bytes) + me * block + n_local, 0, (size_t)(block - n_local) * 4, c->stream));
      }
      else
        ORBX_CUDA(c, cudaMemsetAsync(m->g.n() + me * block + n_local, 0, (size_t)(block - n_local) * 4, c->stream));
    }

    PackArgs pa{};
    pa.rec_stride = rs;
    pa.lay = lay;
    if (m->transport == ORBX_TRANSPORT_PEER)
    {
      pa.n_peers = R;
      for (int r = 0; r < R; ++r)
      {
        if (!m->peer_base[r]) return fail(c, ORBX_ERR_STATE, "peer transport: orbx_comm_open_peers has not mapped every rank");
        pa.peer_desc[r] = m->peer_base[r];
        pa.peer_n[r] = reinterpret_cast<int32_t *>(m->peer_base[r] + m->g.desc_bytes);
      }
    }
    else
    {
      pa.n_peers = 1;
      pa.peer_desc[0] = m->g.desc();
      pa.peer_n[0] = m->g.n();
    }

    // NCCL: the block is exchanged in pieces of piece_frames frames (a multiple of the chunk) on the comm stream while later
    // chunks are still being computed; every rank runs the same number of pieces over the PADDED block so that the grouped
    // send/recv calls match.  A piece is ready once everything enqueued so far on the pipeline streams has run (which
    // also orders the comm stream after the fork of the pipeline streams from the context's stream).
    const int chunk = c->chunk();
    const int piece = std::max(chunk, (m->piece_frames / chunk) * chunk);
    const int64_t n_pieces = use_nccl ? (block + piece - 1) / piece : 0;
    int64_t next_piece = 0;
    auto exchange_piece = [&](int64_t g) -> int {
      const int64_t f0 = g * piece, cnt = std::min<int64_t>(piece, block - f0);
      for (int i = 0; i < c->kPipe; ++i)
      {
        ORBX_CUDA(c, cudaEventRecord(m->piece_ev[i], c->pipe[i]));
        ORBX_CUDA(c, cudaStreamWaitEvent(m->comm_stream, m->piece_ev[i], 0));
      }
      ORBX_NCCL(c, nccl().GroupStart());
      for (int r = 0; r < R; ++r)
      {
        if (r == me) continue;
        ORBX_NCCL(c, nccl().Send(m->g.desc() + (size_t)(me * block + f0) * N * 32, (size_t)cnt * N * 32, kNcclUint8, r, m->nccl_comm, m->comm_stream));
        ORBX_NCCL(c, nccl().Recv(m->g.desc() + (size_t)(r * block + f0) * N * 32, (size_t)cnt * N * 32, kNcclUint8, r, m->nccl_comm, m->comm_stream));
      }
      ORBX_NCCL(c, nccl().GroupEnd());
      return ORBX_OK;
    };

    // per chunk on its pipeline stream: pack -> record copy -> keyframe records -> the NCCL pieces it completes
    auto chunk_out = [&](cudaStream_t s, int d0, int64_t f0, int nf) -> int {
      const Params p = params_at(c, 2 * d0, d0);
      pa.rec = rec_dev ? (uint8_t *)io->records + (size_t)f0 * rs : (rec_host ? c->rec_staging.p + (size_t)d0 * rs : nullptr);
      pa.gframe0 = me * block + f0;
      pack_records_kernel<<<dim3(kPackBlocksPerFrame, nf), kPackThreads, 0, s>>>(p, pa);
      ++c->launches;
      ORBX_CUDA(c, cudaGetLastError());
      if (rec_host) ORBX_CUDA(c, cudaMemcpyAsync((uint8_t *)io->records + (size_t)f0 * rs, c->rec_staging.p + (size_t)d0 * rs, rs * nf, cudaMemcpyDeviceToHost, s));
      if (kio)
      {
        int rc = keyframe_chunk(c, kio, p, s, d0, f0, nf, lo);
        if (rc) return rc;
      }
      const int64_t done = f0 + nf;
      while (next_piece < n_pieces && done >= std::min<int64_t>(n_local, (next_piece + 1) * piece))
      {
        int rc = exchange_piece(next_piece++);
        if (rc) return rc;
      }
      return ORBX_OK;
    };
    int rc = run_stereo_chunks(c, n_local, io->left, io->stride, io->right, io->stride, io->frame_stride, io->input_on_device != 0, true, chunk_out);
    if (rc) return rc;
    while (next_piece < n_pieces)
    { // an empty block, or pieces that lie entirely in this rank's padding
      rc = exchange_piece(next_piece++);
      if (rc) return rc;
    }
    for (int i = 0; i < c->kPipe; ++i) ORBX_CUDA(c, cudaStreamSynchronize(c->pipe[i]));
    if (R > 1 && m->nccl_comm)
    {
      if (use_nccl)
        ORBX_NCCL(c, nccl().AllGather(m->g.n() + me * block, m->g.n(), (size_t)block, kNcclInt32, m->nccl_comm, m->comm_stream));
      else // peer stores of every rank have landed once every rank got here: a one-word all-reduce is the barrier
        ORBX_NCCL(c, nccl().AllReduce(m->d_flag, m->d_flag + 1, 1, kNcclInt32, kNcclSum, m->nccl_comm, m->comm_stream));
      ORBX_CUDA(c, cudaStreamSynchronize(m->comm_stream));
    }
    if (kf_host && n_local > 0) ORBX_CUDA(c, cudaMemcpy(kio->sizes, c->kf_sizes.p, (size_t)n_local * sizeof(int64_t), cudaMemcpyDeviceToHost));
    if (io->gathered_desc_host) ORBX_CUDA(c, cudaMemcpy(io->gathered_desc_host, m->g.desc(), (size_t)F * N * 32, cudaMemcpyDeviceToHost));
    if (io->gathered_n_host) ORBX_CUDA(c, cudaMemcpy(io->gathered_n_host, m->g.n(), (size_t)F * 4, cudaMemcpyDeviceToHost));

    if (res)
    {
      res->frame_lo = lo;
      res->frame_hi = hi;
      res->block = block;
      res->gathered_desc = m->g.desc();
      res->gathered_n = m->g.n();
      res->n_features = (int32_t)N;
      res->world = R;
    }
    return ORBX_OK;
  }

} // extern "C"

namespace orbx
{
// records of device slots [d0, d0 + nf) -> d_rec (device), no gather
int pack_frame_records(orbx_ctx *c, cudaStream_t s, int d0, int nf, uint8_t *d_rec, size_t rec_stride)
{
  PackArgs pa{};
  orbx_record_layout_get(c, &pa.lay);
  pa.rec = d_rec;
  pa.rec_stride = rec_stride;
  pa.n_peers = 0;
  const Params p = params_at(c, 2 * d0, d0);
  pack_records_kernel<<<dim3(kPackBlocksPerFrame, nf), kPackThreads, 0, s>>>(p, pa);
  ++c->launches;
  ORBX_CUDA(c, cudaGetLastError());
  return ORBX_OK;
}

void destroy_self_comm(orbx_ctx *c)
{
  if (c && c->self_comm)
  {
    comm_free(c->self_comm);
    c->self_comm = nullptr;
  }
}
} // namespace orbx
