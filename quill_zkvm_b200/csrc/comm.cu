// Multi-GPU layer: one process per GPU, NCCL over NVLink for the two tiny exchanges the path has (SURVEY 8e):
//   * MSM: bases/scalars are split by index range; each rank runs the whole single-GPU pipeline to one XYZZ partial
//     sum, the partial sums are all-gathered as raw limbs (128 B per rank) and added with the group law on every rank;
//   * sumcheck: tables are split by the top variables; per round the ranks all-gather (deg+1) partial sums (sumcheck.cu).
// NCCL is bound at run time with dlopen (the image carries it inside the torch wheel), so building this library needs
// no NCCL headers and a single-GPU user never loads it.  Group elements are never reduced with ncclSum.
#include <dlfcn.h>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <vector>
#include "comm.cuh"
#include "ctx.cuh"
#include "ec.cuh"
#include "msm.cuh"

namespace {

// minimal NCCL surface (stable ABI since 2.x)
typedef struct {
  char internal[128];
} ncclUniqueIdT;
typedef int ncclResultT;
typedef ncclResultT (*fn_GetUniqueId)(ncclUniqueIdT*);
typedef ncclResultT (*fn_CommInitRank)(ncclComm**, int, ncclUniqueIdT, int);
typedef ncclResultT (*fn_CommDestroy)(ncclComm*);
typedef ncclResultT (*fn_AllGather)(const void*, void*, size_t, int /*ncclDataType_t*/, ncclComm*, cudaStream_t);
typedef const char* (*fn_GetErrorString)(ncclResultT);
constexpr int NCCL_UINT8 = 1;  // ncclUint8

struct NcclApi {
  void* handle = nullptr;
  fn_GetUniqueId GetUniqueId = nullptr;
  fn_CommInitRank CommInitRank = nullptr;
  fn_CommDestroy CommDestroy = nullptr;
  fn_AllGather AllGather = nullptr;
  fn_GetErrorString GetErrorString = nullptr;
  bool ok() const { return handle && GetUniqueId && CommInitRank && AllGather; }
};

NcclApi& nccl() {
  static NcclApi api;
  if (api.handle) return api;
  const char* env = getenv("QZ_NCCL_LIB");
  const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    if (!n || !*n) continue;
    api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (api.handle) break;
  }
  if (!api.handle) return api;
  api.GetUniqueId = (fn_GetUniqueId)dlsym(api.handle, "ncclGetUniqueId");
  api.CommInitRank = (fn_CommInitRank)dlsym(api.handle, "ncclCommInitRank");
  api.CommDestroy = (fn_CommDestroy)dlsym(api.handle, "ncclCommDestroy");
  api.AllGather = (fn_AllGather)dlsym(api.handle, "ncclAllGather");
  api.GetErrorString = (fn_GetErrorString)dlsym(api.handle, "ncclGetErrorString");
  return api;
}

}  // namespace

namespace qz {

// all-gather `bytes` from every rank into recv (rank-major) on the context's stream
int comm_allgather(qz_ctx* ctx, const void* send, void* recv, size_t bytes) {
  if (ctx->nranks == 1) {
    if (send != recv) QZ_CUDA(ctx, cudaMemcpyAsync(recv, send, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return QZ_OK;
  }
  NcclApi& api = nccl();
  if (!api.ok() || !ctx->comm) return ctx->fail(QZ_ERR_NCCL, "communicator not initialised");
  ncclResultT r = api.AllGather(send, recv, bytes, NCCL_UINT8, ctx->comm, ctx->stream);
  if (r != 0) return ctx->fail(QZ_ERR_NCCL, api.GetErrorString ? api.GetErrorString(r) : "ncclAllGather failed");
  return QZ_OK;
}

static void peers_close(qz_ctx* ctx) {
  for (int g = 0; g < QZ_MAX_PEERS; g++) {
    if (ctx->peer_mbox_host[g] && g != ctx->rank) cudaIpcCloseMemHandle(ctx->peer_mbox_host[g]);
    ctx->peer_mbox_host[g] = nullptr;
  }
  if (ctx->peer_mbox_dev) cudaFree(ctx->peer_mbox_dev);
  if (ctx->mbox) cudaFree(ctx->mbox);
  ctx->peer_mbox_dev = nullptr;
  ctx->mbox = nullptr;
  cudaGetLastError();
}

// Map every rank's mailbox into this process (CUDA IPC over the NVLink / NVSwitch peer path).  The 64-byte IPC handles
// travel through the communicator that was just created.  Every rank takes the same decision: a second all-gather
// carries each rank's "all peers opened" bit, and the mailboxes are used only if it is set everywhere; otherwise
// (restricted CUDA_VISIBLE_DEVICES, no peer access, QZ_NO_P2P=1) the exchanges stay on NCCL all-gathers.
static int peers_exchange_handles(qz_ctx* ctx, uint8_t* xchg, int& ok) {
  const int G = ctx->nranks;
  cudaStream_t st = ctx->stream;
  uint8_t* d_mine = xchg + (size_t)128 * G;
  cudaIpcMemHandle_t mine;
  memset(&mine, 0, sizeof mine);
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  if (ok) {
    if (cudaMalloc(&ctx->mbox, sizeof(PeerMailbox)) != cudaSuccess ||
        cudaMemset(ctx->mbox, 0, sizeof(PeerMailbox)) != cudaSuccess ||
        cudaIpcGetMemHandle(&mine, ctx->mbox) != cudaSuccess) {
      cudaGetLastError();
      ok = 0;
    }
  }
  std::vector<uint8_t> all((size_t)64 * G);
  QZ_CUDA(ctx, cudaMemcpyAsync(d_mine, &mine, 64, cudaMemcpyHostToDevice, st));
  int rc = comm_allgather(ctx, d_mine, xchg, 64);
  if (rc) return rc;
  QZ_CUDA(ctx, cudaMemcpyAsync(all.data(), xchg, (size_t)64 * G, cudaMemcpyDeviceToHost, st));
  QZ_CUDA(ctx, cudaStreamSynchronize(st));
  for (int g = 0; g < G && ok; g++) {
    if (g == ctx->rank) {
      ctx->peer_mbox_host[g] = ctx->mbox;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, all.data() + (size_t)64 * g, 64);
    bool zero = true;  // a rank that could not allocate its mailbox sends an all-zero handle
    for (int i = 0; i < 64; i++) zero = zero && all[(size_t)64 * g + i] == 0;
    if (zero || cudaIpcOpenMemHandle(&ctx->peer_mbox_host[g], h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
      cudaGetLastError();
      ctx->peer_mbox_host[g] = nullptr;
      ok = 0;
    }
  }
  // agree: everyone must have opened everything
  uint8_t flag = (uint8_t)ok;
  std::vector<uint8_t> flags(G);
  QZ_CUDA(ctx, cudaMemcpyAsync(d_mine, &flag, 1, cudaMemcpyHostToDevice, st));
  rc = comm_allgather(ctx, d_mine, xchg, 1);
  if (rc) return rc;
  QZ_CUDA(ctx, cudaMemcpyAsync(flags.data(), xchg, G, cudaMemcpyDeviceToHost, st));
  QZ_CUDA(ctx, cudaStreamSynchronize(st));
  for (int g = 0; g < G; g++) ok = ok && flags[g];
  return QZ_OK;
}

static int peers_setup(qz_ctx* ctx) {
  const int G = ctx->nranks;
  if (G > QZ_MAX_PEERS) return QZ_OK;
  uint8_t* xchg = nullptr;  // [G] handles / status bytes, then this rank's contribution
  QZ_CUDA(ctx, cudaMalloc((void**)&xchg, (size_t)128 * G + 128));
  int ok = getenv("QZ_NO_P2P") ? 0 : 1;
  const int rc = peers_exchange_handles(ctx, xchg, ok);
  cudaFree(xchg);
  if (rc || !ok) {
    peers_close(ctx);
    return rc;
  }
  QZ_CUDA(ctx, cudaMalloc((void**)&ctx->peer_mbox_dev, sizeof(void*) * QZ_MAX_PEERS));
  QZ_CUDA(ctx, cudaMemcpy(ctx->peer_mbox_dev, ctx->peer_mbox_host, sizeof(void*) * QZ_MAX_PEERS, cudaMemcpyHostToDevice));
  ctx->mbox_seq = 0;
  return QZ_OK;
}

void comm_destroy(qz_ctx* ctx) {
  peers_close(ctx);
  if (ctx->comm && nccl().CommDestroy) nccl().CommDestroy(ctx->comm);
  ctx->comm = nullptr;
}

}  // namespace qz

using namespace qz;

extern "C" {

int qz_comm_unique_id(uint8_t out_id[128]) {
  if (!out_id) return QZ_ERR_INVALID_ARG;
  NcclApi& api = nccl();
  if (!api.ok()) return QZ_ERR_NCCL;
  ncclUniqueIdT id;
  if (api.GetUniqueId(&id) != 0) return QZ_ERR_NCCL;
  memcpy(out_id, id.internal, 128);
  return QZ_OK;
}

int qz_comm_init(qz_ctx* ctx, const uint8_t unique_id[128], int rank, int nranks) {
  if (!ctx || !unique_id || nranks < 1 || rank < 0 || rank >= nranks) return QZ_ERR_INVALID_ARG;
  if (nranks & (nranks - 1)) return ctx->fail(QZ_ERR_INVALID_ARG, "rank count must be a power of two");
  QZ_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->rank = rank;
  ctx->nranks = nranks;
  if (nranks == 1) return QZ_OK;
  NcclApi& api = nccl();
  if (!api.ok()) return ctx->fail(QZ_ERR_NCCL, "libnccl.so.2 not found (set QZ_NCCL_LIB)");
  ncclUniqueIdT id;
  memcpy(id.internal, unique_id, 128);
  ncclResultT r = api.CommInitRank(&ctx->comm, nranks, id, rank);
  if (r != 0) return ctx->fail(QZ_ERR_NCCL, api.GetErrorString ? api.GetErrorString(r) : "ncclCommInitRank failed");
  return peers_setup(ctx);
}

int qz_comm_peer_memory(const qz_ctx* ctx) { return ctx && comm_has_peers(ctx) ? 1 : 0; }

// The MSM's one exchange through the peer mailboxes: this rank's XYZZ partial sum (4 x 32 B) goes into every rank's
// mailbox, the G partial sums are added with the group law (never ncclSum) and converted to affine -- one launch in
// place of ncclAllGather + msm_sum_points.
__global__ void __launch_bounds__(32) msm_sum_points_peers(const uint8_t* mine_xyzz, qz::PeerMailbox* const* peers, int rank,
                                                          int G, uint32_t seq, uint8_t* out_affine, uint32_t* fault) {
  using namespace qz;
  __shared__ Fr s_vals[4];
  if (threadIdx.x < 4) s_vals[threadIdx.x] = fp_load<FrParams>(mine_xyzz + 32 * threadIdx.x);  // raw limbs of x, y, zz, zzz
  __syncthreads();
  const PeerSlot* got = peer_exchange(peers, rank, G, seq, s_vals, 4);
  if (threadIdx.x == 0) {
    if (*reinterpret_cast<volatile uint32_t*>(&peers[rank]->timed_out)) *fault = 1;
    Xyzz total = xyzz_identity();
    for (int g = 0; g < G; g++) {
      Xyzz p;
      Fr w[4];
      for (int i = 0; i < 4; i++) w[i] = ld_fresh(&got->data[g][i]);
      for (int i = 0; i < 8; i++) {
        p.x.v[i] = w[0].v[i];
        p.y.v[i] = w[1].v[i];
        p.zz.v[i] = w[2].v[i];
        p.zzz.v[i] = w[3].v[i];
      }
      total = xyzz_add(total, p);
    }
    affine_store(out_affine, xyzz_to_affine_serial(total));
  }
}
}  // extern "C"

// all ranks' partial sums (`mine`: 128 B XYZZ on the device) -> affine sum on every rank
int qz::msm_exchange_sum(qz_ctx* ctx, uint8_t* mine, uint8_t* all, uint8_t* out_dev, uint32_t** pinned_fault) {
  const int G = ctx->nranks > 0 ? ctx->nranks : 1;
  if (G > 1 && qz::comm_has_peers(ctx)) {
    uint32_t* fault = (uint32_t*)ctx->arena_alloc(4);
    if (!fault) return ctx->fail(QZ_ERR_ALLOC, "fault flag");
    QZ_CUDA(ctx, cudaMemsetAsync(fault, 0, 4, ctx->stream));
    QZ_LAUNCH(ctx, msm_sum_points_peers, 1, 32, 0, (const uint8_t*)mine, (qz::PeerMailbox* const*)ctx->peer_mbox_dev, ctx->rank, G,
              ++ctx->mbox_seq, out_dev, fault);
    uint32_t* pin = (uint32_t*)ctx->pinned_buf(64);
    if (!pin) return ctx->fail(QZ_ERR_ALLOC, "pinned");
    QZ_CUDA(ctx, cudaMemcpyAsync(pin, fault, 4, cudaMemcpyDeviceToHost, ctx->stream));
    *pinned_fault = pin;
    return QZ_OK;
  }
  if (G > 1) {
    int rc = qz::comm_allgather(ctx, mine, all, 128);
    if (rc) return rc;
  } else {
    all = mine;
  }
  return qz::msm_sum_points_launch(ctx, all, G, out_dev);
}

extern "C" {

int qz_msm_sharded(qz_ctx* ctx, const qz_srs* srs, const void* scalars, size_t n_scalars, int on_device,
                   uint8_t out_xy[64]) {
  return msm_call(ctx, srs, scalars, n_scalars, on_device, MsmMode::sharded, out_xy);
}

// The same product when every rank holds the WHOLE SRS and the WHOLE scalar vector (HyperPlonk's witness and logup
// commits at N > 1): rank g takes the index range [n g / G, n (g + 1) / G), the 128-byte partial sums are gathered
// and added on every rank.  Without a communicator it is qz_kzg_commit.
int qz_msm_split(qz_ctx* ctx, const qz_srs* srs, const void* scalars, size_t n_scalars, int on_device, uint8_t out_xy[64]) {
  return msm_call(ctx, srs, scalars, n_scalars, on_device, MsmMode::split, out_xy);
}

// Re-agree on the mailbox sequence numbers after a sharded call failed somewhere (a rank that left a call early -- an
// allocation failure, a bad argument -- has consumed fewer exchange numbers than the others, and from then on every
// wait would time out).  Collective: every rank of the communicator calls it; all continue from the largest number
// any rank reached, a full ring of slots further, with the timed-out mark of their own mailbox cleared.
int qz_comm_resync(qz_ctx* ctx) {
  if (!ctx) return QZ_ERR_INVALID_ARG;
  if (ctx->nranks <= 1) return QZ_OK;
  QZ_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->arena_reset();
  cudaStream_t st = ctx->stream;
  QZ_CUDA(ctx, cudaStreamSynchronize(st));
  uint32_t mine[2] = {ctx->mbox_seq, ctx->gather_seq};
  uint32_t* d_mine = (uint32_t*)ctx->arena_alloc(8);
  uint32_t* d_all = (uint32_t*)ctx->arena_alloc((size_t)8 * ctx->nranks);
  if (!d_mine || !d_all) return ctx->fail(QZ_ERR_ALLOC, "resync scratch");
  QZ_CUDA(ctx, cudaMemcpyAsync(d_mine, mine, 8, cudaMemcpyHostToDevice, st));
  int rc = comm_allgather(ctx, d_mine, d_all, 8);
  if (rc) return rc;
  std::vector<uint32_t> all(2 * (size_t)ctx->nranks);
  QZ_CUDA(ctx, cudaMemcpyAsync(all.data(), d_all, 8 * (size_t)ctx->nranks, cudaMemcpyDeviceToHost, st));
  QZ_CUDA(ctx, cudaStreamSynchronize(st));
  uint32_t seq = 0, gseq = 0;
  for (int g = 0; g < ctx->nranks; g++) {
    seq = std::max(seq, all[2 * g]);
    gseq = std::max(gseq, all[2 * g + 1]);
  }
  ctx->mbox_seq = seq + 2 * MBOX_SLOTS;  // past every slot a straggler may still be writing
  ctx->gather_seq = gseq + 2;
  if (ctx->mbox)
    QZ_CUDA(ctx, cudaMemsetAsync(&((PeerMailbox*)ctx->mbox)->timed_out, 0, sizeof(uint32_t), st));
  // nobody may start the next exchange before everyone has cleared its mark and taken the new numbers
  rc = comm_allgather(ctx, d_mine, d_all, 8);
  if (rc) return rc;
  QZ_CUDA(ctx, cudaStreamSynchronize(st));
  return QZ_OK;
}

int qz_comm_allgather_host(qz_ctx* ctx, const void* send, void* recv, size_t bytes) {
  if (!ctx || !send || !recv) return QZ_ERR_INVALID_ARG;
  if (bytes == 0) return QZ_OK;
  QZ_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->arena_reset();
  cudaStream_t st = ctx->stream;
  uint8_t* mine = (uint8_t*)ctx->arena_alloc(bytes);
  uint8_t* all = (uint8_t*)ctx->arena_alloc(bytes * ctx->nranks);
  if (!mine || !all) return ctx->fail(QZ_ERR_ALLOC, "all-gather buffers");
  QZ_CUDA(ctx, cudaMemcpyAsync(mine, send, bytes, cudaMemcpyHostToDevice, st));
  int rc = comm_allgather(ctx, mine, all, bytes);
  if (rc) return rc;
  QZ_CUDA(ctx, cudaMemcpyAsync(recv, all, bytes * ctx->nranks, cudaMemcpyDeviceToHost, st));
  QZ_CUDA(ctx, cudaStreamSynchronize(st));
  return QZ_OK;
}

}  // extern "C"
