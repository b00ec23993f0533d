// Context shared by the C-ABI entry points: one device, one stream, a scratch arena, cached constants.
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>  // header-only; ranges are no-ops unless a profiler injects itself
#include <cstdint>
#include <cstdio>
#include <map>
#include <string>
#include <vector>
#include "../../include/quill_b200.h"

struct ncclComm;

// NVTX range per phase of a call (SURVEY section 5): the enqueue of the phase's kernels, visible in nsys / ncu --nvtx
struct QzRange {
  explicit QzRange(const char* name) { nvtxRangePushA(name); }
  ~QzRange() { nvtxRangePop(); }
  QzRange(const QzRange&) = delete;
  QzRange& operator=(const QzRange&) = delete;
};

struct qz_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int sm_count = 148;
  // programmatic dependent launches for the latency-bound rounds of the sumcheck chain (QZ_NO_PDL=1 turns them off).
  // Measured on B200 (tools/sc_pdl_ab.py): -5 us per such round (2^16 product proof 463 -> 440 us, 2^24 proof -28 us);
  // HyperPlonk's generic-expression chains are unaffected (2^20-row proof 2.215 s either way).
  bool pdl = true;
  std::string err;
  uint64_t launches = 0;

  // scratch arena: bump allocation out of cached device blocks, reset at the start of every API call
  struct Block {
    void* p;
    size_t cap, off;
  };
  std::vector<Block> blocks;

  // Device buffers handed to the caller (qz_dev_alloc / the S polynomial of qz_mlpcs_open_begin) come from a pool:
  // qz_dev_free parks a block here instead of calling cudaFree, which is a device-wide synchronisation and, on a
  // prover that allocates and frees the same few hundred MiB per proof, was measured at 0.2 .. 2.5 s per HyperPlonk
  // proof (and growing).  A request reuses the smallest parked block that is large enough and at most 1/8 larger.
  std::multimap<size_t, void*> pool_parked;
  std::map<void*, size_t> pool_live;
  void pool_trim() {
    for (auto& kv : pool_parked) cudaFree(kv.second);
    pool_parked.clear();
  }
  void* pool_alloc(size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    if (bytes == 0) bytes = 256;
    auto it = pool_parked.lower_bound(bytes);
    if (it != pool_parked.end() && it->first <= bytes + bytes / 8 + ((size_t)1 << 16)) {
      void* p = it->second;
      pool_live[p] = it->first;
      pool_parked.erase(it);
      return p;
    }
    void* p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) {
      cudaGetLastError();
      pool_trim();  // give the parked blocks back and try once more
      if (cudaMalloc(&p, bytes) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
      }
    }
    pool_live[p] = bytes;
    return p;
  }
  cudaError_t pool_release(void* p) {
    if (!p) return cudaSuccess;
    auto it = pool_live.find(p);
    if (it == pool_live.end()) return cudaFree(p);  // not ours (e.g. allocated before the pool existed)
    pool_parked.emplace(it->second, p);
    pool_live.erase(it);
    return cudaSuccess;
  }

  // cached device constants: interpolation matrices keyed by degree (< 1000), NTT twiddle tables keyed by 1000 + log2 size
  std::map<int, void*> cache;
  // resident blocks per SM by (kernel, block size): the runtime is asked once per context (sumcheck.cu blocks_per_sm)
  std::map<std::pair<const void*, int>, int> occupancy;

  cudaEvent_t ev_call0 = nullptr, ev_call1 = nullptr, ev_k0 = nullptr, ev_k1 = nullptr;

  // streamed MSM (msm.cu): the scalars' host->device copy, digit extraction and sort of segment s+1 run on `prep_stream`
  // while `stream` accumulates segment s.  Created on first use, destroyed with the context.
  static constexpr int MAX_SEGMENTS = 8;
  cudaStream_t prep_stream = nullptr;
  cudaEvent_t ev_entry = nullptr, ev_seg_ready[MAX_SEGMENTS] = {}, ev_acc0[MAX_SEGMENTS] = {}, ev_acc1[MAX_SEGMENTS] = {};
  int acc_launches = 0;  // accumulate launches of the last MSM whose durations ev_acc0/1 bracket (0: ev_k0/ev_k1 do)
  int ensure_prep_stream() {
    if (prep_stream) return 0;
    if (cudaStreamCreateWithFlags(&prep_stream, cudaStreamNonBlocking) != cudaSuccess) return 1;
    if (cudaEventCreateWithFlags(&ev_entry, cudaEventDisableTiming) != cudaSuccess) return 1;
    for (int i = 0; i < MAX_SEGMENTS; i++) {
      if (cudaEventCreateWithFlags(&ev_seg_ready[i], cudaEventDisableTiming) != cudaSuccess) return 1;
      if (cudaEventCreate(&ev_acc0[i]) != cudaSuccess || cudaEventCreate(&ev_acc1[i]) != cudaSuccess) return 1;
    }
    return 0;
  }
  void destroy_prep_stream() {
    if (!prep_stream) return;
    cudaStreamSynchronize(prep_stream);
    cudaStreamDestroy(prep_stream);
    cudaEventDestroy(ev_entry);
    for (int i = 0; i < MAX_SEGMENTS; i++) {
      cudaEventDestroy(ev_seg_ready[i]);
      cudaEventDestroy(ev_acc0[i]);
      cudaEventDestroy(ev_acc1[i]);
    }
    prep_stream = nullptr;
  }
  // every msm_accumulate launch since the last qz_msm_accumulate_stats(reset) is bracketed by an event pair of this ring
  // (grown on demand, reused after a reset), so that a caller that runs many MSMs per step (MLPCS open: 5, HyperPlonk:
  // ~140) can report the dominant kernel's share and its integer-pipe fraction for the whole step
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> acc_ring;
  size_t acc_ring_used = 0;
  double acc_ring_adds = 0;  // sorted entries of those launches (upper bound of the additions: zero digits are skipped)
  unsigned long long* acc_nonzero_dev = nullptr;  // non-zero digits = additions executed, counted by msm_digits
  bool acc_ring_on = false;
  int acc_ring_next(cudaEvent_t* e0, cudaEvent_t* e1) {
    if (!acc_ring_on) return 1;
    if (acc_ring_used == acc_ring.size()) {
      cudaEvent_t a = nullptr, b = nullptr;
      if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return 1;
      acc_ring.emplace_back(a, b);
    }
    *e0 = acc_ring[acc_ring_used].first;
    *e1 = acc_ring[acc_ring_used].second;
    acc_ring_used++;
    return 0;
  }
  float last_ms[2] = {0.f, 0.f};
  double last_stat[4] = {0, 0, 0, 0};  // last MSM: window bits, digits per scalar, shared bucket set (0/1), mixed additions

  // pinned staging for small results
  void* pinned = nullptr;
  size_t pinned_cap = 0;

  ncclComm* comm = nullptr;
  int rank = 0, nranks = 1;
  // peer mailboxes (comm.cuh): this rank's mailbox, the device array of all ranks' mailbox pointers (own included),
  // the peers' mapped pointers (to close them) and the sequence number of the last exchange
  void* mbox = nullptr;
  void** peer_mbox_dev = nullptr;
  void* peer_mbox_host[16] = {};
  uint32_t mbox_seq = 0;
  uint32_t* pending_fault = nullptr;  // pinned word the current sharded MSM's exchange kernel reports a peer timeout in
  uint32_t gather_seq = 0;  // sharded sumchecks handed over through the mailboxes' gather areas so far (picks the copy)

  int fail(int status, const char* what, cudaError_t ce = cudaSuccess) {
    char buf[512];
    if (ce != cudaSuccess)
      snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(ce));
    else
      snprintf(buf, sizeof buf, "%s", what);
    err = buf;
    // An entry point may fail after it enqueued copies from the caller's buffers or kernels on the prep stream: drain
    // both before the caller sees the error, so that it may free or reuse its buffers and the next call's arena reset
    // cannot hand out scratch that is still being written.
    if (stream_busy_possible) {
      if (stream) cudaStreamSynchronize(stream);
      if (prep_stream) cudaStreamSynchronize(prep_stream);
      cudaGetLastError();
    }
    return status;
  }
  bool stream_busy_possible = true;

  void arena_reset() {
    if (blocks.size() > 1) {  // coalesce into one block for the next call
      size_t total = 0;
      for (auto& b : blocks) {
        total += b.cap;
        cudaFree(b.p);
      }
      blocks.clear();
      void* p = nullptr;
      if (cudaMalloc(&p, total) != cudaSuccess) {
        cudaGetLastError();
        pool_trim();
        if (cudaMalloc(&p, total) != cudaSuccess) {
          cudaGetLastError();
          p = nullptr;  // start over from an empty arena: arena_alloc grows it block by block
        }
      }
      if (p) blocks.push_back(Block{p, total, 0});
    }
    for (auto& b : blocks) b.off = 0;
  }
  void* arena_alloc(size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    if (bytes == 0) bytes = 256;
    for (auto& b : blocks)
      if (b.cap - b.off >= bytes) {
        void* r = (char*)b.p + b.off;
        b.off += bytes;
        return r;
      }
    size_t cap = bytes < ((size_t)64 << 20) ? ((size_t)64 << 20) : bytes;
    void* p = nullptr;
    if (cudaMalloc(&p, cap) != cudaSuccess) {
      cudaGetLastError();
      if (pool_parked.empty()) return nullptr;
      pool_trim();  // the parked caller buffers are the only memory this library can give back
      if (cudaMalloc(&p, cap) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
      }
    }
    blocks.push_back(Block{p, cap, bytes});
    return p;
  }
  // nested scratch: offsets at the time of the mark are restored on release (blocks added later are emptied)
  std::vector<size_t> arena_mark() const {
    std::vector<size_t> m;
    for (auto& b : blocks) m.push_back(b.off);
    return m;
  }
  void arena_release(const std::vector<size_t>& m) {
    for (size_t i = 0; i < blocks.size(); i++) blocks[i].off = i < m.size() ? m[i] : 0;
  }
  void* pinned_buf(size_t bytes) {
    if (bytes > pinned_cap) {
      if (pinned) cudaFreeHost(pinned);
      pinned = nullptr;
      pinned_cap = 0;
      size_t cap = bytes < 65536 ? 65536 : bytes;
      if (cudaMallocHost(&pinned, cap) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
      }
      pinned_cap = cap;
    }
    return pinned;
  }
};

#define QZ_CUDA(ctx, call)                                              \
  do {                                                                  \
    cudaError_t e_ = (call);                                            \
    if (e_ != cudaSuccess) return (ctx)->fail(QZ_ERR_CUDA, #call, e_);  \
  } while (0)

// kernel launch with launch accounting; errors surface at the next QZ_CUDA / sync
#define QZ_LAUNCH_ON(ctx, strm, kernel, grid, block, smem, ...)                \
  do {                                                                        \
    kernel<<<(grid), (block), (smem), (strm)>>>(__VA_ARGS__);                 \
    (ctx)->launches++;                                                        \
    cudaError_t e_ = cudaPeekAtLastError();                                   \
    if (e_ != cudaSuccess) return (ctx)->fail(QZ_ERR_CUDA, #kernel, e_);      \
  } while (0)
#define QZ_LAUNCH(ctx, kernel, grid, block, smem, ...) \
  QZ_LAUNCH_ON(ctx, (ctx)->stream, kernel, grid, block, smem, __VA_ARGS__)

// Programmatic dependent launch for chains of short dependent kernels (the sumcheck rounds): the kernel may become
// resident while its predecessor in the stream still runs and parks at grid_dep_wait(), so launch processing and block
// scheduling overlap the predecessor instead of following it.  Kernels launched this way MUST call grid_dep_wait()
// before touching anything the predecessor writes; the call is a no-op under an ordinary launch.  `pdl` false (or
// QZ_NO_PDL set when the context was created) degrades to an ordinary launch.
#define QZ_LAUNCH_PDL(ctx, pdl, kernel, grid, block, ...)                                  \
  do {                                                                                     \
    cudaLaunchConfig_t cfg_ = {};                                                          \
    cfg_.gridDim = dim3(grid);                                                             \
    cfg_.blockDim = dim3(block);                                                           \
    cfg_.stream = (ctx)->stream;                                                           \
    cudaLaunchAttribute at_[1];                                                            \
    at_[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                        \
    at_[0].val.programmaticStreamSerializationAllowed = 1;                                 \
    cfg_.attrs = at_;                                                                      \
    cfg_.numAttrs = (pdl) ? 1 : 0;                                                         \
    cudaError_t e_ = cudaLaunchKernelEx(&cfg_, kernel, __VA_ARGS__);                       \
    (ctx)->launches++;                                                                     \
    if (e_ != cudaSuccess) return (ctx)->fail(QZ_ERR_CUDA, #kernel, e_);                   \
  } while (0)
