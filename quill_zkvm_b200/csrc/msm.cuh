// Internal interface of the MSM pipeline (msm.cu), shared with the multi-GPU layer (comm.cu).
#pragma once
#include <cstddef>
#include <cstdint>
#include "ctx.cuh"
#include "ff.cuh"

struct qz_srs {
  qz_ctx* ctx;
  uint8_t* bases;  // n affine G1 points on the device, 64 B each (x ‖ y Montgomery; all-zero = infinity)
  size_t n;
  uint8_t* pre;    // optional: pre_W x n affine points, pre[w * n + i] = 2^(pre_c * w) * bases[i] (qz_srs_precompute)
  int pre_c, pre_W;
};

namespace qz {
// sum_i scalars[i] * srs->bases[i], i < n; scalars are Montgomery Fr on the device.  The result is written to device
// memory as XYZZ (128 B) and/or affine (64 B); either pointer may be null.  Asynchronous on ctx->stream.
int msm_device(qz_ctx* ctx, const qz_srs* srs, const uint4* scalars_dev, size_t n, uint8_t* out_xyzz_dev,
               uint8_t* out_affine_dev);
// the same with the scalars in host memory (scalars_host non-null): they are copied into scalars_dev range by range
// on a second stream, overlapped with the accumulation of the previous range.  `first`: the scalars belong to the bases
// first, first + 1, .. (a rank's index range of an MSM over an SRS every rank holds: qz_msm_split)
int msm_run(qz_ctx* ctx, const qz_srs* srs, uint4* scalars_dev, const void* scalars_host, size_t n,
            uint8_t* out_xyzz_dev, uint8_t* out_affine_dev, size_t first = 0);
// KZG::open on the device: x read from device memory, y (32 B) and the affine proof (64 B) written to device memory
int kzg_open_device(qz_ctx* ctx, const qz_srs* srs, const uint4* pdev, size_t n_coeffs,
                    const Fp<FrParams>* x_dev, Fp<FrParams>* y_dev, uint8_t* proof_affine_dev);
// affine(sum of n XYZZ points on the device) -> out_affine_dev (64 B)
int msm_sum_points_launch(qz_ctx* ctx, const uint8_t* pts_dev, int n, uint8_t* out_affine_dev);
// every rank's XYZZ partial sum `mine` (128 B, device; `all`: 128 B per rank) -> their affine sum in out_dev.  With peer
// mailboxes *pinned_fault is set to a pinned word that is non-zero after the stream synchronises if a peer timed out.
int msm_exchange_sum(qz_ctx* ctx, uint8_t* mine, uint8_t* all, uint8_t* out_dev, uint32_t** pinned_fault);

// the C-ABI MSMs qz_msm, qz_msm_sharded and qz_msm_split, by `mode`: arguments checked, scalars staged, the affine
// result copied to out_xy (host memory) and the call's timings recorded
enum class MsmMode { local, sharded, split };
int msm_call(qz_ctx* ctx, const qz_srs* srs, const void* scalars, size_t n_scalars, int on_device, MsmMode mode,
             uint8_t out_xy[64]);
}  // namespace qz
