// Linear-time sumcheck / zero-check prover on the device.
//
// Reference: SumcheckProof::prove (hyperplonk/src/piops/sumcheck.rs:28-114), ZeroCheckProof::prove
// (hyperplonk/src/piops/zerocheck.rs:14-49), fast_eq_eval_hypercube (hyperplonk/src/utils/eq_eval.rs:6-31).
//
// Structure (B200-first, not a translation of the reference's per-pair DensePolynomial loop):
//   * the tables stay in HBM for the whole proof; a round is ONE streaming pass that folds the previous round's
//     challenge into the tables (reads 4 consecutive elements, writes 2) and, in the same pass, evaluates the round
//     polynomial at X = 0..d on the freshly folded pairs -- 128 B of HBM traffic per input element over the proof;
//   * per-thread partial sums -> warp shuffles -> one partial per block -> a one-block "finalize" kernel that sums the
//     partials, interpolates to monomial coefficients, serialises them and runs the blake3 transcript ON THE DEVICE,
//     leaving the next challenge in device memory: no host round trip between rounds;
//   * once a rank's table is down to 2^SC_MID_LOG elements ONE persistent cooperative kernel (sc_mid) runs every remaining
//     round: a round's pairs are spread over the grid (split pass: one work item per folded element, then per (pair,
//     evaluation point)), the last block to arrive closes the round and releases the challenge to the others, peer GPUs
//     exchange through mailboxes from inside the kernel.
#include <algorithm>
#include <cstring>
#include <memory>
#include <mutex>
#include <vector>
#ifdef QZ_SC_TRACE
// measurement build (tools/sc_trace.py): thread 32 of a block stamps (id, block, clock64, globaltimer) at the marked points
namespace qz {
__device__ unsigned long long g_trace[3 * 8192];
__device__ unsigned int g_trace_n;
static __device__ __forceinline__ void sc_trace(int id) {
  if (threadIdx.x == 32) {  // a lane of warp 1: a divergent lane 0 in warp 0 slows the four-lane transcript several-fold
    const unsigned int i = atomicAdd(&g_trace_n, 1u);
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    if (i < 8192) {
      g_trace[3 * i] = (unsigned long long)id | ((unsigned long long)blockIdx.x << 16);
      g_trace[3 * i + 1] = (unsigned long long)clock64();
      g_trace[3 * i + 2] = gt;
    }
  }
}
}  // namespace qz
#define SC_TRACE(id)                                  \
  do {                                                \
    if (((QZ_SC_TRACE) >> (id)) & 1) sc_trace(id);    \
  } while (0)  // QZ_SC_TRACE = bit mask of the stamps to take
#endif
#include "comm.cuh"
#include "ctx.cuh"
#include "sumcheck.cuh"

namespace qz {

constexpr int SC_MID_LOG = 18;  // tables of at most 2^18 elements (per rank): sc_mid runs every remaining round in one launch
constexpr int SC_THREADS = 256;
constexpr int SC_WIDE_THREADS = 128;  // deferred-reduction round kernel: 168 registers, 3 blocks per SM
#ifndef QZ_SC_WIDE_BPS
#define QZ_SC_WIDE_BPS 4
#endif

// ---- loads ---------------------------------------------------------------------------------------------------------------
// The streaming passes ask L2 for the next pair's lines while the current pair is being multiplied: 2.615 -> 2.59 ms over
// the streaming rounds of a 2^24 proof (L1 as the target measured the same).  0 turns it off (tools/build_variant.sh).
#ifndef QZ_SC_PREFETCH
#define QZ_SC_PREFETCH 1
#endif
QZ_DEV void prefetch_line(const void* p) {
#if QZ_SC_PREFETCH == 1
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#elif QZ_SC_PREFETCH == 2
  asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
#else
  (void)p;
#endif
}
QZ_DEV Fr ld_elem(const uint4* base, uint64_t e) { return fp_load<FrParams>(base + 2 * e); }
QZ_DEV void st_elem(uint4* base, uint64_t e, const Fr& v) { fp_store<FrParams>(base + 2 * e, v); }
// the same load past L1 (ld.global.cv): for data another block -- or another GPU -- wrote during this kernel (sc_mid)
QZ_DEV Fr ld_elem_cv(const uint4* base, uint64_t e) {
  const uint4 a = __ldcv(base + 2 * e), b = __ldcv(base + 2 * e + 1);
  Fr r;
  r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w; r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  return r;
}
template <bool CV>
QZ_DEV Fr ld_elem_t(const uint4* base, uint64_t e) {
  return CV ? ld_elem_cv(base, e) : ld_elem(base, e);
}

// multiples of the pending challenge for fp_mul_fixed (ff.cuh), refreshed by the host with a device-to-device copy of the
// table sc_round_close left in device memory, before every pass that folds with it (the large passes).  Constant memory:
// the 64 words are instruction operands, not registers.  One table per device and process: sumcheck_run serialises the
// contexts of a device while it uses it.
__constant__ uint32_t c_fold[64];
// lo + r (hi - lo) with r given by the table
QZ_DEV Fr fold_fixed(const Fr& lo, const Fr& hi) {
  return fp_add<FrParams>(lo, fp_mul_fixed<FrParams>(fp_sub_lazy<FrParams>(hi, lo), c_fold));
}
// lo + r (hi - lo) with r in registers
QZ_DEV Fr fold_by(const Fr& lo, const Fr& hi, const Fr& r) {
  return fp_add<FrParams>(lo, fp_mul<FrParams>(r, fp_sub<FrParams>(hi, lo)));
}

// Pair p of a table, folding the pending challenge first when FOLD (sumcheck.rs:81-92 fused into the next round's
// pass): lo' = a0 + r (a1 - a0), hi' = a2 + r (a3 - a2), both written to the half-size table.  In two steps so that
// the streaming kernels issue all loads of a pair before any arithmetic: one memory round trip, not one per table, is
// exposed per pair (FOLD is a compile-time flag there: no branch splits the block the scheduler can hoist loads across).
template <bool FOLD>
struct RawPair {
  Fr e[FOLD ? 4 : 2];
};
template <bool FOLD, bool CV = false>
QZ_DEV void load_raw(const uint4* in, uint64_t p, RawPair<FOLD>& raw) {
#pragma unroll
  for (int j = 0; j < (FOLD ? 4 : 2); j++) raw.e[j] = ld_elem_t<CV>(in, (FOLD ? 4 : 2) * p + j);
}
template <bool FOLD, bool CF = false>
QZ_DEV void finish_pair(const RawPair<FOLD>& raw, uint4* out, uint64_t p, const Fr& r, Fr& lo, Fr& hi) {
  if (FOLD) {
    if (CF) {
      lo = fold_fixed(raw.e[0], raw.e[1]);
      hi = fold_fixed(raw.e[FOLD ? 2 : 0], raw.e[FOLD ? 3 : 1]);
    } else {
      lo = fold_by(raw.e[0], raw.e[1], r);
      hi = fold_by(raw.e[FOLD ? 2 : 0], raw.e[FOLD ? 3 : 1], r);
    }
    st_elem(out, 2 * p, lo);
    st_elem(out, 2 * p + 1, hi);
  } else {
    lo = raw.e[0];
    hi = raw.e[1];
  }
}
// the same with `fold` a run-time flag (the tail kernels)
template <bool CV = false, bool CF = false>
QZ_DEV void fetch_pair(const uint4* in, uint4* out, uint64_t p, bool fold, const Fr& r, Fr& lo, Fr& hi) {
  if (fold) {
    RawPair<true> raw;
    load_raw<true, CV>(in, p, raw);
    finish_pair<true, CF>(raw, out, p, r, lo, hi);
  } else {
    RawPair<false> raw;
    load_raw<false, CV>(in, p, raw);
    finish_pair<false>(raw, out, p, r, lo, hi);
  }
}

// ---- round kernel, fast path: h = g_0 * g_1 * ... * g_{K-1} --------------------------------------------------------------
// one pair of the product fast path: h = g_0 * ... * g_{K-1}.  Tables are taken two at a time: g_a(X) g_b(X) is a
// quadratic whose coefficients cost 3 products (lo*lo, hi*hi, df*df); its values at X = 0..K then follow by forward
// differences (adds only).  The per-X product over the pairs (and a leftover linear factor when K is odd) costs the
// remaining multiplications: 7 instead of 8 for K = 3, 11 instead of 15 for K = 4.
// per-thread running sums of h at X = 0..K.  WIDE (K >= 3 only): the last multiplication of every term only feeds the
// sum, so its Montgomery reduction is deferred: the 512-bit products accumulate in 17-word sums that are reduced once
// per thread (ff.cuh "deferred reduction") -- 64 instead of 128 multiply-adds for 4 of the 13 products of a K = 3 pair.
// The reduction costs 3 products per sum, so passes with only a few pairs per thread use the narrow sums.
// SKIP1: the value at X = 1 is not summed.  From round 1 on it follows from the previous round's TRUE polynomial,
// s_j(0) + s_j(1) = s_{j-1}(r_{j-1}) (an identity of the tables, whatever the prover's claim was: round 0 still sums
// every point, so a false claimed_sum is proved exactly as the reference proves it, zerocheck.rs:161-211), and the
// finalize step restores it (sc_expand_evals).  One product and one running sum less per pair.  The NS = K or K + 1
// sums are stored compactly: slot 0 = X 0, then X = 2.. (SKIP1) or X = 1.. .
template <int K, bool WIDE, bool SKIP1>
struct ProdAcc {
  static_assert(!WIDE || K >= 3, "nothing to defer below three factors");
  static constexpr int NS = SKIP1 ? K : K + 1;
  FpWide wide[WIDE ? NS : 1];
  Fr narrow[WIDE ? 1 : NS];
  static QZ_DEV constexpr int slot(int x) { return SKIP1 && x > 0 ? x - 1 : x; }
  QZ_DEV void init() {
    if (WIDE) {
#pragma unroll
      for (int x = 0; x < NS; x++) wide_zero(wide[x]);
    } else {
#pragma unroll
      for (int x = 0; x < NS; x++) narrow[x] = fp_zero<FrParams>();
    }
  }
  QZ_DEV void add_product(int x, const Fr& a, const Fr& b) {
    if (SKIP1 && x == 1) return;
    if (WIDE)
      wide_mul_acc<FrParams>(wide[WIDE ? slot(x) : 0], a, b);
    else
      add_value(x, fp_mul<FrParams>(a, b));
  }
  QZ_DEV void add_value(int x, const Fr& v) {
    if (SKIP1 && x == 1) return;
    narrow[WIDE ? 0 : slot(x)] = fp_add<FrParams>(narrow[WIDE ? 0 : slot(x)], v);
  }
  QZ_DEV Fr get_slot(int i) const { return WIDE ? wide_reduce<FrParams>(wide[WIDE ? i : 0]) : narrow[WIDE ? 0 : i]; }
};

// K = 3 with deferred reduction: the cubic is sampled at X = 0, 1, -1 and "infinity" (its leading coefficient) instead of
// X = 0 .. 3.  The quadratic g_0 g_1 = q0 + (q1 - q0 - q2) X + q2 X^2 already has its three samples q0 = q(0), q1 = q(1),
// q2 = q(inf) from the three products, q(-1) = 2 q0 + 2 q2 - q1 and g_2(-1) = 2 lo_2 - hi_2 are the only derived
// values, and every operand of a deferred-reduction product may be ANY 256-bit integer, so they are formed by plain
// additions: 4 modular differences' worth of carry-chain instructions per pair instead of 14 (forward differences of
// the quadratic and the linear factor up to X = 3).  The passes are bound by dependent-issue latency at four warps per
// scheduler, not by the multiplier alone (ncu: stall "wait" 2.7 per issue), so the ~250 fewer serial instructions per
// pair show up directly.  The slots are, in order, X = 0, 1, -1, inf (X = 1 absent under SKIP1); the finalize step
// turns them into coefficients (sc_toom3_to_coeffs).
template <bool SKIP1>
QZ_DEV void prod_core_toom3(const Fr* lo, const Fr* hi, ProdAcc<3, true, SKIP1>& acc) {
  const Fr q0 = fp_mul<FrParams>(lo[0], lo[1]);
  const Fr q1 = fp_mul<FrParams>(hi[0], hi[1]);
  const Fr d0 = fp_sub<FrParams>(hi[0], lo[0]);       // < p: the first operand of a reducing product
  const Fr d1 = fp_sub_lazy<FrParams>(hi[1], lo[1]);  // in (0, 2p)
  const Fr q2 = fp_mul<FrParams>(d0, d1);
  const Fr d2 = fp_sub_lazy<FrParams>(hi[2], lo[2]);  // leading coefficient of g_2, in (0, 2p)
  acc.add_product(0, q0, lo[2]);
  acc.add_product(1, q1, hi[2]);
  acc.add_product(3, q2, d2);
  // q(-1) = 2 (q0 + q2) + (p - q1) in (0, 5p), below 2^256 = 5.29 p;  g_2(-1) = lo_2 + (lo_2 - hi_2 + p) in (0, 3p)
  const Fr s02 = u256_add<FrParams>(q0, q2);
  const Fr qm = u256_add<FrParams>(u256_add<FrParams>(s02, s02), u256_p_minus<FrParams>(q1));
  const Fr gm = u256_add<FrParams>(lo[2], fp_sub_lazy<FrParams>(lo[2], hi[2]));
  acc.add_product(2, qm, gm);
}

// core of a pair once the K (lo, hi) values are in registers
template <int K, bool WIDE, bool SKIP1>
QZ_DEV void prod_core(const Fr* lo, const Fr* hi, ProdAcc<K, WIDE, SKIP1>& acc) {
  if constexpr (K == 3 && WIDE) {
    prod_core_toom3<SKIP1>(lo, hi, acc);
    return;
  }
  constexpr int NP = K / 2;
  Fr val[NP > 0 ? NP : 1], dl[NP > 0 ? NP : 1], q22[NP > 0 ? NP : 1], lin, lin_df;
#pragma unroll
  for (int t = 0; t < NP; t++) {
    const Fr q0 = fp_mul<FrParams>(lo[2 * t], lo[2 * t + 1]);                                   // q(0)
    const Fr q1v = fp_mul<FrParams>(hi[2 * t], hi[2 * t + 1]);                                  // q(1)
    const Fr q2 = fp_mul<FrParams>(fp_sub<FrParams>(hi[2 * t], lo[2 * t]),
                                   fp_sub<FrParams>(hi[2 * t + 1], lo[2 * t + 1]));             // X^2 coefficient
    val[t] = q0;
    dl[t] = fp_sub<FrParams>(q1v, q0);  // q(1) - q(0)
    q22[t] = fp_dbl<FrParams>(q2);      // second difference
  }
  if (K & 1) {
    lin = lo[K - 1];
    lin_df = fp_sub<FrParams>(hi[K - 1], lin);
  }
#pragma unroll
  for (int x = 0; x <= K; x++) {
    if (K >= 3) {
      // all factors but the last are multiplied with full reductions; the last product goes to the running sum
      Fr prod = val[0];
#pragma unroll
      for (int t = 1; t < NP - ((K & 1) ? 0 : 1); t++) prod = fp_mul<FrParams>(prod, val[t]);
      acc.add_product(x, prod, (K & 1) ? lin : val[NP - 1]);
    } else {
      acc.add_value(x, NP > 0 ? val[0] : lin);
    }
    if (x < K) {
#pragma unroll
      for (int t = 0; t < NP; t++) {
        val[t] = fp_add<FrParams>(val[t], dl[t]);   // q(x+1) = q(x) + (q(x+1) - q(x))
        dl[t] = fp_add<FrParams>(dl[t], q22[t]);    // first difference grows by 2*q2
      }
      if (K & 1) lin = fp_add<FrParams>(lin, lin_df);
    }
  }
}

// tail kernel: `fold` is a run-time flag, tables fetched one after the other
template <int K, bool WIDE, bool SKIP1 = false, bool CV = false>
QZ_DEV void prod_pair(const ScTables& tabs, uint64_t p, bool fold, const Fr& r, ProdAcc<K, WIDE, SKIP1>& acc) {
  Fr lo[K], hi[K];
#pragma unroll
  for (int t = 0; t < K; t++) fetch_pair<CV>(tabs.in[t], tabs.out[t], p, fold, r, lo[t], hi[t]);
  prod_core<K, WIDE, SKIP1>(lo, hi, acc);
}

// ---- round kernel, fast path ---------------------------------------------------------------------------------------------
// FOLD rounds (every round but the first) skip X = 1: NS = K sums per block instead of K + 1
template <int K, bool WIDE, bool FOLD>
__global__ void __launch_bounds__(WIDE ? SC_WIDE_THREADS : SC_THREADS, (WIDE ? (K <= 3 ? QZ_SC_WIDE_BPS : 3) : K <= 3 ? 2 : 1))
    sc_round_prod(ScTables tabs, uint64_t n_pairs, const ScHead* head, Fr* partials) {
  constexpr int NS = ProdAcc<K, WIDE, FOLD>::NS;
  __shared__ Fr s_part[(SC_THREADS / 32) * NS];
  grid_dep_launch();
  grid_dep_wait();
  ProdAcc<K, WIDE, FOLD> acc;
  acc.init();
  Fr r = fp_zero<FrParams>();
  if (FOLD) r = head->r;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_pairs; p += stride) {
    RawPair<FOLD> raw[K];
#pragma unroll
    for (int t = 0; t < K; t++) load_raw<FOLD>(tabs.in[t], p, raw[t]);
    if (QZ_SC_PREFETCH && p + stride < n_pairs) {
#pragma unroll
      for (int t = 0; t < K; t++) prefetch_line(tabs.in[t] + (FOLD ? 8 : 4) * (p + stride));
    }
    Fr lo[K], hi[K];
#pragma unroll
    for (int t = 0; t < K; t++) finish_pair<FOLD, WIDE>(raw[t], tabs.out[t], p, r, lo[t], hi[t]);  // WIDE passes fold by c_fold
    prod_core<K, WIDE, FOLD>(lo, hi, acc);
  }
  Fr sums[NS];
#pragma unroll
  for (int x = 0; x < NS; x++) sums[x] = acc.get_slot(x);
  block_sum_many(sums, NS, s_part, &partials[(size_t)blockIdx.x * NS]);
}

// ---- round kernel, zero-check fast path: h = g_0 * ... * g_{K-1}, summed against eq(., z) --------------------------------------
// eq(x, z) = prod_i eq(x_i, z_i) factors over the variables, so the round polynomial of h * eq is
//     s_j(X) = P_j * eq(X, z_j) * t_j(X),   t_j(X) = sum_{x'} E_{j+1}(x') * prod_t g_t(r_0 .. r_{j-1}, X, x'),
// with P_j = prod_{i<j} eq(r_i, z_i) and E_{j+1} the eq table of the variables above j.  Instead of streaming and folding
// eq as one more table of a degree-(K+1) product (zerocheck.rs:25-29 builds exactly that), the pass sums the degree-K
// polynomial t_j with one weight per pair -- 2 extra products per pair (the weight scales one factor) in place of 2 fold
// products + the extra evaluation point + the wider product -- and sc_round_close multiplies by the linear factor.
// The weight tables need no product to shrink: eq(0, z) + eq(1, z) = 1, so E_{j+2}[p] = E_{j+1}[2p] + E_{j+1}[2p+1],
// done in the same pass that folds the g tables.  s_j is the same polynomial, so every output byte is unchanged.
// SKIP1 (FOLD rounds of large proofs only): t_j(1) is restored from t_{j-1}(r_{j-1}) = (1 - z_j) t_j(0) + z_j t_j(1),
// which needs 1 / z_j (sc_begin inverts the z in one batch when asked to)
template <int K, bool WIDE, bool FOLD, bool SKIP1>
__global__ void __launch_bounds__(WIDE ? SC_WIDE_THREADS : SC_THREADS, (WIDE ? QZ_SC_WIDE_BPS : 2))
    sc_round_zc(ScTables tabs, const uint4* e_in, uint4* e_out, uint64_t n_pairs, const ScHead* head, Fr* partials) {
  static_assert(FOLD || !SKIP1, "round 0 sums every point");
  constexpr int NS = ProdAcc<K, WIDE, SKIP1>::NS;
  __shared__ Fr s_part[(SC_THREADS / 32) * NS];
  grid_dep_launch();
  grid_dep_wait();
  ProdAcc<K, WIDE, SKIP1> acc;
  acc.init();
  Fr r = fp_zero<FrParams>();
  if (FOLD) r = head->r;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_pairs; p += stride) {
    RawPair<FOLD> raw[K];
#pragma unroll
    for (int t = 0; t < K; t++) load_raw<FOLD>(tabs.in[t], p, raw[t]);
    // (no prefetch of the next pair here: it helps sc_round_prod by 1 % and costs this kernel 5 %)
    Fr w;
    if (FOLD) {
      w = fp_add<FrParams>(ld_elem(e_in, 2 * p), ld_elem(e_in, 2 * p + 1));
      st_elem(e_out, p, w);
    } else {
      w = ld_elem(e_in, p);
    }
    Fr lo[K], hi[K];
#pragma unroll
    for (int t = 0; t < K; t++) finish_pair<FOLD, WIDE>(raw[t], tabs.out[t], p, r, lo[t], hi[t]);
    lo[0] = fp_mul<FrParams>(w, lo[0]);
    hi[0] = fp_mul<FrParams>(w, hi[0]);
    prod_core<K, WIDE, SKIP1>(lo, hi, acc);
  }
  Fr sums[NS];
#pragma unroll
  for (int x = 0; x < NS; x++) sums[x] = acc.get_slot(x);
  block_sum_many(sums, NS, s_part, &partials[(size_t)blockIdx.x * NS]);
}
// (A variant of these kernels that staged each warp's tiles in shared memory with cp.async, one slot per table refilled a
// pair ahead, was built and measured in round 2: 3.59 ms against 3.19 ms for the streaming rounds of a 2^24 proof.  The
// passes are bound by the integer multiply pipe, not by the exposed load latency; the ring's copy / read / __syncwarp
// instructions and its spills only took issue slots from the multiplier.  Removed.)

// hand-over to sc_mid: the eq table in the form zerocheck.rs:25 would have left it after the same rounds, i.e. with
// the last challenge still to be folded in: out[2p + b] = P_{j-1} * eq(b, z_{j-1}) * E_j[p]
// The running claim changes meaning with it: the eq-factored rounds kept t_j(r_j), the rounds that follow sum h * eq as
// the reference does and expect s_j(r_j) = P_{j+1} t_j(r_j).
__global__ void __launch_bounds__(256) zc_materialize_eq(const uint4* e_tab, uint64_t half, ScHead* head, const Fr* z_prev,
                                                        uint4* out) {
  const uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p == 0) head->claim = fp_mul<FrParams>(head->zc_prefix, head->claim);
  if (p >= half) return;
  const Fr z = *z_prev, P = head->zc_prefix_prev, e = ld_elem(e_tab, p);
  const Fr hi = fp_mul<FrParams>(fp_mul<FrParams>(P, z), e);
  const Fr lo = fp_sub<FrParams>(fp_mul<FrParams>(P, e), hi);  // P (1 - z) E
  st_elem(out, 2 * p, lo);
  st_elem(out, 2 * p + 1, hi);
}

// ---- round kernel, generic expression tree -----------------------------------------------------------------------------------
// skip1: X = 1 is not evaluated (see ProdAcc); the sums are stored compactly, acc[0] = X 0, acc[x - 1] = X x >= 2
template <bool CV = false, bool CF = false>
QZ_DEV void generic_pair(const ScTables& tabs, uint64_t p, bool fold, const Fr& r, const uint32_t* s_ops,
                         uint32_t n_ops, int k, int d, const Fr* consts, Fr* acc, bool skip1 = false) {
  Fr cur[SC_MAX_K], df[SC_MAX_K];
  for (int t = 0; t < k; t++) {
    Fr hi;
    fetch_pair<CV, CF>(tabs.in[t], tabs.out[t], p, fold, r, cur[t], hi);
    df[t] = fp_sub<FrParams>(hi, cur[t]);
  }
  for (int x = 0; x <= d; x++) {
    if (!(skip1 && x == 1)) {
      const int sl = skip1 && x > 0 ? x - 1 : x;
      acc[sl] = fp_add<FrParams>(acc[sl], sc_eval_program(s_ops, n_ops, consts, cur));
    }
    if (x < d)
      for (int t = 0; t < k; t++) cur[t] = fp_add<FrParams>(cur[t], df[t]);
  }
}

// CF: fold by the challenge table in constant memory (large passes; the host refreshes c_fold first)
template <bool CF>
__global__ void __launch_bounds__(SC_THREADS) sc_round_generic(ScTables tabs, uint64_t n_pairs, int fold,
                                                              const ScHead* head, const ScProgram* prog,
                                                              const Fr* consts, Fr* partials) {
  __shared__ Fr s_part[(SC_THREADS / 32) * SC_MAX_COEFFS];
  __shared__ uint32_t s_ops[SC_MAX_OPS];
  grid_dep_launch();
  const uint32_t n_ops = prog->n_ops;  // the program and the constants are uploaded before the first round
  const int d = (int)prog->degree, k = (int)prog->k;
  for (uint32_t i = threadIdx.x; i < n_ops; i += blockDim.x) s_ops[i] = prog->ops[i];
  __syncthreads();
  grid_dep_wait();
  Fr acc[SC_MAX_COEFFS];
  for (int x = 0; x <= d; x++) acc[x] = fp_zero<FrParams>();
  Fr r = fp_zero<FrParams>();
  if (fold) r = head->r;
  const bool skip1 = fold != 0 && d >= 1;  // every round but the first (see ProdAcc)
  const int ns = skip1 ? d : d + 1;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_pairs; p += stride)
    generic_pair<false, CF>(tabs, p, fold != 0, r, s_ops, n_ops, k, d, consts, acc, skip1);
  block_sum_many(acc, ns, s_part, &partials[(size_t)blockIdx.x * ns]);
}

// ---- finalize: sum `n_parts` partial vectors, close the round (transcript on the device) -----------------------------------
// this thread's share of the sum of the n_parts vectors of ns values in `partials` (block_sum_many adds the shares)
QZ_DEV void sum_partials(const Fr* partials, int n_parts, int ns, Fr* v) {
  for (int x = 0; x < ns; x++) v[x] = fp_zero<FrParams>();
  for (int b = threadIdx.x; b < n_parts; b += blockDim.x)
    for (int x = 0; x < ns; x++) v[x] = fp_add<FrParams>(v[x], partials[(size_t)b * ns + x]);
}

// Sharded rounds with peer mailboxes (comm.cuh): this rank's ns sums in s_evals go to every rank's mailbox over NVLink,
// and s_evals[x] <- the sum of the G vectors addressed to this rank (field addition is exact, so the order does not
// matter): every rank runs the same transcript on the same sums and draws the same challenge.  Ends with a barrier.
QZ_DEV void peer_sum(PeerMailbox* const* peers, int rank, int G, uint32_t seq, ScHead* head, Fr* s_evals, int ns) {
  const PeerSlot* got = peer_exchange(peers, rank, G, seq, s_evals, ns);
  if (threadIdx.x == 0 && *reinterpret_cast<volatile uint32_t*>(&peers[rank]->timed_out)) head->peer_fault = 1;
  if ((int)threadIdx.x < ns) {
    Fr sum = fp_zero<FrParams>();
    for (int g = 0; g < G; g++) sum = fp_add<FrParams>(sum, ld_fresh(&got->data[g][threadIdx.x]));
    s_evals[threadIdx.x] = sum;
  }
  __syncthreads();
}

// derive1: the partial vectors hold ns = d sums (X = 0, 2, .., d); X = 1 is restored from the running claim
// (sc_expand_evals).  zc_zinv: 1 / z_j for that step on the eq-factored zero-check path.
__global__ void __launch_bounds__(SC_THREADS) sc_finalize(const Fr* partials, int n_parts, int d, ScHead* head,
                                                         const Fr* vinv, Fr* out_coeffs_row, uint32_t* out_len,
                                                         Fr* out_point_slot, int max_coeffs, const Fr* zc_z, int derive1,
                                                         const Fr* zc_zinv, uint32_t* foldc, int toom) {
  __shared__ Fr s_part[(SC_THREADS / 32) * SC_MAX_COEFFS];
  __shared__ Fr s_evals[SC_MAX_COEFFS];
  __shared__ Fr s_coef[SC_MAX_COEFFS];
  __shared__ Fr s_prod[SC_PROD_SLOTS];
  __shared__ __align__(16) uint32_t s_msg[SC_MSG_WORDS];
  grid_dep_launch();
  grid_dep_wait();
  const int ns = derive1 ? d : d + 1;
  Fr v[SC_MAX_COEFFS];
  sum_partials(partials, n_parts, ns, v);
  block_sum_many(v, ns, s_part, s_evals);
  if (derive1) sc_expand_evals(head, d, s_evals, zc_z, zc_zinv);
  if (toom) sc_toom3_to_coeffs(s_evals);  // the sums are samples at X = 0, 1, -1, inf (prod_core_toom3)
  sc_round_close(head, toom ? nullptr : vinv, d, s_evals, s_coef, s_msg, s_prod, out_coeffs_row, out_len, out_point_slot,
                 max_coeffs, zc_z, true, foldc);
}

// Sharded mode with peer mailboxes: ONE launch per round after the round kernel, in place of sc_reduce_partials +
// ncclAllGather + sc_finalize.
__global__ void __launch_bounds__(SC_THREADS) sc_finalize_peers(const Fr* partials, int n_parts, int d,
                                                               PeerMailbox* const* peers, int rank, int G, uint32_t seq,
                                                               ScHead* head, const Fr* vinv, Fr* out_coeffs_row,
                                                               uint32_t* out_len, Fr* out_point_slot, int max_coeffs,
                                                               const Fr* zc_z, int derive1, const Fr* zc_zinv,
                                                               uint32_t* foldc, int toom) {
  __shared__ Fr s_part[(SC_THREADS / 32) * SC_MAX_COEFFS];
  __shared__ Fr s_evals[SC_MAX_COEFFS];
  __shared__ Fr s_coef[SC_MAX_COEFFS];
  __shared__ Fr s_prod[SC_PROD_SLOTS];
  __shared__ __align__(16) uint32_t s_msg[SC_MSG_WORDS];
  grid_dep_launch();
  grid_dep_wait();
  const int ns = derive1 ? d : d + 1;
  Fr v[SC_MAX_COEFFS];
  sum_partials(partials, n_parts, ns, v);
  block_sum_many(v, ns, s_part, s_evals);
  peer_sum(peers, rank, G, seq, head, s_evals, ns);
  if (derive1) sc_expand_evals(head, d, s_evals, zc_z, zc_zinv);
  if (toom) sc_toom3_to_coeffs(s_evals);
  sc_round_close(head, toom ? nullptr : vinv, d, s_evals, s_coef, s_msg, s_prod, out_coeffs_row, out_len, out_point_slot,
                 max_coeffs, zc_z, true, foldc);
}

// reduce block partials to one vector per rank (sharded mode: the vectors are all-gathered, then sc_finalize)
__global__ void __launch_bounds__(SC_THREADS) sc_reduce_partials(const Fr* partials, int n_parts, int d, Fr* out) {
  __shared__ Fr s_part[(SC_THREADS / 32) * SC_MAX_COEFFS];
  Fr v[SC_MAX_COEFFS];
  sum_partials(partials, n_parts, d + 1, v);
  block_sum_many(v, d + 1, s_part, out);
}

// ---- the short rounds: one persistent kernel runs every remaining round ----------------------------------------------------------
// Once a table is down to 2^SC_MID_LOG elements a round is pure latency (two launches, ~30 us, whatever its size: r01).
// sc_mid takes the proof from there to the end in ONE launch.  While a round still has more pairs than one block has
// threads it is spread over the (co-resident, cooperatively launched) grid: every block folds and evaluates its pairs
// and parks one partial vector, the block that arrives LAST at the round's counter sums the vectors, closes the round
// (interpolation, blake3 transcript, challenge -- sc_round_close) and releases a flag the other blocks spin on.  Blocks
// whose index is beyond a round's pairs exit (rounds only shrink); from 2^SC_TAIL_LOG elements on block 0 is alone and no
// counter is touched.  Data written by other blocks during the kernel is read past L1 (ld.cv).
// Sharded proofs (G > 1): the closing block also exchanges the partial vector with the peers' mailboxes, exactly as
// sc_finalize_peers does, and when G x the local size is down to 2^SC_TAIL_LOG every rank stores its shard into every
// peer's gather area (rank order = index order) and finishes the remaining rounds alone -- no collective launch.
// in[t]: current tables of `size` elements; bufs.a / bufs.b: scratch of >= max(size, 2^SC_TAIL_LOG) / 2 elements per table.
struct ScTailBufs {
  uint4* a[SC_MAX_K];
  uint4* b[SC_MAX_K];
};
struct ScMidSync {
  unsigned int arrive;  // blocks that finished their share of a round, cumulative over the rounds
  unsigned int flag;    // number of rounds closed so far (release / acquire)
};
QZ_DEV unsigned int ld_acquire_gpu(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
QZ_DEV void st_release_gpu(unsigned int* p, unsigned int v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// one block's share of a round: pairs first, first + step, ... ; the ns sums land in acc[0 .. ns)
template <int KP, bool SKIP1>
QZ_DEV void mid_block_pass(const ScTables& view, uint64_t first, uint64_t step, uint64_t n_pairs, bool fold, const Fr& r,
                           const uint32_t* s_ops, uint32_t n_ops, int k, int d, const Fr* consts, Fr* acc) {
  if (KP > 0) {
    constexpr int KX = KP > 0 ? KP : 1;
    ProdAcc<KX, false, SKIP1> pa;
    pa.init();
    for (uint64_t p = first; p < n_pairs; p += step) prod_pair<KX, false, SKIP1, true>(view, p, fold, r, pa);
#pragma unroll
    for (int x = 0; x < ProdAcc<KX, false, SKIP1>::NS; x++) acc[x] = pa.get_slot(x);
  } else {
    for (int x = 0; x <= d; x++) acc[x] = fp_zero<FrParams>();
    for (uint64_t p = first; p < n_pairs; p += step) generic_pair<true>(view, p, fold, r, s_ops, n_ops, k, d, consts, acc, SKIP1);
  }
}

// ---- the split pass: a short round as two levels of products spread over the whole block ------------------------------------------
// A thread that owns a whole pair runs its 12 products (K = 3: 6 folds, 3 + 3 for the sums) one after the other -- a
// lone product is ~810 cycles of dependent carry chains (tools/latbench.cu) and nothing overlaps them, so a round costs
// ~7 us however few pairs it has (tools/sc_trace.py).  Here a tile of pairs is worked on by the whole block:
//   level 1: one work item per ELEMENT of the folded tables (2 k per pair): load 2, fold, store to the half-size table
//            and to shared memory;
//   level 2: one work item per (pair, evaluation point): the k values at X by additions, then the k - 1 products of
//            the fast path (or the interpreter) -- the same count as the quadratic trick of prod_core for K = 3.  The
//            threads form one row per evaluation point (32 * (8 / ns) threads, whole warps), so a thread only ever
//            sums one point and a row is reduced by one shuffle sum per thread.
// Two product latencies and a memory round trip for a tile of <= 32 pairs instead of twelve; larger tiles loop over
// the items and approach the multiplier's throughput.  The plan (blocks per round, pairs per block) is made by the
// host, which also sizes the grid with it, and travels as a kernel argument.
constexpr int SC_TILE_ELEMS = 512;  // shared-memory tile of the split pass, in field elements (16 KiB)
constexpr int SC_SPLIT_MAX_CHUNK = 128;  // pairs per block up to which a round runs the split pass
struct ScMidPlan {
  uint16_t nblk[SC_MAX_VARS];    // blocks that work on round j of this launch
  uint16_t future[SC_MAX_VARS];  // max of nblk over rounds >= j: blocks beyond it leave the kernel
  uint32_t chunk[SC_MAX_VARS];   // split rounds: pairs per block; 0: the round keeps whole pairs per thread
  uint32_t tile;                 // pairs per tile of the split pass
};
// does the shape fit the split pass, and with which tile?  k tables, at most d + 1 evaluation points
inline int mid_tile_pairs(int k, int d) {
  if (k > 8 || d + 1 > 8) return 0;
  int tile = 256;
  while (2 * k * tile > SC_TILE_ELEMS) tile >>= 1;
  return tile;
}
// rounds of an sc_mid launch from (size, pending) on; returns the grid it needs (<= cap)
inline unsigned int mid_make_plan(ScMidPlan& plan, uint64_t size, int pending, int k, int d, unsigned int cap, int G) {
  memset(&plan, 0, sizeof plan);
  const int tile = mid_tile_pairs(k, d);
  plan.tile = (uint32_t)tile;
  bool gathered = G == 1;
  int j = 0;
  while (j < SC_MAX_VARS) {
    if (!gathered && size * (uint64_t)G <= ((uint64_t)1 << SC_TAIL_LOG)) {
      size *= (uint64_t)G;
      gathered = true;
    }
    if (size <= 1 || (pending && size == 2)) break;
    const uint64_t n_pairs = pending ? size / 4 : size / 2;
    // split: at least 32 pairs per block (below that the round is two product latencies whatever the count).  Once a
    // block would get more than SC_SPLIT_MAX_CHUNK pairs its multiplier is busy either way and whole pairs per thread
    // (one pair per thread and more) need no tiles, no barriers and one product less per pair in round 0.
    // A round of up to 128 pairs stays on one block: two tiles cost ~3 us more than one, gathering the vectors of
    // several blocks ~5 us (tools/sc_trace.py).
    uint64_t nb = n_pairs <= 128 ? 1 : std::max<uint64_t>(1, std::min<uint64_t>((n_pairs + 31) / 32, cap));
    uint64_t ch = (n_pairs + nb - 1) / nb;
    if (tile > 0 && ch <= (uint64_t)SC_SPLIT_MAX_CHUNK) {
      nb = (n_pairs + ch - 1) / ch;
    } else {
      nb = std::max<uint64_t>(1, std::min<uint64_t>((n_pairs + SC_THREADS - 1) / SC_THREADS, cap));
      ch = 0;
    }
    plan.nblk[j] = (uint16_t)nb;
    plan.chunk[j] = (uint32_t)ch;
    if (pending) size >>= 1;
    pending = 1;
    j++;
  }
  uint16_t best = 1;
  for (int i = j - 1; i >= 0; i--) {
    best = std::max(best, plan.nblk[i]);
    plan.future[i] = best;
  }
  for (int i = j; i < SC_MAX_VARS; i++) plan.nblk[i] = plan.future[i] = 1;
  return best;
}

// this block's pairs [p_begin, p_end) of a round, tile by tile; dst[x] (x < ns <= 8) <- the block's sums.  Ends with a
// barrier.  s_tile: SC_TILE_ELEMS Fr of shared memory, s_rows: SC_THREADS / 32 Fr.
template <int KP>
QZ_DEV void mid_split_pass(const ScTables& view, uint64_t p_begin, uint64_t p_end, bool fold, bool skip1, const Fr& r,
                           const uint32_t* s_ops, uint32_t n_ops, int k, int ns, const Fr* consts, int tile_pairs,
                           Fr* s_tile, Fr* s_rows, Fr* dst) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wpr = 8 / ns, rw = 32 * wpr;             // warps / threads per row
  const int xi = tid / rw, ri = tid % rw;            // level 2: evaluation point index, position in its row
  const int x = skip1 && xi > 0 ? xi + 1 : xi;       // SKIP1 rounds: X = 0, 2, 3, ..
  Fr acc = fp_zero<FrParams>();
  for (uint64_t tile = p_begin; tile < p_end; tile += (uint64_t)tile_pairs) {
    const int np = (int)(p_end - tile < (uint64_t)tile_pairs ? p_end - tile : (uint64_t)tile_pairs);
    for (int item = tid; item < 2 * k * np; item += SC_THREADS) {
      const int ft = item / (2 * np), fe = item - ft * 2 * np;  // table, element of the tile
      const uint64_t idx = 2 * tile + (uint64_t)fe;             // element of the tables this round sums over
      Fr v;
      if (fold) {
        v = fold_by(ld_elem_cv(view.in[ft], 2 * idx), ld_elem_cv(view.in[ft], 2 * idx + 1), r);
        st_elem(view.out[ft], idx, v);
      } else {
        v = ld_elem_cv(view.in[ft], idx);
      }
      s_tile[item] = v;
    }
    __syncthreads();
    SC_TRACE(8);
    if (xi < ns) {
      for (int pr = ri; pr < np; pr += rw) {
        constexpr int KC = KP > 0 ? KP : 8;
        Fr cur[KC];
#pragma unroll
        for (int t = 0; t < KC; t++) {
          if (t < k) {
            const Fr lo = s_tile[t * 2 * np + 2 * pr], hi = s_tile[t * 2 * np + 2 * pr + 1];
            if (x == 0) {
              cur[t] = lo;
            } else {
              const Fr df = fp_sub<FrParams>(hi, lo);
              Fr v = hi;
              for (int i = 1; i < x; i++) v = fp_add<FrParams>(v, df);
              cur[t] = v;
            }
          }
        }
        Fr val;
        if (KP > 0) {
          val = cur[0];
#pragma unroll
          for (int t = 1; t < KC; t++) val = fp_mul<FrParams>(val, cur[t]);
        } else {
          val = sc_eval_program(s_ops, n_ops, consts, cur);
        }
        acc = fp_add<FrParams>(acc, val);
      }
    }
    __syncthreads();
    SC_TRACE(9);
  }
  acc = warp_sum(acc);
  if (lane == 0) s_rows[warp] = acc;
  __syncthreads();
  if (tid < ns) {
    Fr sum = s_rows[tid * wpr];
    for (int w = 1; w < wpr; w++) sum = fp_add<FrParams>(sum, s_rows[tid * wpr + w]);
    dst[tid] = sum;
  }
  __syncthreads();
}

// the closing block's sum of the nblk parked vectors.  ns <= 8: a row of 32 * (8 / ns) threads per evaluation point, one
// shuffle sum per thread (block_sum_many runs ns of them back to back).  dst[x] written by thread x.  Ends with a barrier.
QZ_DEV void mid_sum_parked(const Fr* partials, unsigned int nblk, int ns, Fr* s_part, Fr* dst) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (ns <= 8) {
    const int wpr = 8 / ns, rw = 32 * wpr;  // warps / threads per row
    const int x = tid / rw, i = tid % rw;
    Fr v = fp_zero<FrParams>();
    if (x < ns)
      for (unsigned int b = (unsigned int)i; b < nblk; b += (unsigned int)rw)
        v = fp_add<FrParams>(v, ld_elem_cv(reinterpret_cast<const uint4*>(partials), (uint64_t)b * ns + x));
    v = warp_sum(v);
    if (lane == 0) s_part[warp] = v;
    __syncthreads();
    if (tid < ns) {
      Fr s = s_part[tid * wpr];
      for (int w = 1; w < wpr; w++) s = fp_add<FrParams>(s, s_part[tid * wpr + w]);
      dst[tid] = s;
    }
    __syncthreads();
  } else {
    Fr acc[SC_MAX_COEFFS];
    for (int x = 0; x < ns; x++)
      acc[x] = (unsigned int)tid < nblk ? ld_elem_cv(reinterpret_cast<const uint4*>(partials), (uint64_t)tid * ns + x)
                                        : fp_zero<FrParams>();
    block_sum_many(acc, ns, s_part, dst);
  }
}

// blocks other than the closing one wait here until `target` rounds are closed
QZ_DEV void mid_wait_closed(ScMidSync* sync, unsigned int target, ScHead* head) {
  if (threadIdx.x == 0 && ld_acquire_gpu(&sync->flag) < target) {
    // the closing block may itself be waiting for a peer GPU (20 s at most, comm.cuh); give up a little later than that
    // rather than hang the device: the proof is void (peer_fault) and every block runs on to the end on stale data.
    // The clock is read once per 256 polls: reading it costs more than the poll.
    const unsigned long long t0 = global_timer_ns();
    for (unsigned int polls = 1; ld_acquire_gpu(&sync->flag) < target; polls++)
      if ((polls & 255u) == 0 && global_timer_ns() - t0 > PEER_WAIT_NS + PEER_WAIT_NS / 2) {
        head->peer_fault = 2;
        break;
      }
  }
  __syncthreads();
}

// KP > 0: h is a product of KP distinct tables (same fast path as sc_round_prod); KP == 0: interpret the program
template <int KP>
__global__ void __launch_bounds__(SC_THREADS) sc_mid(ScTables tabs, ScTailBufs bufs, uint64_t size, int pending_fold,
                                                    ScHead* head, const ScProgram* prog, const Fr* consts, const Fr* vinv,
                                                    Fr* out_coeffs, uint32_t* out_lens, Fr* out_point, int round,
                                                    int max_coeffs, Fr* partials, ScMidSync* sync,
                                                    PeerMailbox* const* peers, int rank, int G, uint32_t seq,
                                                    int gather_par, const Fr* zc_z, int zc_n,
                                                    const __grid_constant__ ScMidPlan plan) {
  __shared__ Fr s_part[(SC_THREADS / 32) * SC_MAX_COEFFS];
  __shared__ Fr s_evals[SC_MAX_COEFFS];
  __shared__ Fr s_coef[SC_MAX_COEFFS];
  __shared__ Fr s_prod[SC_PROD_SLOTS];
  __shared__ Fr s_tile[SC_TILE_ELEMS];
  __shared__ __align__(16) uint32_t s_msg[SC_MSG_WORDS];
  __shared__ uint32_t s_ops[SC_MAX_OPS];
  __shared__ int s_last;
  grid_dep_wait();
  const uint32_t n_ops = prog->n_ops;
  const int d = (int)prog->degree, k = (int)prog->k;
  for (uint32_t i = threadIdx.x; i < n_ops; i += blockDim.x) s_ops[i] = prog->ops[i];
  __syncthreads();
  ScTables view;
  for (int t = 0; t < k; t++) view.in[t] = tabs.in[t];
  int flip = 0;
  bool gathered = G == 1;
  unsigned int arrive_target = 0, rounds_closed = 0;
  int pj = 0;  // round of this launch (index into the plan)
  // `size` elements per table with (pending_fold) the last challenge still to be folded in.  Each round is ONE pass:
  // fold (reads 4, writes 2) fused with the evaluation of the new pairs, exactly like the streaming kernel.
  for (;;) {
    // blocks no later round will use leave (the count is not monotone: a split round spreads thinner than the
    // whole-pair round before it, and the rounds after a gather have more pairs than the ones just before it)
    if (blockIdx.x >= plan.future[pj]) return;
    if (!gathered && size * (uint64_t)G <= ((uint64_t)1 << SC_TAIL_LOG)) {
      // hand-over of a sharded proof: block 0 stores this rank's shard into every rank's gather area (rank order =
      // index order) and exchanges flags with the peers; the step is closed like a round for the other blocks
      PeerMailbox* mine = peers[rank];
      const int par = gather_par;
      if (blockIdx.x == 0) {
        for (int t = 0; t < k; t++)
          for (uint64_t i = threadIdx.x; i < size; i += blockDim.x) {
            const Fr v = ld_elem_cv(view.in[t], i);
            for (int g = 0; g < G; g++) fp_store<FrParams>(&peers[g]->gather[par][t][(uint64_t)rank * size + i], v);
          }
        __syncthreads();
        if (threadIdx.x == 0) s_evals[0] = fp_zero<FrParams>();
        __syncthreads();
        peer_exchange(peers, rank, G, seq, s_evals, 1);  // fence + flags: every rank's stores above are visible after it
        if (threadIdx.x == 0) {
          if (*reinterpret_cast<volatile uint32_t*>(&mine->timed_out)) head->peer_fault = 1;
          __threadfence();
          st_release_gpu(&sync->flag, rounds_closed + 1);
        }
        __syncthreads();
      } else {
        mid_wait_closed(sync, rounds_closed + 1, head);
      }
      rounds_closed++;
      seq++;
      for (int t = 0; t < k; t++) view.in[t] = reinterpret_cast<const uint4*>(&mine->gather[par][t][0]);
      size *= (uint64_t)G;
      gathered = true;
    }
    if (size <= 1 || (pending_fold && size == 2)) break;
    const uint64_t n_pairs = pending_fold ? size / 4 : size / 2;
    const uint64_t chunk = plan.chunk[pj];
    const bool split = chunk != 0;
    const unsigned int nblk = plan.nblk[pj];
    const bool skip1 = pending_fold && d >= 1;  // X = 1 from the running claim (ProdAcc)
    const int ns = skip1 ? d : d + 1;
    bool closer = false;
    SC_TRACE(1);
    if (blockIdx.x < nblk) {
      for (int t = 0; t < k; t++) view.out[t] = flip ? bufs.b[t] : bufs.a[t];
      Fr r = fp_zero<FrParams>();
      if (pending_fold) r = ld_elem_cv(reinterpret_cast<const uint4*>(&head->r), 0);
      Fr* dst = nblk > 1 ? &partials[(size_t)blockIdx.x * ns] : s_evals;
      if (split) {
        const uint64_t p0 = (uint64_t)blockIdx.x * chunk, p1 = p0 + chunk < n_pairs ? p0 + chunk : n_pairs;
        mid_split_pass<KP>(view, p0, p1, pending_fold != 0, skip1, r, s_ops, n_ops, k, ns, consts, (int)plan.tile, s_tile, s_part,
                           dst);
      } else {
        Fr acc[SC_MAX_COEFFS];
        const uint64_t first = (uint64_t)blockIdx.x * SC_THREADS + threadIdx.x, step = (uint64_t)nblk * SC_THREADS;
        if (skip1) mid_block_pass<KP, true>(view, first, step, n_pairs, true, r, s_ops, n_ops, k, d, consts, acc);
        else mid_block_pass<KP, false>(view, first, step, n_pairs, pending_fold != 0, r, s_ops, n_ops, k, d, consts, acc);
        block_sum_many(acc, ns, s_part, dst);
      }
      SC_TRACE(2);
      closer = true;
      if (nblk > 1) {  // this block's vector is parked; the last block to arrive closes the round
        arrive_target += nblk;
        if (threadIdx.x == 0) {
          __threadfence();
          s_last = atomicAdd(&sync->arrive, 1u) + 1u == arrive_target;
        }
        __syncthreads();
        closer = s_last != 0;
        if (closer) {
          __threadfence();
          mid_sum_parked(partials, nblk, ns, s_part, s_evals);
        }
      }
    } else if (nblk > 1) {
      arrive_target += nblk;  // idle this round, needed by a later one
    }
    SC_TRACE(3);
    if (closer) {
      if (!gathered) peer_sum(peers, rank, G, seq, head, s_evals, ns);
      SC_TRACE(4);
      if (skip1) sc_expand_evals(head, d, s_evals, nullptr, nullptr);
      // The other blocks are released as soon as the challenge is out, provided this block works on the next round too:
      // its arrival there orders the claim it is still computing before the next closing block reads it.
      const bool multi = gridDim.x > 1;
      const bool early = multi && pj + 1 < SC_MAX_VARS && blockIdx.x < plan.nblk[pj + 1];
      sc_round_close(head, vinv, d, s_evals, s_coef, s_msg, s_prod, out_coeffs + (size_t)round * max_coeffs,
                     out_lens + round, out_point + round, max_coeffs, nullptr, true, nullptr,
                     early ? &sync->flag : nullptr, rounds_closed + 1);
      SC_TRACE(6);
      if (multi && !early) {
        __syncthreads();
        if (threadIdx.x == 0) {
          __threadfence();
          st_release_gpu(&sync->flag, rounds_closed + 1);
        }
      }
    }
    rounds_closed++;
    if (!gathered) seq++;
    if (!closer) mid_wait_closed(sync, rounds_closed, head);
    SC_TRACE(7);
    round++;
    pj++;
    if (pending_fold) {
      for (int t = 0; t < k; t++) view.in[t] = flip ? bufs.b[t] : bufs.a[t];
      flip ^= 1;
      size >>= 1;
    }
    pending_fold = 1;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {  // sumcheck.rs:81-100: last fold, then h(g_1(r), ..., g_k(r))
    Fr fin[SC_MAX_K];
    const Fr r = fr_ld_cv(&head->r);
    for (int t = 0; t < k; t++) {
      Fr lo = ld_elem_cv(view.in[t], 0);
      if (pending_fold && size == 2) lo = fold_by(lo, ld_elem_cv(view.in[t], 1), r);
      fin[t] = lo;
    }
    Fr ev = sc_eval_program(s_ops, n_ops, consts, fin);
    if (zc_n > 0) {  // zerocheck.rs:34-40: the claim of h = the claim of h * eq divided by eq_eval(z, point) (eq_eval.rs:33-43)
      const Fr one = fp_one<FrParams>();
      Fr e = one;
      for (int i = 0; i < zc_n; i++) {
        const Fr x = zc_z[i], ri = out_point[i];
        e = fp_mul<FrParams>(e, fp_add<FrParams>(fp_mul<FrParams>(x, ri), fp_mul<FrParams>(fp_sub<FrParams>(one, x), fp_sub<FrParams>(one, ri))));
      }
      ev = fp_mul<FrParams>(ev, fp_inv_serial<FrParams>(e));
    }
    head->evaluation = ev;
  }
}

// test hook (qz_test_fold): out[i] = a0[i] + r (a1[i] - a0[i]) through the challenge table and fp_mul_fixed
__global__ void k_fold_table(Fr r, uint32_t* foldc) {
  if (threadIdx.x < 8) fold_table_row(r, threadIdx.x, foldc);
}
__global__ void k_fold_fixed(const uint4* a0, const uint4* a1, uint4* out, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) st_elem(out, i, fold_fixed(ld_elem(a0, i), ld_elem(a1, i)));
}

// ---- small helper kernels ---------------------------------------------------------------------------------------------------------
// Opens a proof in one launch (one warp; the transcript runs on lanes 0..3, tr_*_quad): the caller's transcript state;
// for a zero-check the n challenges drawn before the header (zerocheck.rs:20-22); then num_vars (u64 LE) and
// claimed_sum are absorbed (sumcheck.rs:35-36).  zinv (optional): 1 / z_j for the SKIP1 rounds of the eq-factored
// zero-check, by one batched inversion (Montgomery's trick: 3 products per element + one binary-Euclid inverse).
// The caller's transcript state and the compiled program travel as kernel ARGUMENTS (32 B + 2 KiB of the 4 KiB parameter
// space) and are written to device memory here: a proof without constants needs no host-to-device copy at all (the
// copy's DMA round trip was ~8 us of a small proof's ~85 us of fixed cost).
struct ScStateArg {
  uint8_t b[32];
};
__global__ void __launch_bounds__(32) sc_begin(ScHead* head, const __grid_constant__ ScStateArg state_in, uint64_t num_vars,
                                               Fr claimed_sum, int zc_n, Fr* z, Fr* zinv, ScMidSync* sync, PeerMailbox* mbox,
                                               const __grid_constant__ ScProgram prog_in, ScProgram* prog_out) {
  __shared__ __align__(16) uint32_t buf[32];
  const int t = threadIdx.x;
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(&prog_in);
    uint32_t* dst = reinterpret_cast<uint32_t*>(prog_out);
    const int words = 4 + (int)prog_in.n_ops;  // header + the ops in use
    for (int i = t; i < words; i += 32) dst[i] = src[i];
  }
  if (t == 0) {
    sync->arrive = 0;
    sync->flag = 0;
    if (mbox) mbox->timed_out = 0;  // a wait that timed out in an earlier proof must not void this one
    for (int i = 0; i < 32; i++) head->tstate[i] = state_in.b[i];
    head->r = fp_zero<FrParams>();
    head->evaluation = fp_zero<FrParams>();
    head->zc_prefix = fp_one<FrParams>();
    head->zc_prefix_prev = fp_one<FrParams>();
    head->claim = fp_zero<FrParams>();
    head->peer_fault = 0;
    head->zc_degenerate = 0;
  }
  __syncwarp();
  if (t < 4) {
    uint32_t* state = reinterpret_cast<uint32_t*>(head->tstate);
    for (int i = 0; i < zc_n; i++) {
      const Fr zi = tr_draw_fr_quad(state, buf);
      if (t == 0) z[i] = zi;
    }
    for (int i = t; i < 32; i += 4) buf[i] = 0;
    __syncwarp(B3_QUAD);
    if (t == 0) {
      buf[8] = (uint32_t)num_vars;
      buf[9] = (uint32_t)(num_vars >> 32);
    }
    __syncwarp(B3_QUAD);
    tr_absorb_quad(state, buf, 8);
    if (t == 0) {
      const Fr can = fp_from_mont<FrParams>(claimed_sum);
      for (int i = 0; i < 8; i++) buf[8 + i] = can.v[i];
    }
    __syncwarp(B3_QUAD);
    tr_absorb_quad(state, buf, 32);
  }
  if (t == 0 && zinv && zc_n > 0) {
    Fr run = fp_one<FrParams>();
    for (int i = 0; i < zc_n; i++) {
      const Fr zi = z[i];
      if (fp_is_zero<FrParams>(zi)) head->zc_degenerate = 1;
      zinv[i] = run;
      run = fp_mul<FrParams>(run, zi);
    }
    Fr inv = fp_inv_serial<FrParams>(run);
    for (int i = zc_n - 1; i >= 0; i--) {
      const Fr zi = z[i];
      zinv[i] = fp_mul<FrParams>(inv, zinv[i]);
      inv = fp_mul<FrParams>(inv, zi);
    }
  }
}
// eq(x, z) tables over the low `a` variables and the remaining high variables
__global__ void eq_half_tables(const Fr* z, int n, int a, Fr* lo_tab, Fr* hi_tab) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t nlo = (uint64_t)1 << a, nhi = (uint64_t)1 << (n - a);
  if (i >= nlo + nhi) return;
  const bool is_lo = i < nlo;
  const uint64_t idx = is_lo ? i : i - nlo;
  const int first = is_lo ? 0 : a, cnt = is_lo ? a : n - a;
  Fr acc = fp_one<FrParams>();
  const Fr one = fp_one<FrParams>();
  for (int j = 0; j < cnt; j++) {
    Fr zj = z[first + j];
    Fr f = ((idx >> j) & 1) ? zj : fp_sub<FrParams>(one, zj);
    acc = fp_mul<FrParams>(acc, f);
  }
  (is_lo ? lo_tab : hi_tab)[idx] = acc;
}
// eq_eval.rs:6-31: table[i] = prod_j (bit_j(i) ? z_j : 1 - z_j) = lo_tab[i mod 2^a] * hi_tab[i >> a]
// `base` is the global index of out[0] (a rank's shard of the table starts at rank * shard_len).
__global__ void __launch_bounds__(256) eq_expand(const Fr* lo_tab, const Fr* hi_tab, int a, uint64_t base,
                                                uint64_t n_elems, uint4* out) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x, mask = ((uint64_t)1 << a) - 1;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_elems; i += stride) {
    const uint64_t g = base + i;
    st_elem(out, i, fp_mul<FrParams>(lo_tab[g & mask], hi_tab[g >> a]));
  }
}
// Inverse Vandermonde on nodes 0..d: vinv[i*(d+1)+j] = coefficient of X^i in the Lagrange basis polynomial L_j
__global__ void sc_build_vinv(int d, Fr* vinv) {
  const int j = threadIdx.x;
  if (j > d) return;
  Fr small[SC_MAX_COEFFS];  // Montgomery form of 0..d
  small[0] = fp_zero<FrParams>();
  for (int i = 1; i <= d; i++) small[i] = fp_add<FrParams>(small[i - 1], fp_one<FrParams>());
  Fr c[SC_MAX_COEFFS];  // numerator prod_{m != j} (X - m)
  c[0] = fp_one<FrParams>();
  int len = 1;
  Fr denom = fp_one<FrParams>();
  for (int m = 0; m <= d; m++) {
    if (m == j) continue;
    c[len] = fp_zero<FrParams>();
    for (int i = len; i >= 0; i--) {  // c <- c * (X - m)
      Fr lower = i > 0 ? c[i - 1] : fp_zero<FrParams>();
      c[i] = fp_sub<FrParams>(lower, fp_mul<FrParams>(small[m], c[i]));
    }
    len++;
    Fr diff = j > m ? small[j - m] : fp_neg<FrParams>(small[m - j]);
    denom = fp_mul<FrParams>(denom, diff);
  }
  Fr inv = fp_inv<FrParams>(denom);
  for (int i = 0; i <= d; i++) vinv[i * (d + 1) + j] = fp_mul<FrParams>(c[i], inv);
}


// ---- logup denominators (hyperplonk/src/piops/multiset_check.rs:43-95) -----------------------------------------------------------
// out[i] = m(row_i) / (gamma + h(row_i)).  The reference inverts every row separately (`.inverse().unwrap()`, :51,:63);
// here a thread owns LOGUP_CHAIN rows strided by the block size (coalesced), multiplies them up, inverts once
// (Montgomery's trick: 3 products per row + one Fermat inversion per chain) and walks back.  A zero denominator makes
// the reference panic; it is reported through `err`.
constexpr int LOGUP_CHAIN = 32;
__global__ void __launch_bounds__(128) logup_denominators(ScTables tabs, uint64_t n_rows, const ScProgram* prog_h,
                                                         const ScProgram* prog_m, const Fr* consts, Fr gamma,
                                                         uint4* out, uint4* scratch, int* err) {
  __shared__ uint32_t s_ops[2][SC_MAX_OPS];
  const uint32_t nh = prog_h->n_ops, nm = prog_m ? prog_m->n_ops : 0;
  const int k = (int)prog_h->k;  // both programs index the same dense table list
  for (uint32_t i = threadIdx.x; i < nh; i += blockDim.x) s_ops[0][i] = prog_h->ops[i];
  for (uint32_t i = threadIdx.x; i < nm; i += blockDim.x) s_ops[1][i] = prog_m->ops[i];
  __syncthreads();
  const uint64_t tile = (uint64_t)blockIdx.x * blockDim.x * LOGUP_CHAIN;
  Fr prod = fp_one<FrParams>();
  int cnt = 0;
  for (int j = 0; j < LOGUP_CHAIN; j++) {
    const uint64_t i = tile + (uint64_t)j * blockDim.x + threadIdx.x;
    if (i >= n_rows) break;
    Fr vals[SC_MAX_K];
    for (int t = 0; t < k; t++) vals[t] = ld_elem(tabs.in[t], i);
    const Fr v = fp_add<FrParams>(gamma, sc_eval_program(s_ops[0], nh, consts, vals));
    if (fp_is_zero<FrParams>(v)) atomicExch(err, 1);
    st_elem(scratch, i, prod);  // product of the chain's earlier denominators
    st_elem(out, i, v);
    prod = fp_mul<FrParams>(prod, v);
    cnt++;
  }
  Fr inv = fp_inv<FrParams>(prod);
  for (int j = cnt - 1; j >= 0; j--) {
    const uint64_t i = tile + (uint64_t)j * blockDim.x + threadIdx.x;
    const Fr v = ld_elem(out, i);
    Fr d = fp_mul<FrParams>(inv, ld_elem(scratch, i));  // 1 / v_j
    inv = fp_mul<FrParams>(inv, v);
    if (nm) {
      Fr vals[SC_MAX_K];
      for (int t = 0; t < k; t++) vals[t] = ld_elem(tabs.in[t], i);
      d = fp_mul<FrParams>(d, sc_eval_program(s_ops[1], nm, consts, vals));  // :85-87
    }
    st_elem(out, i, d);
  }
}

}  // namespace qz

// =====================================================================================================================
// host side
// =====================================================================================================================
using namespace qz;

namespace {

struct Compiled {
  ScProgram prog;
  std::vector<uint32_t> active;  // active[j] = original table index of dense input j
  int product_k = 0;             // > 0: h is a product of `product_k` distinct inputs (fast path)
};

// VirtualPolyExpr -> postfix program over densely renumbered inputs; degree: Input 1, Const 0, Add max, Mul sum
int compile_expr(qz_ctx* ctx, const qz_expr_node* nodes, size_t n_nodes, size_t k, size_t n_consts, Compiled& out) {
  if (n_nodes == 0) return ctx->fail(QZ_ERR_EXPR, "empty expression");
  std::vector<int> remap(k, -1);
  std::vector<uint32_t> ops;
  bool ok = true;
  bool pure_product = true;
  std::vector<uint32_t> prod_inputs;
  struct Rec {
    const qz_expr_node* nodes;
    size_t n_nodes, k, n_consts;
    std::vector<int>& remap;
    std::vector<uint32_t>& active;
    std::vector<uint32_t>& ops;
    bool& ok;
    bool& pure_product;
    std::vector<uint32_t>& prod_inputs;
    int max_stack = 0;
    // returns degree; depth = current stack height before evaluating this node
    int go(size_t idx, int depth, int guard) {
      if (!ok || idx >= n_nodes || guard > 4096 || ops.size() > (size_t)SC_MAX_OPS) {
        ok = false;
        return 0;
      }
      const qz_expr_node& e = nodes[idx];
      if (depth + 1 > max_stack) max_stack = depth + 1;
      switch (e.op) {
        case QZ_EX_INPUT: {
          if (e.a >= k) {
            ok = false;
            return 0;
          }
          if (remap[e.a] < 0) {
            remap[e.a] = (int)active.size();
            active.push_back(e.a);
          }
          ops.push_back((SC_OP_IN << 16) | (uint32_t)remap[e.a]);
          prod_inputs.push_back(e.a);
          return 1;
        }
        case QZ_EX_CONST: {
          if (e.a >= n_consts || e.a > 0xffff) {
            ok = false;
            return 0;
          }
          ops.push_back((SC_OP_CONST << 16) | e.a);
          pure_product = false;
          return 0;
        }
        case QZ_EX_ADD:
        case QZ_EX_MUL: {
          if (e.a >= idx || e.b >= idx) {  // children must precede parents
            ok = false;
            return 0;
          }
          int da = go(e.a, depth, guard + 1), db = go(e.b, depth + 1, guard + 1);
          ops.push_back(((e.op == QZ_EX_ADD ? SC_OP_ADD : SC_OP_MUL) << 16));
          if (e.op == QZ_EX_ADD) pure_product = false;
          return e.op == QZ_EX_ADD ? std::max(da, db) : da + db;
        }
        default: ok = false; return 0;
      }
    }
  } rec{nodes, n_nodes, k, n_consts, remap, out.active, ops, ok, pure_product, prod_inputs};
  int deg = rec.go(n_nodes - 1, 0, 0);
  if (!ok) return ctx->fail(QZ_ERR_EXPR, "malformed expression tree");
  if (ops.size() > (size_t)SC_MAX_OPS) return ctx->fail(QZ_ERR_EXPR, "expression too large (ops)");
  if (rec.max_stack > SC_MAX_STACK) return ctx->fail(QZ_ERR_EXPR, "expression too deep (stack)");
  if (out.active.size() > (size_t)SC_MAX_K) return ctx->fail(QZ_ERR_EXPR, "too many tables referenced by h");
  if (deg > SC_MAX_DEG) return ctx->fail(QZ_ERR_EXPR, "expression degree too high");
  memset(&out.prog, 0, sizeof out.prog);
  out.prog.n_ops = (uint32_t)ops.size();
  out.prog.degree = (uint32_t)deg;
  out.prog.k = (uint32_t)out.active.size();
  out.prog.n_consts = (uint32_t)n_consts;
  memcpy(out.prog.ops, ops.data(), ops.size() * 4);
  out.product_k = 0;
  if (pure_product && prod_inputs.size() == out.active.size() && prod_inputs.size() >= 1 && prod_inputs.size() <= 4)
    out.product_k = (int)prod_inputs.size();  // distinct inputs, each used once
  return QZ_OK;
}

int get_vinv(qz_ctx* ctx, int d, Fr** out) {
  auto it = ctx->cache.find(d);
  if (it != ctx->cache.end()) {
    *out = (Fr*)it->second;
    return QZ_OK;
  }
  void* p = nullptr;
  QZ_CUDA(ctx, cudaMalloc(&p, sizeof(Fr) * (d + 1) * (d + 1)));
  QZ_LAUNCH(ctx, sc_build_vinv, 1, 64, 0, d, (Fr*)p);
  ctx->cache[d] = p;
  *out = (Fr*)p;
  return QZ_OK;
}

// resident blocks per SM of a kernel, asked of the runtime once per context (the query costs microseconds and a proof
// asked three or four of them: a tenth of a small proof's fixed cost)
template <class Kernel>
int blocks_per_sm(qz_ctx* ctx, Kernel kern, int threads) {
  const std::pair<const void*, int> key((const void*)kern, threads);
  auto it = ctx->occupancy.find(key);
  if (it != ctx->occupancy.end()) return it->second;
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, 0) != cudaSuccess) {
    cudaGetLastError();
    occ = 0;
  }
  ctx->occupancy[key] = occ;
  return occ;
}

int round_grid(qz_ctx* ctx, uint64_t n_pairs, int blocks_per_sm, int threads = SC_THREADS) {
  uint64_t want = (n_pairs + threads - 1) / threads;
  uint64_t cap = (uint64_t)ctx->sm_count * blocks_per_sm;
  return (int)std::max<uint64_t>(1, std::min(want, cap));
}

// resident blocks per SM of a proof's streaming-round kernels: the narrow one (at least 1) and the deferred-reduction one
// (0: there is none).  zc: the zero-check fast path's kernels of nf factors; otherwise the product kernels of nf
// factors, or the interpreter for nf = 0.  The folding instance stands for its family.
struct RoundOcc {
  int narrow, wide;
};
RoundOcc round_occupancy(qz_ctx* ctx, bool zc, int nf) {
  RoundOcc o = {1, 0};
  if (zc) {
    if (nf == 1) o.narrow = blocks_per_sm(ctx, sc_round_zc<1, false, true, false>, SC_THREADS);
    else if (nf == 2) o.narrow = blocks_per_sm(ctx, sc_round_zc<2, false, true, false>, SC_THREADS);
    else {
      o.narrow = blocks_per_sm(ctx, sc_round_zc<3, false, true, false>, SC_THREADS);
      o.wide = blocks_per_sm(ctx, sc_round_zc<3, true, true, false>, SC_WIDE_THREADS);
    }
  } else if (nf == 1) {
    o.narrow = blocks_per_sm(ctx, sc_round_prod<1, false, true>, SC_THREADS);
  } else if (nf == 2) {
    o.narrow = blocks_per_sm(ctx, sc_round_prod<2, false, true>, SC_THREADS);
  } else if (nf == 3) {
    o.narrow = blocks_per_sm(ctx, sc_round_prod<3, false, true>, SC_THREADS);
    o.wide = blocks_per_sm(ctx, sc_round_prod<3, true, true>, SC_WIDE_THREADS);
  } else if (nf == 4) {
    o.narrow = blocks_per_sm(ctx, sc_round_prod<4, false, true>, SC_THREADS);
    o.wide = blocks_per_sm(ctx, sc_round_prod<4, true, true>, SC_WIDE_THREADS);
  } else {
    o.narrow = blocks_per_sm(ctx, sc_round_generic<true>, SC_THREADS);
  }
  o.narrow = std::max(o.narrow, 1);
  return o;
}
// a streaming round's kernel variant and grid
struct RoundShape {
  bool wide;
  int grid;
};

}  // namespace

namespace qz {

// c_fold is one table per device: proofs of different contexts on the same device take turns
static std::recursive_mutex g_fold_table_lock[16];

// elements [base, base + n_elems) of eq(., z) over n variables
int eq_table_device(qz_ctx* ctx, int n, const Fr* z_dev, uint4* out_dev, uint64_t base, uint64_t n_elems) {
  const int a = n / 2;
  Fr* lo_tab = (Fr*)ctx->arena_alloc(sizeof(Fr) << a);
  Fr* hi_tab = (Fr*)ctx->arena_alloc(sizeof(Fr) << (n - a));
  if (!lo_tab || !hi_tab) return ctx->fail(QZ_ERR_ALLOC, "eq table scratch");
  const uint64_t small = ((uint64_t)1 << a) + ((uint64_t)1 << (n - a));
  QZ_LAUNCH(ctx, eq_half_tables, (unsigned)((small + 127) / 128), 128, 0, z_dev, n, a, lo_tab, hi_tab);
  int grid = (int)std::max<uint64_t>(1, std::min<uint64_t>((n_elems + 255) / 256, (uint64_t)ctx->sm_count * 8));
  QZ_LAUNCH(ctx, eq_expand, grid, 256, 0, lo_tab, hi_tab, a, base, n_elems, out_dev);
  return QZ_OK;
}

// multiset_check.rs:43-95: out[i] = m(row_i) / (gamma + h(row_i)); m omitted (n_nodes_m == 0) means 1
int logup_denominators_run(qz_ctx* ctx, size_t num_vars, size_t k, const void* const* tables, int tables_on_device,
                           const qz_expr_node* nodes_h, size_t n_nodes_h, const qz_expr_node* nodes_m, size_t n_nodes_m,
                           const uint8_t* consts, size_t n_consts, const uint8_t* gamma, void* out, int out_on_device) {
  if (!ctx || !gamma || !out || (k && !tables) || !nodes_h || n_nodes_h == 0 || (n_consts && !consts) ||
      num_vars >= (size_t)SC_MAX_VARS)
    return ctx ? ctx->fail(QZ_ERR_INVALID_ARG, "bad arguments") : QZ_ERR_INVALID_ARG;
  QZ_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->arena_reset();
  cudaStream_t st = ctx->stream;
  const uint64_t N = (uint64_t)1 << num_vars;
  // both expressions are compiled against ONE dense table list: compile m after h, sharing the remap, by joining them
  // under a throw-away Add root and splitting the program at the boundary
  Compiled ch, cm;
  int rc;
  std::vector<qz_expr_node> joined(nodes_h, nodes_h + n_nodes_h);
  if (n_nodes_m) {
    const uint32_t off = (uint32_t)n_nodes_h;
    for (size_t i = 0; i < n_nodes_m; i++) {
      qz_expr_node e = nodes_m[i];
      if (e.op == QZ_EX_ADD || e.op == QZ_EX_MUL) {
        e.a += off;
        e.b += off;
      }
      joined.push_back(e);
    }
    joined.push_back(qz_expr_node{QZ_EX_ADD, off - 1, (uint32_t)joined.size() - 1});
  }
  Compiled cj;
  rc = compile_expr(ctx, joined.data(), joined.size(), k, n_consts, cj);
  if (rc) return rc;
  // recompile each part on its own, then rewrite its Input indices into the joint numbering
  auto remap_to_joint = [&](Compiled& c) {
    for (uint32_t i = 0; i < c.prog.n_ops; i++) {
      uint32_t op = c.prog.ops[i];
      if ((op >> 16) == SC_OP_IN) {
        uint32_t orig = c.active[op & 0xffffu], dense = 0;
        for (uint32_t j = 0; j < cj.active.size(); j++)
          if (cj.active[j] == orig) dense = j;
        c.prog.ops[i] = (SC_OP_IN << 16) | dense;
      }
    }
    c.prog.k = cj.prog.k;
  };
  rc = compile_expr(ctx, nodes_h, n_nodes_h, k, n_consts, ch);
  if (rc) return rc;
  remap_to_joint(ch);
  if (n_nodes_m) {
    rc = compile_expr(ctx, nodes_m, n_nodes_m, k, n_consts, cm);
    if (rc) return rc;
    remap_to_joint(cm);
  }
  const int ka = (int)cj.prog.k;
  ScTables tabs;
  memset(&tabs, 0, sizeof tabs);
  for (int j = 0; j < ka; j++) {
    const uint32_t orig = cj.active[j];
    if (!tables[orig]) return ctx->fail(QZ_ERR_INVALID_ARG, "null table");
    if (tables_on_device) {
      tabs.in[j] = (const uint4*)tables[orig];
    } else {
      void* p = ctx->arena_alloc(32 * N);
      if (!p) return ctx->fail(QZ_ERR_ALLOC, "table copy");
      QZ_CUDA(ctx, cudaMemcpyAsync(p, tables[orig], 32 * N, cudaMemcpyHostToDevice, st));
      tabs.in[j] = (const uint4*)p;
    }
  }
  ScProgram* d_ph = (ScProgram*)ctx->arena_alloc(sizeof(ScProgram));
  ScProgram* d_pm = n_nodes_m ? (ScProgram*)ctx->arena_alloc(sizeof(ScProgram)) : nullptr;
  Fr* d_consts = (Fr*)ctx->arena_alloc(32 * std::max<size_t>(1, n_consts));
  uint4* d_out = out_on_device ? (uint4*)out : (uint4*)ctx->arena_alloc(32 * N);
  uint4* d_scratch = (uint4*)ctx->arena_alloc(32 * N);
  int* d_err = (int*)ctx->arena_alloc(4);
  if (!d_ph || (n_nodes_m && !d_pm) || !d_consts || !d_out || !d_scratch || !d_err)
    return ctx->fail(QZ_ERR_ALLOC, "logup scratch");
  QZ_CUDA(ctx, cudaMemcpyAsync(d_ph, &ch.prog, sizeof(ScProgram), cudaMemcpyHostToDevice, st));
  if (n_nodes_m) QZ_CUDA(ctx, cudaMemcpyAsync(d_pm, &cm.prog, sizeof(ScProgram), cudaMemcpyHostToDevice, st));
  if (n_consts) QZ_CUDA(ctx, cudaMemcpyAsync(d_consts, consts, 32 * n_consts, cudaMemcpyHostToDevice, st));
  QZ_CUDA(ctx, cudaMemsetAsync(d_err, 0, 4, st));
  Fr g;
  memcpy(g.v, gamma, 32);
  const uint64_t per_block = (uint64_t)128 * LOGUP_CHAIN;
  QZ_LAUNCH(ctx, logup_denominators, (unsigned)((N + per_block - 1) / per_block), 128, 0, tabs, N, d_ph, d_pm, d_consts, g,
            d_out, d_scratch, d_err);
  int err = 0;
  QZ_CUDA(ctx, cudaMemcpyAsync(&err, d_err, 4, cudaMemcpyDeviceToHost, st));
  if (!out_on_device) QZ_CUDA(ctx, cudaMemcpyAsync(out, d_out, 32 * N, cudaMemcpyDeviceToHost, st));
  QZ_CUDA(ctx, cudaStreamSynchronize(st));
  if (err) return ctx->fail(QZ_ERR_INVALID_ARG, "logup denominator is zero (the reference panics on inverse().unwrap())");
  return QZ_OK;
}

// The whole proof.  `sharded`: `tables` hold this rank's contiguous shard, elements [rank * 2^num_vars / nranks, ...),
// i.e. the tables are split by the top variables so every (2p, 2p+1) pair is local (sumcheck.rs:56-57).
// allow_zc_skip1 false: a zero-check runs without the SKIP1 rounds (the redo after some z_j = 0).
static int sumcheck_prove(qz_ctx* ctx, size_t num_vars, size_t k, const void* const* tables, int tables_on_device,
                          const qz_expr_node* nodes, size_t n_nodes, const uint8_t* consts, size_t n_consts,
                          const uint8_t* claimed_sum, uint8_t* state, size_t max_coeffs, uint8_t* out_coeffs,
                          uint32_t* out_lens, uint8_t* out_point, uint8_t* out_eval, bool zerocheck, uint8_t* out_z,
                          bool sharded, bool allow_zc_skip1) {
  if (!ctx || !state || !out_eval || (num_vars && (!out_coeffs || !out_lens || !out_point)))
    return ctx ? ctx->fail(QZ_ERR_INVALID_ARG, "null pointer") : QZ_ERR_INVALID_ARG;
  if (num_vars > (size_t)SC_MAX_VARS - 1 || (k && !tables) || (n_nodes && !nodes) || (n_consts && !consts))
    return ctx->fail(QZ_ERR_INVALID_ARG, "bad sizes");
  if (!zerocheck && !claimed_sum) return ctx->fail(QZ_ERR_INVALID_ARG, "claimed_sum is null");
  if (zerocheck && num_vars && !out_z) return ctx->fail(QZ_ERR_INVALID_ARG, "out_z is null");
  QZ_CUDA(ctx, cudaSetDevice(ctx->device));
  std::lock_guard<std::recursive_mutex> fold_table_guard(g_fold_table_lock[ctx->device & 15]);
  QzRange nvtx_call(zerocheck ? "qz:zerocheck_prove" : "qz:sumcheck_prove");
  ctx->arena_reset();

  // h, or h_hat = Mul(h, Input(eq)) with eq appended as the last store polynomial (zerocheck.rs:27-29)
  std::vector<qz_expr_node> nd(nodes, nodes + n_nodes);
  size_t k_total = k;
  if (zerocheck) {
    if (n_nodes == 0) return ctx->fail(QZ_ERR_EXPR, "empty expression");
    uint32_t root = (uint32_t)n_nodes - 1;
    nd.push_back(qz_expr_node{QZ_EX_INPUT, (uint32_t)k, 0});
    nd.push_back(qz_expr_node{QZ_EX_MUL, root, root + 1});
    k_total = k + 1;
  }
  Compiled cp;
  int rc = compile_expr(ctx, nd.data(), nd.size(), k_total, n_consts, cp);
  if (rc) return rc;
  const int d = (int)cp.prog.degree, ka = (int)cp.prog.k;
  if ((size_t)d + 1 > max_coeffs) return ctx->fail(QZ_ERR_EXPR, "deg(h)+1 exceeds max_coeffs");
  const int mc = (int)max_coeffs;
  const int G = sharded ? ctx->nranks : 1;
  if (((uint64_t)1 << num_vars) < (uint64_t)G) return ctx->fail(QZ_ERR_INVALID_ARG, "fewer table entries than ranks");
  const uint64_t N = ((uint64_t)1 << num_vars) / G;  // entries per table held by this rank

  cudaStream_t st = ctx->stream;
  QZ_CUDA(ctx, cudaEventRecord(ctx->ev_call0, st));

  // Device-resident proof state.  The small inputs (transcript state, program, constants) travel in ONE copy from the
  // pinned staging buffer and the outputs (head, coefficients, lengths, point, z) come back in ONE copy: every extra
  // cudaMemcpyAsync is ~5-10 us on a call whose fixed cost is otherwise ~100 us.
  auto up32 = [](size_t v) { return (v + 31) & ~(size_t)31; };
  const size_t in_prog = 32, in_consts = in_prog + up32(sizeof(ScProgram)), in_bytes = in_consts + 32 * n_consts;
  const size_t coeff_bytes = 32 * num_vars * max_coeffs, lens_bytes = 4 * num_vars, pt_bytes = 32 * num_vars;
  const size_t o_head = 0, o_coeffs = up32(sizeof(ScHead)), o_lens = o_coeffs + coeff_bytes, o_point = o_lens + up32(lens_bytes),
               o_z = o_point + pt_bytes, out_bytes = o_z + pt_bytes;
  uint8_t* d_in = (uint8_t*)ctx->arena_alloc(in_bytes);
  uint8_t* d_out = (uint8_t*)ctx->arena_alloc(out_bytes);
  uint8_t* pin = (uint8_t*)ctx->pinned_buf(up32(in_bytes) + out_bytes);
  if (!d_in || !d_out || !pin) return ctx->fail(QZ_ERR_ALLOC, "sumcheck state");
  uint8_t* pin_out = pin + up32(in_bytes);
  ScHead* head = (ScHead*)(d_out + o_head);
  Fr* d_coeffs = (Fr*)(d_out + o_coeffs);
  uint32_t* d_lens = (uint32_t*)(d_out + o_lens);
  Fr* d_point = (Fr*)(d_out + o_point);
  Fr* d_z = (Fr*)(d_out + o_z);
  ScProgram* d_prog = (ScProgram*)(d_in + in_prog);
  Fr* d_consts = (Fr*)(d_in + in_consts);
  if (n_consts) {  // the constants are the only small input that still needs a copy
    memcpy(pin + in_consts, consts, 32 * n_consts);
    QZ_CUDA(ctx, cudaMemcpyAsync(d_in + in_consts, pin + in_consts, 32 * n_consts, cudaMemcpyHostToDevice, st));
  }

  // streaming rounds run while a rank's table has more than 2^SC_MID_LOG entries (with peer mailboxes or one GPU; the
  // NCCL fallback streams down to the gather size), then sc_mid takes every remaining round
  const bool mid_sharded = G == 1 || comm_has_peers(ctx);
  static const int mid_log = [] {  // QZ_SC_MID_LOG: measurement switch for the hand-over size (DESIGN.md section 10)
    const char* e = getenv("QZ_SC_MID_LOG");
    const int v = e ? atoi(e) : SC_MID_LOG;
    return v >= SC_TAIL_LOG && v <= 24 ? v : SC_MID_LOG;
  }();
  auto streaming = [&](uint64_t sz) {
    return mid_sharded ? sz > ((uint64_t)1 << mid_log) : sz * G > ((uint64_t)1 << SC_TAIL_LOG);
  };
  // zero-check fast path (see sc_round_zc): h is a product of up to three tables and at least one streaming round runs.
  // From 2^21 entries on it skips X = 1 from round 1 on, which repays the batched inversion of the z in sc_begin
  // (~30 us on one thread).
  const bool zc_fast =
      zerocheck && cp.product_k >= 2 && cp.product_k <= 4 && streaming(N) && !getenv("QZ_ZC_STREAM_EQ");
  const bool zc_skip1 = zc_fast && num_vars >= 21 && allow_zc_skip1 && !getenv("QZ_ZC_NO_SKIP1");
  Fr* d_zinv = nullptr;
  if (zc_skip1) {
    d_zinv = (Fr*)ctx->arena_alloc(32 * num_vars);
    if (!d_zinv) return ctx->fail(QZ_ERR_ALLOC, "zero-check inverses");
  }
  ScMidSync* d_sync = (ScMidSync*)ctx->arena_alloc(sizeof(ScMidSync));
  uint32_t* d_foldc = (uint32_t*)ctx->arena_alloc(64 * sizeof(uint32_t));  // multiples of the last challenge (sc_round_close)
  if (!d_sync || !d_foldc) return ctx->fail(QZ_ERR_ALLOC, "round counters");
  {
    Fr cs;
    memset(&cs, 0, sizeof cs);
    if (!zerocheck) memcpy(cs.v, claimed_sum, 32);
    ScStateArg state_arg;
    memcpy(state_arg.b, state, 32);
    QZ_LAUNCH(ctx, sc_begin, 1, 32, 0, head, state_arg, (uint64_t)num_vars, cs, zerocheck ? (int)num_vars : 0, d_z, d_zinv,
              d_sync, (PeerMailbox*)(sharded && comm_has_peers(ctx) ? ctx->mbox : nullptr), cp.prog,
              d_prog);  // zerocheck.rs:20-22, sumcheck.rs:35-36
  }

  // Host tables of a large proof are copied in UP_CHUNKS slices on the second stream and round 0 (evaluate only: every
  // pair is independent) runs slice by slice behind the copies, so only the last slice's round-0 work is exposed after
  // the PCIe transfer; from round 1 on the challenge depends on all of the data.
  constexpr int UP_CHUNKS = 8;
  static_assert(UP_CHUNKS <= qz_ctx::MAX_SEGMENTS, "one ready-event per slice");
  const int up_chunks = (!tables_on_device && G == 1 && !zerocheck && N >= ((uint64_t)1 << 21)) ? UP_CHUNKS : 1;
  uint8_t* up_dst[SC_MAX_K];
  const uint8_t* up_src[SC_MAX_K];
  int n_up = 0;
  // tables referenced by h: device copies (host input) or the caller's device buffers.  A zero-check always has the eq
  // slot: h_hat's root multiplies by it.
  ScTables tabs;
  memset(&tabs, 0, sizeof tabs);
  int eq_slot = -1;
  for (int j = 0; j < ka; j++) {
    uint32_t orig = cp.active[j];
    if (zerocheck && orig == k) {
      eq_slot = j;
      continue;
    }
    if (!tables[orig]) return ctx->fail(QZ_ERR_INVALID_ARG, "null table");
    if (tables_on_device) {
      tabs.in[j] = (const uint4*)tables[orig];
    } else {
      void* p = ctx->arena_alloc(32 * N);
      if (!p) return ctx->fail(QZ_ERR_ALLOC, "table copy");
      if (up_chunks > 1) {  // copied chunk by chunk under round 0 (below)
        up_dst[n_up] = (uint8_t*)p;
        up_src[n_up++] = (const uint8_t*)tables[orig];
      } else {
        QZ_CUDA(ctx, cudaMemcpyAsync(p, tables[orig], 32 * N, cudaMemcpyHostToDevice, st));
      }
      tabs.in[j] = (const uint4*)p;
    }
  }
  if (zerocheck && !zc_fast) {
    void* p = ctx->arena_alloc(32 * N);
    if (!p) return ctx->fail(QZ_ERR_ALLOC, "eq table");
    rc = eq_table_device(ctx, (int)num_vars, d_z, (uint4*)p, (uint64_t)ctx->rank * N * (G > 1), N);  // zerocheck.rs:25
    if (rc) return rc;
    tabs.in[eq_slot] = (const uint4*)p;
  }

  if (num_vars > 0) {
    Fr* vinv = nullptr;
    rc = get_vinv(ctx, d, &vinv);
    if (rc) return rc;
    // ping-pong scratch: A holds N/2 elements per table, B holds N/4
    uint4 *bufA[SC_MAX_K], *bufB[SC_MAX_K];
    for (int j = 0; j < ka; j++) {
      bufA[j] = (uint4*)ctx->arena_alloc(32 * std::max<uint64_t>(1, N / 2));
      bufB[j] = (uint4*)ctx->arena_alloc(32 * std::max<uint64_t>(1, N / 4));
      if (!bufA[j] || !bufB[j]) return ctx->fail(QZ_ERR_ALLOC, "fold scratch");
    }
    // The streaming rounds fold the nt tables ft.in[i] = tabs.in[slot_of[i]]: every table of h, or on the zero-check
    // fast path the K tables of h without the eq slot, whose fold scratch holds the weight tables instead.  nf: factors
    // of the round kernel's product (0: the interpreter); deg, vinv_r: degree and interpolation matrix of the sums.
    const int nf = zc_fast ? cp.product_k - 1 : cp.product_k, deg = zc_fast ? nf : d;
    Fr* vinv_r = vinv;
    if (zc_fast) {
      rc = get_vinv(ctx, deg, &vinv_r);
      if (rc) return rc;
    }
    ScTables ft;
    memset(&ft, 0, sizeof ft);
    int slot_of[SC_MAX_K], nt = 0;
    for (int j = 0; j < ka; j++)
      if (!zc_fast || j != eq_slot) {
        ft.in[nt] = tabs.in[j];
        slot_of[nt++] = j;
      }
    // occupancy-sized grids.  `partials` holds a vector per block of the product kernel of all of h's tables; the
    // zero-check fast path's kernels are capped at that many blocks per SM.
    const bool narrow_only = getenv("QZ_SC_NARROW") != nullptr;  // measurement switch: force the fully reduced sums
    RoundOcc occ = round_occupancy(ctx, false, cp.product_k);
    if (narrow_only) occ.wide = 0;
    const int part_bps = std::max(occ.narrow, occ.wide);
    if (zc_fast) {
      const RoundOcc z = round_occupancy(ctx, true, nf);
      occ = {std::min(z.narrow, part_bps), narrow_only ? 0 : std::min(z.wide, part_bps)};
    }
    // deferred reduction pays once a thread sums several pairs (its one-off reduction is 3 products per sum)
    auto pick = [&](uint64_t n_pairs) {
      RoundShape s;
      s.wide = occ.wide > 0 && n_pairs >= (uint64_t)8 * SC_WIDE_THREADS * ctx->sm_count * occ.wide;
      s.grid = s.wide ? round_grid(ctx, n_pairs, occ.wide, SC_WIDE_THREADS) : round_grid(ctx, n_pairs, occ.narrow);
      return s;
    };
    Fr* partials = (Fr*)ctx->arena_alloc(sizeof(Fr) * std::max<size_t>((size_t)ctx->sm_count * part_bps, SC_THREADS) * (d + 1) * up_chunks);
    Fr* rank_evals = (Fr*)ctx->arena_alloc(sizeof(Fr) * (d + 1));
    Fr* all_evals = (Fr*)ctx->arena_alloc(sizeof(Fr) * (size_t)(d + 1) * G);
    if (!partials || !rank_evals || !all_evals) return ctx->fail(QZ_ERR_ALLOC, "partials");

    uint64_t size = N;  // current (pre-fold) table size
    int pending = 0, round = 0, flip = 0;
    // the round chain uses programmatic dependent launches, except around NCCL collectives (not written for them)
    // Measured (tools/sc_pdl_ab.py): -5 us per round while a round is latency-bound,
    // but +10..20 us on the rounds that stream 2^21 entries or more, so only the short rounds are chained this way.
    const bool pdl_ok = ctx->pdl && (G == 1 || comm_has_peers(ctx));
    std::unique_ptr<QzRange> nvtx_stream(new QzRange("qz:sumcheck:streaming-rounds"));
    QZ_CUDA(ctx, cudaEventRecord(ctx->ev_k0, st));
    // zero-check fast path: E_j, the weight table of round j, ping-pongs between the eq slot's fold scratch; E_1 = eq
    // table of z_1 .. z_{n-1}, this rank's N/2 entries
    uint4* e_buf[2] = {nullptr, nullptr};
    int e_cur = 0;
    if (zc_fast) {
      e_buf[0] = bufA[eq_slot];
      e_buf[1] = bufB[eq_slot];
      rc = eq_table_device(ctx, (int)num_vars - 1, d_z + 1, e_buf[0], (uint64_t)ctx->rank * (N / 2) * (G > 1), N / 2);
      if (rc) return rc;
    }
    // one round kernel over `n_pairs` pairs of `tb` (fold of the pending challenge fused when `pend`)
    const uint64_t generic_cf_pairs = (uint64_t)1 << 16;
    auto launch_round = [&](const ScTables& tb, uint64_t n_pairs, int pend, const RoundShape& rs, bool pdl, Fr* parts) -> int {
      const int grid = rs.grid;
      // the deferred-reduction passes (finish_pair<FOLD, WIDE>) and the large interpreted ones (sc_round_generic<true>)
      // fold through the challenge table in constant memory: bring it up to date first
      const bool generic_cf = nf == 0 && pend && n_pairs >= generic_cf_pairs;
      if (pend && (rs.wide || generic_cf))
        QZ_CUDA(ctx, cudaMemcpyToSymbolAsync(c_fold, d_foldc, 64 * sizeof(uint32_t), 0, cudaMemcpyDeviceToDevice, st));
      if (zc_fast) {
        const uint4* e_in = e_buf[e_cur];
        uint4* e_out = e_buf[e_cur ^ 1];
        const bool skip1 = pend && zc_skip1;
#define QZ_ROUND_ZC(KK, W, T)                                                                                      \
  do {                                                                                                             \
    if (skip1) QZ_LAUNCH_PDL(ctx, pdl, (sc_round_zc<KK, W, true, true>), grid, T, tb, e_in, e_out, n_pairs, (const ScHead*)head, parts); \
    else if (pend) QZ_LAUNCH_PDL(ctx, pdl, (sc_round_zc<KK, W, true, false>), grid, T, tb, e_in, e_out, n_pairs, (const ScHead*)head, parts); \
    else QZ_LAUNCH_PDL(ctx, pdl, (sc_round_zc<KK, W, false, false>), grid, T, tb, e_in, e_out, n_pairs, (const ScHead*)head, parts);        \
  } while (0)
        switch (nf) {
          case 1: QZ_ROUND_ZC(1, false, SC_THREADS); break;
          case 2: QZ_ROUND_ZC(2, false, SC_THREADS); break;
          default:
            if (rs.wide) QZ_ROUND_ZC(3, true, SC_WIDE_THREADS);
            else QZ_ROUND_ZC(3, false, SC_THREADS);
        }
#undef QZ_ROUND_ZC
        return QZ_OK;
      }
#define QZ_ROUND_PROD(K, W, T)                                                                                  \
  do {                                                                                                          \
    if (pend) QZ_LAUNCH_PDL(ctx, pdl, (sc_round_prod<K, W, true>), grid, T, tb, n_pairs, (const ScHead*)head, parts); \
    else QZ_LAUNCH_PDL(ctx, pdl, (sc_round_prod<K, W, false>), grid, T, tb, n_pairs, (const ScHead*)head, parts);     \
  } while (0)
      switch (nf) {
        case 1: QZ_ROUND_PROD(1, false, SC_THREADS); break;
        case 2: QZ_ROUND_PROD(2, false, SC_THREADS); break;
        case 3:
          if (rs.wide) QZ_ROUND_PROD(3, true, SC_WIDE_THREADS);
          else QZ_ROUND_PROD(3, false, SC_THREADS);
          break;
        case 4:
          if (rs.wide) QZ_ROUND_PROD(4, true, SC_WIDE_THREADS);
          else QZ_ROUND_PROD(4, false, SC_THREADS);
          break;
        default:
          if (generic_cf)
            QZ_LAUNCH_PDL(ctx, pdl, sc_round_generic<true>, grid, SC_THREADS, tb, n_pairs, pend, (const ScHead*)head,
                          (const ScProgram*)d_prog, (const Fr*)d_consts, parts);
          else
            QZ_LAUNCH_PDL(ctx, pdl, sc_round_generic<false>, grid, SC_THREADS, tb, n_pairs, pend, (const ScHead*)head,
                          (const ScProgram*)d_prog, (const Fr*)d_consts, parts);
      }
#undef QZ_ROUND_PROD
      return QZ_OK;
    };
    // Close round `rnd` from the n_parts partial vectors in `parts` (transcript on the device): on one GPU, through the
    // peers' mailboxes, or (NCCL fallback) by all-gathering one vector per rank, after which every rank runs the same
    // transcript on the same sums.  Every round but the first leaves X = 1 to the running claim (ProdAcc, generic_pair).
    auto close_round = [&](const Fr* parts, int n_parts, int rnd, int pend, bool wide, bool pdl) -> int {
      const int derive1 = pend && (zc_fast ? zc_skip1 : d >= 1) ? 1 : 0, ns = derive1 ? deg : deg + 1;
      const Fr* z_j = zc_fast ? d_z + rnd : nullptr;
      const Fr* zinv_j = zc_skip1 ? d_zinv + rnd : nullptr;
      const int toom = wide && nf == 3 ? 1 : 0;  // the sums are samples at X = 0, 1, -1, inf (prod_core_toom3)
      Fr* coeffs = d_coeffs + (size_t)rnd * mc;
      if (G == 1) {
        QZ_LAUNCH_PDL(ctx, pdl, sc_finalize, 1, SC_THREADS, parts, n_parts, deg, head, (const Fr*)vinv_r, coeffs,
                      d_lens + rnd, d_point + rnd, mc, z_j, derive1, zinv_j, d_foldc, toom);
      } else if (comm_has_peers(ctx)) {
        QZ_LAUNCH_PDL(ctx, pdl, sc_finalize_peers, 1, SC_THREADS, parts, n_parts, deg,
                      (PeerMailbox* const*)ctx->peer_mbox_dev, ctx->rank, G, ++ctx->mbox_seq, head, (const Fr*)vinv_r,
                      coeffs, d_lens + rnd, d_point + rnd, mc, z_j, derive1, zinv_j, d_foldc, toom);
      } else {
        QZ_LAUNCH(ctx, sc_reduce_partials, 1, SC_THREADS, 0, parts, n_parts, ns - 1, rank_evals);
        const int rca = comm_allgather(ctx, rank_evals, all_evals, sizeof(Fr) * ns);
        if (rca) return rca;
        QZ_LAUNCH(ctx, sc_finalize, 1, SC_THREADS, 0, all_evals, G, deg, head, vinv_r, coeffs, d_lens + rnd,
                  d_point + rnd, mc, z_j, derive1, zinv_j, d_foldc, toom);
      }
      return QZ_OK;
    };
    if (up_chunks > 1) {  // round 0 behind the host -> device copies, slice by slice
      if (ctx->ensure_prep_stream()) return ctx->fail(QZ_ERR_CUDA, "prep stream");
      cudaStream_t ps = ctx->prep_stream;
      QZ_CUDA(ctx, cudaEventRecord(ctx->ev_entry, st));  // earlier users of the arena are done before the copies land
      QZ_CUDA(ctx, cudaStreamWaitEvent(ps, ctx->ev_entry, 0));
      const uint64_t per = N / up_chunks, pairs_c = per / 2;
      const RoundShape rs = pick(pairs_c);
      for (int c = 0; c < up_chunks; c++) {
        for (int u = 0; u < n_up; u++)
          QZ_CUDA(ctx, cudaMemcpyAsync(up_dst[u] + 32 * per * c, up_src[u] + 32 * per * c, 32 * per, cudaMemcpyHostToDevice, ps));
        QZ_CUDA(ctx, cudaEventRecord(ctx->ev_seg_ready[c], ps));
        QZ_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_seg_ready[c], 0));
        ScTables slice = ft;
        for (int i = 0; i < nt; i++) slice.in[i] = ft.in[i] + 2 * per * c;
        rc = launch_round(slice, pairs_c, 0, rs, false, partials + (size_t)c * rs.grid * (d + 1));
        if (rc) return rc;
      }
      rc = close_round(partials, rs.grid * up_chunks, 0, 0, rs.wide, false);
      if (rc) return rc;
      pending = 1;
      round = 1;
    }
    while (streaming(size)) {
      const uint64_t n_pairs = pending ? size / 4 : size / 2;
      const bool pdl = pdl_ok && n_pairs <= ((uint64_t)1 << 18);
      for (int i = 0; i < nt; i++) ft.out[i] = flip ? bufB[slot_of[i]] : bufA[slot_of[i]];
      const RoundShape rs = pick(n_pairs);
      rc = launch_round(ft, n_pairs, pending, rs, pdl, partials);
      if (rc) return rc;
      rc = close_round(partials, rs.grid, round, pending, rs.wide, pdl);
      if (rc) return rc;
      if (pending) {
        for (int i = 0; i < nt; i++) ft.in[i] = ft.out[i];
        flip ^= 1;
        size >>= 1;
        if (zc_fast) e_cur ^= 1;  // this round wrote E_{round+1}
      }
      pending = 1;
      round++;
    }
    for (int i = 0; i < nt; i++) tabs.in[slot_of[i]] = ft.in[i];
    if (zc_fast) {  // hand over to sc_mid: h's tables where they stand, eq materialised in the reference's form (pending fold)
      uint4* eq_full = (uint4*)ctx->arena_alloc(32 * size);
      if (!eq_full) return ctx->fail(QZ_ERR_ALLOC, "eq hand-over");
      QZ_LAUNCH(ctx, zc_materialize_eq, (unsigned)((size / 2 + 255) / 256), 256, 0, e_buf[e_cur], size / 2, head,
                (const Fr*)(d_z + (round - 1)), eq_full);
      tabs.in[eq_slot] = eq_full;
    }
    QZ_CUDA(ctx, cudaEventRecord(ctx->ev_k1, st));
    nvtx_stream.reset();
    QzRange nvtx_mid("qz:sumcheck:short-rounds");
    ScTailBufs tb;
    memset(&tb, 0, sizeof tb);
    int mid_G = G;
    if (G > 1 && !mid_sharded) {
      // NCCL fallback: gather the ranks' shards (rank order = index order); every rank finishes the remaining rounds alone
      for (int j = 0; j < ka; j++) {
        uint4* full = (uint4*)ctx->arena_alloc(32 * size * G);
        if (!full) return ctx->fail(QZ_ERR_ALLOC, "gathered tables");
        rc = comm_allgather(ctx, tabs.in[j], full, 32 * size);
        if (rc) return rc;
        tabs.in[j] = full;
      }
      size *= G;
      mid_G = 1;
    }
    // sc_mid's fold scratch (never aliases its input): the first fold writes size / 2 elements, the second size / 4, ...;
    // after a gather the tables have 2^SC_TAIL_LOG elements again
    const uint64_t tail_half = ((uint64_t)1 << SC_TAIL_LOG) / 2;
    for (int j = 0; j < ka; j++) {
      tb.a[j] = (uint4*)ctx->arena_alloc(32 * std::max<uint64_t>(size / 2, tail_half));
      tb.b[j] = (uint4*)ctx->arena_alloc(32 * std::max<uint64_t>(size / 4, tail_half));
      if (!tb.a[j] || !tb.b[j]) return ctx->fail(QZ_ERR_ALLOC, "fold scratch of the short rounds");
    }
    // exchanges sc_mid will make with the peers: one per round before the gather, one for the gather itself
    uint32_t seq0 = 0;
    int gather_par = 0;
    if (mid_G > 1) {
      uint32_t n_ex = 0;
      uint64_t sz = size;
      for (int pend = pending; sz * G > ((uint64_t)1 << SC_TAIL_LOG); pend = 1) {
        n_ex++;
        if (pend) sz >>= 1;
      }
      n_ex++;
      seq0 = ctx->mbox_seq + 1;
      ctx->mbox_seq += n_ex;
      gather_par = (int)(ctx->gather_seq++ & 1);
    }
    {
      auto kern = sc_mid<0>;
      switch (cp.product_k) {
        case 1: kern = sc_mid<1>; break;
        case 2: kern = sc_mid<2>; break;
        case 3: kern = sc_mid<3>; break;
        case 4: kern = sc_mid<4>; break;
      }
      // the grid: as many blocks as the widest remaining round uses (the kernel derives every round's share from
      // gridDim.x with the same plan), all co-resident, and never more than a block has threads (the closing block
      // reads the parked vectors one per thread)
      int occ = blocks_per_sm(ctx, kern, SC_THREADS);
      if (occ < 1) occ = 1;
      const unsigned int cap = (unsigned int)std::min<uint64_t>(SC_THREADS, (uint64_t)ctx->sm_count * occ);
      ScMidPlan plan;
      const int grid = (int)mid_make_plan(plan, size, pending, ka, d, cap, mid_G);
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(grid);
      cfg.blockDim = dim3(SC_THREADS);
      cfg.stream = st;
      cudaLaunchAttribute at[1];
      if (grid > 1) {  // the blocks wait for one another: they must all be resident
        at[0].id = cudaLaunchAttributeCooperative;
        at[0].val.cooperative = 1;
      } else {
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
      }
      cfg.attrs = at;
      cfg.numAttrs = grid > 1 || (pdl_ok && G == 1) ? 1 : 0;
      QZ_CUDA(ctx, cudaLaunchKernelEx(&cfg, kern, tabs, tb, size, pending, head, (const ScProgram*)d_prog,
                                      (const Fr*)d_consts, (const Fr*)vinv, d_coeffs, d_lens, d_point, round, mc, partials,
                                      d_sync, (PeerMailbox* const*)ctx->peer_mbox_dev, ctx->rank, mid_G, seq0, gather_par,
                                      (const Fr*)d_z, zerocheck ? (int)num_vars : 0, plan));
      ctx->launches++;
    }
  }

  // results -> pinned staging -> caller
  QZ_CUDA(ctx, cudaMemcpyAsync(pin_out, d_out, zerocheck ? out_bytes : o_z, cudaMemcpyDeviceToHost, st));
  QZ_CUDA(ctx, cudaEventRecord(ctx->ev_call1, st));
  QZ_CUDA(ctx, cudaStreamSynchronize(st));
  const ScHead* h = (const ScHead*)(pin_out + o_head);
  if (h->peer_fault == 2) return ctx->fail(QZ_ERR_CUDA, "a block of the persistent round kernel never saw its round closed");
  if (h->peer_fault) return ctx->fail(QZ_ERR_NCCL, "a peer did not deliver its partial sums (peer mailbox wait timed out)");
  if (zc_skip1 && h->zc_degenerate)  // some z_j = 0 (probability 2^-254 per challenge): redo without the 1 / z_j shortcut
    return sumcheck_prove(ctx, num_vars, k, tables, tables_on_device, nodes, n_nodes, consts, n_consts, claimed_sum,
                          state, max_coeffs, out_coeffs, out_lens, out_point, out_eval, zerocheck, out_z, sharded,
                          false);  // every rank draws the same z, so every rank takes this branch
  memcpy(state, h->tstate, 32);
  memcpy(out_eval, h->evaluation.v, 32);
  if (num_vars) {
    memcpy(out_coeffs, pin_out + o_coeffs, coeff_bytes);
    memcpy(out_lens, pin_out + o_lens, lens_bytes);
    memcpy(out_point, pin_out + o_point, pt_bytes);
    if (zerocheck) memcpy(out_z, pin_out + o_z, pt_bytes);
  }
  cudaEventElapsedTime(&ctx->last_ms[0], ctx->ev_call0, ctx->ev_call1);
  if (num_vars > 0) cudaEventElapsedTime(&ctx->last_ms[1], ctx->ev_k0, ctx->ev_k1);
  else ctx->last_ms[1] = 0.f;
  return QZ_OK;
}

int sumcheck_run(qz_ctx* ctx, size_t num_vars, size_t k, const void* const* tables, int tables_on_device,
                 const qz_expr_node* nodes, size_t n_nodes, const uint8_t* consts, size_t n_consts,
                 const uint8_t* claimed_sum, uint8_t* state, size_t max_coeffs, uint8_t* out_coeffs,
                 uint32_t* out_lens, uint8_t* out_point, uint8_t* out_eval, bool zerocheck, uint8_t* out_z,
                 bool sharded) {
  return sumcheck_prove(ctx, num_vars, k, tables, tables_on_device, nodes, n_nodes, consts, n_consts, claimed_sum, state,
                        max_coeffs, out_coeffs, out_lens, out_point, out_eval, zerocheck, out_z, sharded, true);
}

}  // namespace qz

#ifdef QZ_SC_TRACE
extern "C" int qz_debug_trace(unsigned long long* out, int max_records) {
  unsigned int n = 0;
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(&n, qz::g_trace_n, 4);
  if (n > 8192) n = 8192;
  if ((int)n > max_records) n = max_records;
  cudaMemcpyFromSymbol(out, qz::g_trace, (size_t)n * 24);
  unsigned int zero = 0;
  cudaMemcpyToSymbol(qz::g_trace_n, &zero, 4);
  return (int)n;
}
#endif

// test hook (host logic only, no device needed): the plan sumcheck_run hands to sc_mid for tables of `size` entries per rank
// (pending != 0: a challenge is still to be folded in), k tables, degree d, at most `cap` co-resident blocks, G ranks.
// out_nblk / out_future / out_chunk: QZ_TEST_PLAN_ROUNDS entries each; returns the grid the launch would use.
extern "C" int qz_test_mid_plan(uint64_t size, int pending, int k, int d, unsigned int cap, int G, uint32_t* out_nblk,
                                uint32_t* out_future, uint32_t* out_chunk, uint32_t* out_tile) {
  if (!out_nblk || !out_future || !out_chunk || !out_tile || cap == 0 || G < 1) return -1;
  qz::ScMidPlan plan;
  const unsigned int grid = qz::mid_make_plan(plan, size, pending, k, d, cap, G);
  for (int j = 0; j < qz::SC_MAX_VARS; j++) {
    out_nblk[j] = plan.nblk[j];
    out_future[j] = plan.future[j];
    out_chunk[j] = plan.chunk[j];
  }
  *out_tile = plan.tile;
  return (int)grid;
}

extern "C" int qz_test_fold(qz_ctx* ctx, const uint8_t r[32], const uint8_t* a0, const uint8_t* a1, uint8_t* out, size_t n) {
  if (!ctx || !r || !a0 || !a1 || !out) return QZ_ERR_INVALID_ARG;
  if (n == 0) return QZ_OK;
  QZ_CUDA(ctx, cudaSetDevice(ctx->device));
  std::lock_guard<std::recursive_mutex> guard(qz::g_fold_table_lock[ctx->device & 15]);
  ctx->arena_reset();
  cudaStream_t st = ctx->stream;
  uint4 *d0 = (uint4*)ctx->arena_alloc(32 * n), *d1 = (uint4*)ctx->arena_alloc(32 * n), *dd = (uint4*)ctx->arena_alloc(32 * n);
  uint32_t* tab = (uint32_t*)ctx->arena_alloc(256);
  if (!d0 || !d1 || !dd || !tab) return ctx->fail(QZ_ERR_ALLOC, "scratch");
  Fr rr;
  memcpy(rr.v, r, 32);
  QZ_CUDA(ctx, cudaMemcpyAsync(d0, a0, 32 * n, cudaMemcpyHostToDevice, st));
  QZ_CUDA(ctx, cudaMemcpyAsync(d1, a1, 32 * n, cudaMemcpyHostToDevice, st));
  QZ_LAUNCH(ctx, k_fold_table, 1, 32, 0, rr, tab);
  QZ_CUDA(ctx, cudaMemcpyToSymbolAsync(qz::c_fold, tab, 256, 0, cudaMemcpyDeviceToDevice, st));
  QZ_LAUNCH(ctx, k_fold_fixed, (unsigned)((n + 127) / 128), 128, 0, (const uint4*)d0, (const uint4*)d1, dd, n);
  QZ_CUDA(ctx, cudaMemcpyAsync(out, dd, 32 * n, cudaMemcpyDeviceToHost, st));
  QZ_CUDA(ctx, cudaStreamSynchronize(st));
  return QZ_OK;
}
