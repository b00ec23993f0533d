// KZG commit = multi-scalar multiplication over BN254 G1, Pippenger style, for sm_100a.
//
// Reference: KZG::commit (pcs/src/kzg.rs:61-73), whose work is ark-ec 0.5.0's VariableBaseMSM::msm_unchecked on the
// affine-normalised SRS; KZG::open (pcs/src/kzg.rs:75-96); KZG::trusted_setup's G1 powers (pcs/src/kzg.rs:35-59).
//
// Pipeline (msm_run, after msm_plan; the first three stages run per range of the points, see segment_weights):
//   prep_segment         on the prep stream when there are several ranges, overlapped with the previous accumulation:
//     msm_digits         scalar: Montgomery -> canonical -> signed c-bit digits; one (key, value) per (window, scalar)
//                        key = window << c | |digit|, value = point index | sign << 31
//     radix sort         (key, value) pairs by key (cub::DeviceRadixSort) -> every bucket's points are contiguous
//   pair_levels          optional (QZ_MSM_PAIR_LEVELS = k, off by default): k halvings of the sorted list by affine
//                        additions with a shared inversion (msm_pair_*, section 4b below; DESIGN.md section 3)
//   msm_accumulate       the hot kernel: the sorted list is cut into fixed chunks of 32..128 entries, one thread per
//                        chunk, XYZZ += affine (8M + 2S) per entry with the next base prefetched; load is balanced
//                        whatever the scalar distribution.  A chunk's first / last runs may be partial buckets and go
//                        to a list of partial runs, interior runs are complete buckets and are written in place.
//   reduce_partial_runs  the list of partial runs is reduced by the same chunked rule, level by level, until it fits
//                        one chunk: no thread ever walks a whole bucket, however skewed the scalars are
//   reduce_and_combine   the ranges' bucket copies are added; per window sum_b b * B_b by segmented running sums + a
//                        tree reduction; Horner over windows (c doublings each) + one inversion to affine
// Bases are normalised to affine ONCE at SRS upload; the reference re-normalises on every commit (kzg.rs:67-71).
#include <cub/cub.cuh>
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>
#include "ctx.cuh"
#include "ec.cuh"
#include "msm.cuh"

namespace qz {

constexpr int ACC_CHUNK_MIN = 32;    // sorted entries per accumulate thread: 32 .. 128, longer for large inputs (every
constexpr int ACC_CHUNK_MAX = 128;   // chunk leaves up to two partial runs behind, each a full addition to merge later)
constexpr int ACC_THREADS = 128;
constexpr int RED_SEG = 32;          // buckets per bucket-reduce thread
constexpr uint32_t KEY_NONE = 0xffffffffu;

// ---- 1. digits ------------------------------------------------------------------------------------------------------------
// collapse_stride != 0: all windows share one bucket set (key = |digit|) and the value addresses the precomputed
// multiple 2^(c w) P_i stored at index w * collapse_stride + i (see srs_precompute).
// A segment of the points (streamed MSM, see msm_run) passes its scalars, its first point's index and `set_base`, the
// index of its first bucket set: segments are told apart by the key's high bits exactly as windows are.
__global__ void __launch_bounds__(256) msm_digits(const uint4* scalars, uint32_t n, uint32_t index_base, int c, int W,
                                                  uint32_t collapse_stride, uint32_t set_base, uint32_t* keys,
                                                  uint32_t* vals, unsigned long long* nonzero_digits) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t nz = 0;
  if (i < n) {
    const Fr k = fp_from_mont<FrParams>(fp_load<FrParams>(scalars + 2 * (size_t)i));
    const uint32_t mask = (1u << c) - 1, half = 1u << (c - 1);
    uint32_t carry = 0;
    for (int w = 0; w < W; w++) {
      const int bit = w * c, limb = bit >> 5, off = bit & 31;
      uint64_t two = 0;
      if (limb < 8) two = k.v[limb];
      if (limb + 1 < 8) two |= (uint64_t)k.v[limb + 1] << 32;
      uint32_t d = ((uint32_t)(two >> off) & mask) + carry;
      uint32_t neg = 0;
      carry = 0;
      if (d > half) {  // d in (2^(c-1), 2^c]  ->  -(2^c - d), carry one into the next window
        d = (1u << c) - d;
        neg = 1;
        carry = 1;
      }
      keys[(size_t)w * n + i] = ((set_base + (collapse_stride ? 0u : (uint32_t)w)) << c) | d;
      vals[(size_t)w * n + i] = ((uint32_t)w * collapse_stride + index_base + i) | (neg << 31);
      nz += d != 0;
    }
  }
  if (nonzero_digits) {  // measurement (qz_msm_accumulate_stats): the additions msm_accumulate will execute
    __shared__ uint32_t s_nz;
    if (threadIdx.x == 0) s_nz = 0;
    __syncthreads();
    nz = __reduce_add_sync(0xffffffffu, nz);
    if ((threadIdx.x & 31) == 0 && nz) atomicAdd(&s_nz, nz);
    __syncthreads();
    if (threadIdx.x == 0 && s_nz) atomicAdd(nonzero_digits, (unsigned long long)s_nz);
  }
}

// ---- 4. accumulate ----------------------------------------------------------------------------------------------------------
// A value with VAL_PAIR set addresses the array of pair sums (pair levels, below) instead of the bases.
constexpr uint32_t VAL_PAIR = 1u << 30;
constexpr uint32_t VAL_INDEX = VAL_PAIR - 1;
QZ_DEV const uint8_t* entry_point(const uint8_t* bases, const uint8_t* sums, uint32_t val) {
  return ((val & VAL_PAIR) ? sums : bases) + (size_t)(val & VAL_INDEX) * 64;
}
QZ_DEV Affine load_base(const uint8_t* bases, uint32_t val) {
  Affine a = affine_load(bases + (size_t)(val & 0x7fffffffu) * 64);
  if (val >> 31) a.y = fp_neg<FqParams>(a.y);
  return a;
}
QZ_DEV Affine load_entry(const uint8_t* bases, const uint8_t* sums, uint32_t val) {
  Affine a = affine_load(entry_point(bases, sums, val));
  if (val >> 31) a.y = fp_neg<FqParams>(a.y);
  return a;
}
QZ_DEV uint32_t bucket_slot(uint32_t key, int c) {  // dense slot of a non-zero digit: window * 2^(c-1) + |d| - 1
  const uint32_t w = key >> c, d = key & ((1u << c) - 1);
  return (w << (c - 1)) + d - 1;
}

// Partial runs go to a list of (key, XYZZ) slots, two per chunk: slot 2*chunk = the run touching the chunk's start,
// slot 2*chunk + 1 = the run touching its end (KEY_NONE = empty).  Keys of non-empty slots are non-decreasing.
// PAIRED: the list went through the pair levels first -- its length is read from device memory (the launch covers the
// `n_chunks` chunks of the longest list possible; chunks past the end leave empty slots) and values may address `sums`.
template <bool PAIRED>
__global__ void __launch_bounds__(ACC_THREADS, 4) msm_accumulate(const uint32_t* keys, const uint32_t* vals, uint64_t m_host,
                                                              const uint64_t* m_dev, uint64_t n_chunks, int chunk_len,
                                                              const uint8_t* bases, const uint8_t* sums, int c,
                                                              uint8_t* buckets, uint8_t* ppts, uint32_t* pkeys) {
  const uint64_t chunk = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t begin = chunk * chunk_len;
  uint64_t m = m_host;
  if constexpr (PAIRED) {
    m = *m_dev;
    if (begin >= m) {
      if (chunk < n_chunks) {
        pkeys[2 * chunk] = KEY_NONE;
        pkeys[2 * chunk + 1] = KEY_NONE;
      }
      return;
    }
  } else {
    if (begin >= m) return;
  }
  auto load = [&](uint32_t val) { return PAIRED ? load_entry(bases, sums, val) : load_base(bases, val); };
  uint8_t* heads = ppts;             // slot 2*chunk
  uint8_t* tails = ppts + 128;       // slot 2*chunk + 1
  const uint64_t end = begin + chunk_len < m ? begin + chunk_len : m;
  const uint32_t dmask = (1u << c) - 1;
  Xyzz acc = xyzz_identity();
  uint32_t cur_key = keys[begin];
  bool first = true;
  uint32_t hk = KEY_NONE, tk = KEY_NONE;
  uint32_t nk = cur_key, nv = vals[begin];
  Affine npt = (nk & dmask) ? load(nv) : Affine{fp_zero<FqParams>(), fp_zero<FqParams>()};
  for (uint64_t j = begin; j < end; j++) {
    const uint32_t k = nk;
    const Affine pt = npt;
    if (j + 1 < end) {  // prefetch the next entry's base while this one is added
      nk = keys[j + 1];
      nv = vals[j + 1];
      if (nk & dmask) npt = load(nv);
    }
    if (k != cur_key) {  // the run of cur_key ended inside the chunk
      if (cur_key & dmask) {
        if (first) {  // it started at the chunk border: possibly the tail end of a bucket begun in earlier chunks
          xyzz_store(heads + chunk * 256, acc);
          hk = cur_key;
        } else {  // strictly interior: a complete bucket
          xyzz_store(buckets + (size_t)bucket_slot(cur_key, c) * 128, acc);
        }
      }
      acc = xyzz_identity();
      cur_key = k;
      first = false;
    }
    if (k & dmask) acc = xyzz_add_affine(acc, pt);
  }
  if (cur_key & dmask) {  // the last run touches the chunk's end and may continue in the next chunk
    if (first) {
      xyzz_store(heads + chunk * 256, acc);
      hk = cur_key;
    } else {
      xyzz_store(tails + chunk * 256, acc);
      tk = cur_key;
    }
  }
  pkeys[2 * chunk] = hk;
  pkeys[2 * chunk + 1] = tk;
}

// ---- 4b. pair levels: affine additions with a shared inversion, ahead of the accumulation --------------------------
// A mixed addition into an XYZZ accumulator is 10 products.  Two AFFINE points add in 1 inversion + 3 products, and
// Montgomery's trick turns n inversions into one inversion + 3 (n - 1) products, i.e. ~6 products per addition when
// the batch is large.  A level pairs the entries at positions (2p, 2p + 1) of the sorted list: when both carry the same
// non-zero key, their sum is written to the array of pair sums and ONE entry (key, VAL_PAIR | index of the sum) takes
// their place; any other pair passes through unchanged (zero digits are dropped), so the output is again a list sorted
// by key whose entries sum to the same buckets, about half as long.  L levels leave runs of ~r / 2^L entries for the
// XYZZ accumulation, where r = entries per bucket.  Pairs that cannot be added by the affine chord rule -- equal x
// (P + P, P - P) or an infinite point -- pass through as well: the complete XYZZ law downstream handles them, which
// keeps this stage free of special cases.
// A block owns a tile of PAIR_TILE consecutive pairs; thread i takes pairs i, i + 128, i + 256, .. of the tile, so that
// a warp's accesses to the keys, values, prefixes, outputs and (from level 2 on) the points are to neighbouring
// addresses.  One level = three passes, with no thread ever waiting on an inversion:
//   scan   d = x_b - x_a per pair; running product of the thread's d's (prefix[pair] = the product BEFORE the pair),
//          the thread's total, a code per pair (outputs 0..2, summed or not) and the tile's output / sum counts
//   invert the threads' totals, by a product tree of fan-in PAIR_G: up to ONE root, inverted by one thread (binary
//          Euclid), and down again; every step is a short launch of chains of PAIR_G products
//   apply  walks the thread's pairs backwards: 1/d = inv * prefix, inv *= d; lambda = (y_b - y_a) / d,
//          x3 = lambda^2 - x_a - x_b, y3 = lambda (x_a - x3) - y_a.  Outputs land, in list order, at the tile's base
//          (exclusive scan of the tiles' counts) + the pair's offset inside the tile (block scan of the codes).
// The list lengths live on the device (PairCtl): launches cover the longest list possible and tiles past the end
// return, so the host never synchronises.  The sums written by all levels number at most m - 1 (every sum shortens
// the list by one): the array of m slots cannot overflow whatever the input.
constexpr int PAIR_B = 16;            // pairs per thread
constexpr int PAIR_THREADS = 128;
constexpr int PAIR_TILE = PAIR_B * PAIR_THREADS;  // pairs per block
constexpr int PAIR_G = 16;            // fan-in of the inversion's product tree (short chains: the tree is pure latency)
constexpr int PAIR_TREE_MAX = 10;     // depths: 16^8 threads' totals and more
constexpr int PAIR_MAX_LEVELS = 8;
struct PairCtl {
  uint64_t m[PAIR_MAX_LEVELS + 1];     // m[l]: entries entering level l; m[L]: entries left for msm_accumulate
  uint64_t sums[PAIR_MAX_LEVELS + 1];  // sums[l]: pair sums written by the levels before l
};
__global__ void msm_pair_init(PairCtl* ctl, uint64_t m, unsigned long long* counts_last) {
  for (int l = 0; l <= PAIR_MAX_LEVELS; l++) {
    ctl->m[l] = l == 0 ? m : 0;
    ctl->sums[l] = 0;
  }
  *counts_last = 0;  // the scan's extra item: offs[n_tiles] = the totals
}
// entries a = 2p, a + 1 of pair p: keys and values (0 past the end of the list: a zero digit)
QZ_DEV void pair_entries(const uint32_t* keys, const uint32_t* vals, uint64_t a, uint64_t m, uint32_t& ka, uint32_t& kb,
                         uint32_t& va, uint32_t& vb) {
  ka = kb = va = vb = 0;
  if (a + 1 < m) {  // a is even and the lists are 8-byte aligned
    const uint2 k2 = *reinterpret_cast<const uint2*>(keys + a), v2 = *reinterpret_cast<const uint2*>(vals + a);
    ka = k2.x, kb = k2.y, va = v2.x, vb = v2.y;
  } else if (a < m) {
    ka = keys[a], va = vals[a];
  }
}
// codes: bits 0-1 = outputs of the pair (0..2), bit 2 = the pair is summed (then one output)
__global__ void __launch_bounds__(PAIR_THREADS, 8) msm_pair_scan(const uint32_t* keys, const uint32_t* vals, const PairCtl* ctl,
                                                               int level, uint32_t dmask, const uint8_t* bases,
                                                               const uint8_t* sums, uint8_t* prefix, uint8_t* totals,
                                                               uint8_t* codes, unsigned long long* counts) {
  __shared__ unsigned long long s_cnt[PAIR_THREADS / 32];
  const uint64_t m = ctl->m[level], tile0 = (uint64_t)blockIdx.x * PAIR_TILE;
  const int i = threadIdx.x;
  if (2 * tile0 >= m) {
    if (i == 0) counts[blockIdx.x] = 0;
    return;
  }
  Fq run = fp_one<FqParams>();
  uint32_t n_out = 0, n_sum = 0;
#pragma unroll 1
  for (int j = 0; j < PAIR_B; j++) {
    const uint64_t p = tile0 + (uint64_t)j * PAIR_THREADS + i, a = 2 * p;
    uint32_t ka, kb, va, vb;
    pair_entries(keys, vals, a, m, ka, kb, va, vb);
    uint32_t code = ((ka & dmask) != 0) + ((kb & dmask) != 0);
    if (ka == kb && (ka & dmask)) {
      const Fq xa = fp_load<FqParams>(entry_point(bases, sums, va));
      const Fq xb = fp_load<FqParams>(entry_point(bases, sums, vb));
      const Fq d = fp_sub<FqParams>(xb, xa);
      if (!fp_is_zero<FqParams>(xa) && !fp_is_zero<FqParams>(xb) && !fp_is_zero<FqParams>(d)) {
        code = 4 | 1;
        fp_store<FqParams>(prefix + p * 32, run);
        run = fp_mul<FqParams>(run, d);
      }
    }
    codes[p] = (uint8_t)code;
    n_out += code & 3;
    n_sum += code >> 2;
  }
  fp_store<FqParams>(totals + ((uint64_t)blockIdx.x * PAIR_THREADS + i) * 32, run);
  unsigned long long cnt = (unsigned long long)n_out | ((unsigned long long)n_sum << 32);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) cnt += __shfl_down_sync(0xffffffffu, cnt, off);
  if ((i & 31) == 0) s_cnt[i >> 5] = cnt;
  __syncthreads();
  if (i == 0) {
    unsigned long long total = 0;
    for (int w = 0; w < PAIR_THREADS / 32; w++) total += s_cnt[w];
    counts[blockIdx.x] = total;
  }
}
// elements of the inversion tree at `depth` above the threads' totals (depth 0) for the list entering `level`
QZ_DEV uint64_t pair_tree_count(const PairCtl* ctl, int level, int depth) {
  uint64_t n = (ctl->m[level] + 2 * PAIR_TILE - 1) / (2 * PAIR_TILE) * PAIR_THREADS;
  for (int k = 0; k < depth; k++) n = (n + PAIR_G - 1) / PAIR_G;
  return n;
}
__global__ void __launch_bounds__(128) msm_pair_tree_up(const PairCtl* ctl, int level, int depth, const uint8_t* v, uint8_t* pre,
                                                        uint8_t* v_up) {
  const uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t n = pair_tree_count(ctl, level, depth);
  if (u * PAIR_G >= n) return;
  const uint64_t end = u * PAIR_G + PAIR_G < n ? u * PAIR_G + PAIR_G : n;
  Fq run = fp_one<FqParams>();
  for (uint64_t i = u * PAIR_G; i < end; i++) {
    fp_store<FqParams>(pre + i * 32, run);
    run = fp_mul<FqParams>(run, fp_load<FqParams>(v + i * 32));
  }
  fp_store<FqParams>(v_up + u * 32, run);
}
// the root: ONE element (the host climbs until the longest list possible is down to one), inverted by one thread
__global__ void msm_pair_tree_root(const PairCtl* ctl, int level, uint8_t* v) {
  if (pair_tree_count(ctl, level, 0) == 0) return;  // empty list: nothing was written below, nothing to invert
  fp_store<FqParams>(v, fp_inv_serial<FqParams>(fp_load<FqParams>(v)));  // a product of non-zero d's: never 0
}
__global__ void __launch_bounds__(128) msm_pair_tree_down(const PairCtl* ctl, int level, int depth, uint8_t* v, const uint8_t* pre,
                                                          const uint8_t* v_up) {
  const uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t n = pair_tree_count(ctl, level, depth);
  if (u * PAIR_G >= n) return;
  const uint64_t end = u * PAIR_G + PAIR_G < n ? u * PAIR_G + PAIR_G : n;
  Fq inv = fp_load<FqParams>(v_up + u * 32);  // 1 / (product of this thread's elements)
  for (uint64_t i = end; i-- > u * PAIR_G;) {
    const Fq x = fp_load<FqParams>(v + i * 32);
    fp_store<FqParams>(v + i * 32, fp_mul<FqParams>(inv, fp_load<FqParams>(pre + i * 32)));
    inv = fp_mul<FqParams>(inv, x);
  }
}
__global__ void __launch_bounds__(PAIR_THREADS, 4) msm_pair_apply(const uint32_t* keys, const uint32_t* vals, PairCtl* ctl, int level,
                                                                uint32_t dmask, const uint8_t* bases, uint8_t* sums,
                                                                const uint8_t* prefix, const uint8_t* totals_inv,
                                                                const uint8_t* codes, const unsigned long long* offs,
                                                                uint32_t n_tiles, uint32_t* keys_out, uint32_t* vals_out) {
  // per pair: offset of its outputs inside the tile (bits 0-15) and of its sum (bits 16-28), its code (bits 29-31)
  __shared__ uint32_t s_off[PAIR_B][PAIR_THREADS];
  __shared__ uint32_t s_warp[PAIR_B][PAIR_THREADS / 32];
  const uint64_t m = ctl->m[level], sum_base = ctl->sums[level], tile0 = (uint64_t)blockIdx.x * PAIR_TILE;
  const int i = threadIdx.x, lane = i & 31, warp = i >> 5;
  if (blockIdx.x == 0 && i == 0) {  // the next level's list length and first free sum slot
    const unsigned long long total = offs[n_tiles];
    ctl->m[level + 1] = total & 0xffffffffull;
    ctl->sums[level + 1] = sum_base + (total >> 32);
  }
  if (2 * tile0 >= m) return;
#pragma unroll
  for (int j = 0; j < PAIR_B; j++) {  // offsets in list order: row j of the tile = pairs j * 128 .. j * 128 + 127
    const uint32_t code = codes[tile0 + (uint64_t)j * PAIR_THREADS + i];
    const uint32_t v = (code & 3) | ((code >> 2) << 16);
    uint32_t incl = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const uint32_t up = __shfl_up_sync(0xffffffffu, incl, off);
      if (lane >= off) incl += up;
    }
    s_off[j][i] = (incl - v) | (code << 29);
    if (lane == 31) s_warp[j][warp] = incl;
  }
  __syncthreads();
  if (i == 0) {
    uint32_t running = 0;
    for (int j = 0; j < PAIR_B; j++)
      for (int w = 0; w < PAIR_THREADS / 32; w++) {
        const uint32_t t = s_warp[j][w];
        s_warp[j][w] = running;
        running += t;
      }
  }
  __syncthreads();
  const unsigned long long tile_off = offs[blockIdx.x];
  const uint64_t pos_base = tile_off & 0xffffffffull, sidx_base = sum_base + (tile_off >> 32);
  Fq inv = fp_load<FqParams>(totals_inv + ((uint64_t)blockIdx.x * PAIR_THREADS + i) * 32);
#pragma unroll 1
  for (int j = PAIR_B - 1; j >= 0; j--) {
    const uint32_t packed = s_off[j][i], code = packed >> 29;
    if ((code & 3) == 0) continue;  // nothing to write (both digits zero, or past the end of the list)
    const uint32_t off = (packed & 0x1fffffffu) + s_warp[j][warp];
    const uint64_t p = tile0 + (uint64_t)j * PAIR_THREADS + i, a = 2 * p;
    uint64_t pos = pos_base + (off & 0xffffu);
    uint32_t ka, kb, va, vb;
    pair_entries(keys, vals, a, m, ka, kb, va, vb);
    if (code & 4) {
      // both points and the prefix are requested together: one memory round trip per pair
      const uint8_t* pa = entry_point(bases, sums, va);
      const uint8_t* pb = entry_point(bases, sums, vb);
      const Fq xa = fp_load<FqParams>(pa), xb = fp_load<FqParams>(pb);
      Fq ya = fp_load<FqParams>(pa + 32), yb = fp_load<FqParams>(pb + 32);
      const Fq pre = fp_load<FqParams>(prefix + p * 32);
      const Fq d = fp_sub<FqParams>(xb, xa);
      if (va >> 31) ya = fp_neg<FqParams>(ya);
      if (vb >> 31) yb = fp_neg<FqParams>(yb);
      const Fq dinv = fp_mul<FqParams>(inv, pre);
      inv = fp_mul<FqParams>(inv, d);
      const Fq lam = fp_mul<FqParams>(fp_sub<FqParams>(yb, ya), dinv);
      Affine r;
      r.x = fp_sub<FqParams>(fp_sub<FqParams>(fp_sqr<FqParams>(lam), xa), xb);
      r.y = fp_sub<FqParams>(fp_mul<FqParams>(lam, fp_sub<FqParams>(xa, r.x)), ya);
      const uint64_t sidx = sidx_base + (off >> 16);
      affine_store(sums + sidx * 64, r);
      keys_out[pos] = ka;
      vals_out[pos] = VAL_PAIR | (uint32_t)sidx;
    } else {
      if (ka & dmask) {
        keys_out[pos] = ka;
        vals_out[pos] = va;
        pos++;
      }
      if (kb & dmask) {
        keys_out[pos] = kb;
        vals_out[pos] = vb;
      }
    }
  }
}

// ---- 5. merge the partial runs, level by level ---------------------------------------------------------------------
// The partial list is cut into chunks of PART_CHUNK slots, one thread per chunk, and reduced by the same rule as the
// points were: a run of equal keys strictly inside a chunk is a complete bucket (written in place), the runs touching
// the chunk's ends go to the next level's list.  At the level that fits one chunk every run is complete.  The depth is
// log_{PART_CHUNK/2}(#chunks) and every level is fully parallel, so one huge bucket (all scalars equal, selector
// columns, small witness values) costs no more than a uniform distribution.
// A level is latency-bound (a full addition is ~5 us on a lone warp and a thread adds its slots serially), so the
// chunks are short: every level divides the list by PART_CHUNK / 2 in about PART_CHUNK addition latencies.
constexpr int PART_CHUNK = 8;
__global__ void __launch_bounds__(128) msm_partials_reduce(const uint32_t* pkeys_in, const uint8_t* ppts_in, uint64_t n_in,
                                                           int c, uint8_t* buckets, uint32_t* pkeys_out, uint8_t* ppts_out,
                                                           int last_level) {
  const uint64_t chunk = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t begin = chunk * PART_CHUNK;
  if (begin >= n_in) return;
  const uint64_t end = begin + PART_CHUNK < n_in ? begin + PART_CHUNK : n_in;
  Xyzz acc = xyzz_identity();
  uint32_t cur = KEY_NONE, hk = KEY_NONE, tk = KEY_NONE;
  bool first = true;
  for (uint64_t i = begin; i < end; i++) {
    const uint32_t k = pkeys_in[i];
    if (k == KEY_NONE) continue;
    if (cur != KEY_NONE && k != cur) {  // the run of `cur` ended inside the chunk
      if (first && !last_level) {
        xyzz_store(ppts_out + chunk * 256, acc);
        hk = cur;
      } else {
        xyzz_store(buckets + (size_t)bucket_slot(cur, c) * 128, acc);
      }
      acc = xyzz_identity();
      first = false;
    }
    cur = k;
    Xyzz p;
    xyzz_load(p, ppts_in + i * 128);
    acc = xyzz_add(acc, p);
  }
  if (cur != KEY_NONE) {
    if (last_level) {
      xyzz_store(buckets + (size_t)bucket_slot(cur, c) * 128, acc);
    } else if (first) {
      xyzz_store(ppts_out + chunk * 256, acc);
      hk = cur;
    } else {
      xyzz_store(ppts_out + chunk * 256 + 128, acc);
      tk = cur;
    }
  }
  if (!last_level) {
    pkeys_out[2 * chunk] = hk;
    pkeys_out[2 * chunk + 1] = tk;
  }
}

// Last levels in one launch: once the list is short (<= FIN_SLOTS) the level-by-level rule is pure latency (each level
// a launch plus up to PART_CHUNK dependent additions for a handful of runs: ~33 us x 7 levels at 2^21 points).  One
// block compacts the non-empty slots and runs a segmented Hillis-Steele scan over them -- keys ascend, so slot i may
// add slot i-d whenever their keys are equal -- stopping as soon as a step adds nothing (runs at this depth are
// mostly pairs: two or three steps).  The last slot of every run then holds the bucket.
constexpr int FIN_SLOTS = 2048, FIN_THREADS = 512;  // 512 threads: the full addition needs ~128 registers
__global__ void __launch_bounds__(FIN_THREADS) msm_partials_finish(const uint32_t* pkeys_in, const uint8_t* ppts_in,
                                                                   int n_in, int c, uint8_t* buckets, uint8_t* scratch_a,
                                                                   uint8_t* scratch_b) {
  __shared__ uint32_t ck[FIN_SLOTS];
  __shared__ uint16_t src[FIN_SLOTS];
  __shared__ int warp_tot[FIN_THREADS / 32];
  __shared__ int s_m;
  constexpr int PER = FIN_SLOTS / FIN_THREADS;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  // compact: thread t owns slots [t * PER, t * PER + PER)
  uint32_t k[PER];
  int cnt = 0;
#pragma unroll
  for (int j = 0; j < PER; j++) {
    const int i = t * PER + j;
    k[j] = i < n_in ? pkeys_in[i] : KEY_NONE;
    cnt += k[j] != KEY_NONE;
  }
  int incl = cnt;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, off);
    if (lane >= off) incl += v;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int v = lane < FIN_THREADS / 32 ? warp_tot[lane] : 0;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, v, off);
      if (lane >= off) v += u;
    }
    if (lane < FIN_THREADS / 32) warp_tot[lane] = v;  // inclusive totals per warp
    if (lane == 31) s_m = v;
  }
  __syncthreads();
  int pos = incl - cnt + (warp ? warp_tot[warp - 1] : 0);
#pragma unroll
  for (int j = 0; j < PER; j++)
    if (k[j] != KEY_NONE) {
      ck[pos] = k[j];
      src[pos] = (uint16_t)(t * PER + j);
      pos++;
    }
  __syncthreads();
  const int m = s_m;
  // segmented inclusive scan over the m compacted slots; step 0 reads the input list through src[]
  const uint8_t* in = nullptr;
  uint8_t* out = scratch_a;
  for (int d = 1; d < m || d == 1; d <<= 1) {
    int added = 0;
    for (int i = t; i < m; i += FIN_THREADS) {
      Xyzz a;
      xyzz_load(a, in ? in + (size_t)i * 128 : ppts_in + (size_t)src[i] * 128);
      if (i >= d && ck[i - d] == ck[i]) {
        Xyzz b;
        xyzz_load(b, in ? in + (size_t)(i - d) * 128 : ppts_in + (size_t)src[i - d] * 128);
        a = xyzz_add(a, b);
        added = 1;
      }
      xyzz_store(out + (size_t)i * 128, a);
    }
    const int any = __syncthreads_or(added);  // also orders this step's stores before the next step's loads
    in = out;
    out = out == scratch_a ? scratch_b : scratch_a;
    if (!any) break;
  }
  for (int i = t; i < m; i += FIN_THREADS)
    if (i + 1 == m || ck[i + 1] != ck[i]) {
      Xyzz a;
      xyzz_load(a, in + (size_t)i * 128);
      xyzz_store(buckets + (size_t)bucket_slot(ck[i], c) * 128, a);
    }
}

// streamed MSM: every segment of the points filled its own copy of the bucket sets; add copies 1 .. S-1 into copy 0
__global__ void __launch_bounds__(128) msm_bucket_merge(uint8_t* buckets, uint32_t n_slots, int S) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_slots) return;
  Xyzz acc;
  xyzz_load(acc, buckets + (size_t)t * 128);
  for (int s = 1; s < S; s++) {
    Xyzz p;
    xyzz_load(p, buckets + ((size_t)s * n_slots + t) * 128);
    acc = xyzz_add(acc, p);
  }
  xyzz_store(buckets + (size_t)t * 128, acc);
}

// ---- 6. bucket reduction: window sum = sum_{b=1..2^(c-1)} b * B_b ----------------------------------------------------------
// thread t of a window owns buckets (digits) lo+1 .. lo+seg with lo = t*seg:  sum_j (lo + j) B_{lo+j} = acc + lo * S
__global__ void __launch_bounds__(128) msm_bucket_reduce(const uint8_t* buckets, int c, int W, int seg, uint8_t* partial) {
  const uint32_t per_w = 1u << (c - 1), threads_per_w = per_w / seg;
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (uint32_t)W * threads_per_w) return;
  const uint32_t w = t / threads_per_w, tw = t % threads_per_w, lo = tw * seg;
  const uint8_t* base = buckets + ((size_t)w * per_w + lo) * 128;
  Xyzz running = xyzz_identity(), acc = xyzz_identity();
  for (int j = seg - 1; j >= 0; j--) {
    Xyzz b;
    xyzz_load(b, base + (size_t)j * 128);
    running = xyzz_add(running, b);
    acc = xyzz_add(acc, running);
  }
  if (lo && !xyzz_is_identity(running)) {  // + lo * S (double-and-add, lo < 2^15)
    Xyzz mul = xyzz_identity();
    for (int bit = 31 - __clz(lo); bit >= 0; bit--) {
      mul = xyzz_dbl(mul);
      if ((lo >> bit) & 1) mul = xyzz_add(mul, running);
    }
    acc = xyzz_add(acc, mul);
  }
  xyzz_store(partial + (size_t)t * 128, acc);
}
// tree-sum of XYZZ points: block (w, j) adds elements [j * SUM_SPAN, (j + 1) * SUM_SPAN) of window w's `per_in` inputs
// and writes output j of `per_out`; applied repeatedly until one point per window is left
constexpr uint32_t SUM_SPAN = 1024;
__global__ void __launch_bounds__(128) msm_block_sum(const uint8_t* in, uint32_t per_in, uint32_t per_out, uint8_t* out) {
  __shared__ __align__(16) uint8_t sh[128 * 128];
  const uint32_t w = blockIdx.x / per_out, j = blockIdx.x % per_out;
  const uint32_t begin = j * SUM_SPAN, end = begin + SUM_SPAN < per_in ? begin + SUM_SPAN : per_in;
  Xyzz acc = xyzz_identity();
  for (uint32_t i = begin + threadIdx.x; i < end; i += blockDim.x) {
    Xyzz p;
    xyzz_load(p, in + ((size_t)w * per_in + i) * 128);
    acc = xyzz_add(acc, p);
  }
  xyzz_store(sh + threadIdx.x * 128, acc);
  __syncthreads();
  for (int s = blockDim.x / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) {
      Xyzz a, b;
      xyzz_load(a, sh + threadIdx.x * 128);
      xyzz_load(b, sh + (threadIdx.x + s) * 128);
      xyzz_store(sh + threadIdx.x * 128, xyzz_add(a, b));
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    Xyzz r;
    xyzz_load(r, sh);
    xyzz_store(out + ((size_t)w * per_out + j) * 128, r);
  }
}

// ---- 7. window combine + affine conversion --------------------------------------------------------------------------------
__global__ void msm_combine(const uint8_t* window_sums, int c, int W, uint8_t* out_xyzz, uint8_t* out_affine) {
  Xyzz total;
  xyzz_load(total, window_sums + (size_t)(W - 1) * 128);
  for (int w = W - 2; w >= 0; w--) {
    for (int j = 0; j < c; j++) total = xyzz_dbl(total);
    Xyzz p;
    xyzz_load(p, window_sums + (size_t)w * 128);
    total = xyzz_add(total, p);
  }
  if (out_xyzz) xyzz_store(out_xyzz, total);
  if (out_affine) affine_store(out_affine, xyzz_to_affine_serial(total));
}
// sum of `n` XYZZ points (multi-GPU: the gathered per-rank partial sums) -> affine
__global__ void msm_sum_points(const uint8_t* pts, int n, uint8_t* out_affine) {
  Xyzz total = xyzz_identity();
  for (int i = 0; i < n; i++) {
    Xyzz p;
    xyzz_load(p, pts + (size_t)i * 128);
    total = xyzz_add(total, p);
  }
  affine_store(out_affine, xyzz_to_affine_serial(total));
}

// ---- SRS generation: points[i] = tau^i * g (kzg.rs:44-47), fixed-base 8-bit windows -------------------------------------
// table[w*255 + d-1] = (d << 8w) * g, affine
__global__ void srs_table_bases(Affine g, uint8_t* pow_bases /*32 affine: 2^(8w) g*/) {
  const int w = threadIdx.x;
  if (w >= 32) return;
  Xyzz p = xyzz_from_affine(g);
  for (int i = 0; i < 8 * w; i++) p = xyzz_dbl(p);
  affine_store(pow_bases + w * 64, xyzz_to_affine(p));
}
__global__ void srs_table_fill(const uint8_t* pow_bases, uint8_t* table) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 32 * 255) return;
  const int w = idx / 255, d = idx % 255 + 1;
  const Affine b = affine_load(pow_bases + w * 64);
  Xyzz acc = xyzz_identity();
  for (int bit = 7; bit >= 0; bit--) {
    acc = xyzz_dbl(acc);
    if ((d >> bit) & 1) acc = xyzz_add_affine(acc, b);
  }
  affine_store(table + (size_t)idx * 64, xyzz_to_affine(acc));
}
// Affine conversion of a thread's batch of points with ONE inversion (Montgomery's trick on the denominators zz * zzz):
// 8 products per point instead of the 380 of a Fermat inversion.  pts[0 .. cnt) stay in local memory; `store(j, a)`
// receives the affine point.  Identity points (zz = 0) are skipped in the product and come out as (0, 0).
template <int MAXN, class Store>
QZ_DEV void xyzz_batch_to_affine(const Xyzz* pts, int cnt, Store store) {
  Fq pref[MAXN];
  Fq run = fp_one<FqParams>();
  for (int j = 0; j < cnt; j++) {
    pref[j] = run;
    if (!xyzz_is_identity(pts[j])) run = fp_mul<FqParams>(run, fp_mul<FqParams>(pts[j].zz, pts[j].zzz));
  }
  Fq inv = fp_inv<FqParams>(run);
  for (int j = cnt - 1; j >= 0; j--) {
    Affine a;
    a.x = fp_zero<FqParams>();
    a.y = fp_zero<FqParams>();
    if (!xyzz_is_identity(pts[j])) {
      const Fq dinv = fp_mul<FqParams>(inv, pref[j]);  // 1 / (zz_j zzz_j)
      inv = fp_mul<FqParams>(inv, fp_mul<FqParams>(pts[j].zz, pts[j].zzz));
      a.x = fp_mul<FqParams>(pts[j].x, fp_mul<FqParams>(dinv, pts[j].zzz));
      a.y = fp_mul<FqParams>(pts[j].y, fp_mul<FqParams>(dinv, pts[j].zz));
    }
    store(j, a);
  }
}

constexpr int SRS_CHUNK = 8;
__global__ void __launch_bounds__(128) srs_generate(const uint8_t* table, Fr tau, uint64_t n, uint8_t* out) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t begin = t * SRS_CHUNK;
  if (begin >= n) return;
  // tau^begin by square-and-multiply
  Fr ti = fp_one<FrParams>();
  for (int bit = 63 - __clzll(begin | 1); bit >= 0; bit--) {
    ti = fp_sqr<FrParams>(ti);
    if ((begin >> bit) & 1) ti = fp_mul<FrParams>(ti, tau);
  }
  const uint64_t end = begin + SRS_CHUNK < n ? begin + SRS_CHUNK : n;
  Xyzz pts[SRS_CHUNK];
  for (uint64_t i = begin; i < end; i++) {
    const Fr k = fp_from_mont<FrParams>(ti);
    Xyzz acc = xyzz_identity();
    for (int w = 0; w < 32; w++) {
      const uint32_t d = (k.v[w >> 2] >> (8 * (w & 3))) & 0xffu;
      if (d) acc = xyzz_add_affine(acc, affine_load(table + (size_t)(w * 255 + d - 1) * 64));
    }
    pts[i - begin] = acc;
    ti = fp_mul<FrParams>(ti, tau);
  }
  xyzz_batch_to_affine<SRS_CHUNK>(pts, (int)(end - begin), [&](int j, const Affine& a) { affine_store(out + (begin + j) * 64, a); });
}

// pre[w * n + i] = 2^(c w) * P_i (affine), w < W: with these multiples every window of a scalar lands in ONE shared set
// of buckets, so an MSM needs ceil(256 / c) * n mixed additions with a c far larger than a per-window bucket array
// would allow (c = 22, 12 additions per point at n = 2^24 instead of 16), one bucket reduction and no window-combine
// doublings.  It costs W x the SRS in HBM (12 GiB at 2^24): a trade a 180 GB part can make.
// A thread walks its point through the windows in XYZZ and converts PRE_BATCH multiples to affine with one inversion.
constexpr int PRE_BATCH = 16;
__global__ void __launch_bounds__(128) srs_precompute(const uint8_t* bases, uint64_t n, int c, int W, uint8_t* pre) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Affine p = affine_load(bases + i * 64);
  affine_store(pre + i * 64, p);
  Xyzz acc = xyzz_from_affine(p);
  Xyzz pts[PRE_BATCH];
  for (int w0 = 1; w0 < W; w0 += PRE_BATCH) {
    const int cnt = W - w0 < PRE_BATCH ? W - w0 : PRE_BATCH;
    for (int j = 0; j < cnt; j++) {
      for (int b = 0; b < c; b++) acc = xyzz_dbl(acc);
      pts[j] = acc;
    }
    xyzz_batch_to_affine<PRE_BATCH>(pts, cnt, [&](int j, const Affine& a) { affine_store(pre + ((uint64_t)(w0 + j) * n + i) * 64, a); });
  }
}

// ---- KZG::open pieces (kzg.rs:75-96) -----------------------------------------------------------------------------------------------
// The quotient of p(X) - p(x) by (X - x) is q_{i-1} = p_i + x q_i, i.e. q_{i-1} = sum_{j >= i} p_j x^{j-i}: a suffix
// scan with multiplier x.  Three passes over chunks of OPEN_CHUNK coefficients:
//   A. per chunk: local Horner value  h_c = sum_{j in chunk} p_j x^{j - start_c}
//   B. one block: carry_c = value entering chunk c from the right = sum_{c' > c} h_{c'} x^{start_{c'} - end_c}
//   C. per chunk: rerun the recurrence with the carry, writing q; chunk 0's final value is y = p(x).
constexpr int OPEN_CHUNK = 64;
__global__ void __launch_bounds__(128) open_local(const uint4* p, uint64_t n, const Fr* xp, Fr* h) {
  const Fr x = *xp;
  const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t begin = c * OPEN_CHUNK;
  if (begin >= n) return;
  const uint64_t end = begin + OPEN_CHUNK < n ? begin + OPEN_CHUNK : n;
  Fr acc = fp_zero<FrParams>();
  for (uint64_t j = end; j-- > begin;) acc = fp_add<FrParams>(fp_mul<FrParams>(acc, x), fp_load<FrParams>(p + 2 * j));
  h[c] = acc;
}
// carry[c] = sum_{c' > c} h[c'] * xL^(c' - c - 1) over the `n` level-2 groups, by one block: every thread owns a run of
// consecutive groups (local Horner value), a Hillis-Steele suffix scan with multipliers X^(2^k), X = xL^run, links the
// runs in log2(256) steps, and every thread re-walks its run with the carry entering from the right.  All runs but the
// last non-empty one are full, and that one is only ever multiplied by powers belonging to the full runs to its left.
// (Was a single thread walking all n/4096 groups: 0.7 ms at 2^23 coefficients.)
__global__ void __launch_bounds__(256) open_carry_scan(const Fr* h, uint64_t n, const Fr* xLp, Fr* carry) {
  __shared__ Fr s_v[256];
  const Fr xL = *xLp;
  const int t = threadIdx.x;
  const uint64_t per = (n + 255) / 256, begin = (uint64_t)t * per < n ? (uint64_t)t * per : n;
  const uint64_t end = begin + per < n ? begin + per : n;
  Fr v = fp_zero<FrParams>();
  for (uint64_t c = end; c-- > begin;) v = fp_add<FrParams>(fp_mul<FrParams>(v, xL), h[c]);
  Fr pw = fp_one<FrParams>();  // xL^per
  for (int bit = 63 - __clzll(per | 1); bit >= 0; bit--) {
    pw = fp_sqr<FrParams>(pw);
    if ((per >> bit) & 1) pw = fp_mul<FrParams>(pw, xL);
  }
  s_v[t] = v;
  for (int d = 1; d < 256; d <<= 1) {
    __syncthreads();
    const Fr right = t + d < 256 ? s_v[t + d] : fp_zero<FrParams>();
    __syncthreads();
    v = fp_add<FrParams>(v, fp_mul<FrParams>(pw, right));
    s_v[t] = v;
    pw = fp_sqr<FrParams>(pw);
  }
  __syncthreads();
  Fr acc = t + 1 < 256 ? s_v[t + 1] : fp_zero<FrParams>();
  for (uint64_t c = end; c-- > begin;) {
    carry[c] = acc;
    acc = fp_add<FrParams>(fp_mul<FrParams>(acc, xL), h[c]);
  }
}
__global__ void __launch_bounds__(256) open_carry_level(const Fr* h, uint64_t nchunks, const Fr* xLp, int group,
                                                       Fr* group_h) {
  const Fr xL = *xLp;
  // level-2 local values over groups of `group` chunks
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t begin = g * group;
  if (begin >= nchunks) return;
  const uint64_t end = begin + group < nchunks ? begin + group : nchunks;
  Fr acc = fp_zero<FrParams>();
  for (uint64_t c = end; c-- > begin;) acc = fp_add<FrParams>(fp_mul<FrParams>(acc, xL), h[c]);
  group_h[g] = acc;
}
__global__ void __launch_bounds__(256) open_carry_expand(const Fr* h, uint64_t nchunks, const Fr* xLp, int group,
                                                        const Fr* group_carry, Fr* carry) {
  const Fr xL = *xLp;
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t begin = g * group;
  if (begin >= nchunks) return;
  const uint64_t end = begin + group < nchunks ? begin + group : nchunks;
  Fr acc = group_carry[g];
  for (uint64_t c = end; c-- > begin;) {
    carry[c] = acc;
    acc = fp_add<FrParams>(fp_mul<FrParams>(acc, xL), h[c]);
  }
}
__global__ void __launch_bounds__(128) open_write(const uint4* p, uint64_t n, const Fr* xp, const Fr* carry, uint4* q,
                                                  Fr* y) {
  const Fr x = *xp;
  const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t begin = c * OPEN_CHUNK;
  if (begin >= n) return;
  const uint64_t end = begin + OPEN_CHUNK < n ? begin + OPEN_CHUNK : n;
  Fr acc = carry[c];  // = q_{end-1} (the value of the recurrence entering this chunk from the right)
  for (uint64_t j = end; j-- > begin;) {
    // invariant: acc = q_j (with q_{n-1} = 0);  q_{j-1} = p_j + x q_j
    acc = fp_add<FrParams>(fp_mul<FrParams>(acc, x), fp_load<FrParams>(p + 2 * j));
    if (j > 0) fp_store<FrParams>(q + 2 * (j - 1), acc);
    else *y = acc;  // the remainder of the division = p(x)
  }
}
__global__ void fr_pow_small(const Fr* xp, uint32_t e, Fr* out) {
  const Fr x = *xp;
  Fr acc = fp_one<FrParams>();
  for (int bit = 31; bit >= 0; bit--) {
    acc = fp_sqr<FrParams>(acc);
    if ((e >> bit) & 1) acc = fp_mul<FrParams>(acc, x);
  }
  *out = acc;
}

}  // namespace qz

using namespace qz;

namespace qz {

// cost model (in field multiplications): n*W mixed adds (10) + the bucket reduction, 2 full adds (14) per bucket, which
// is latency-bound and therefore weighted x4
static double msm_cost(size_t n, int c, bool collapsed) {
  const int W = (256 + c - 1) / c;
  const double buckets = (double)(1ull << (c - 1)) * (collapsed ? 1 : W);
  // weights fitted on B200 at 2^20..2^24: per-window reductions are short dependent chains (x4), the single large
  // reduction of the collapsed layout fills the machine better (x2; measured optimum c = 22 at 2^24)
  return (double)n * W * 10.0 + buckets * 2.0 * 14.0 * (collapsed ? 2.0 : 4.0);
}
static int pick_window(size_t n) {
  int best = 4;
  for (int c = 4; c <= 16; c++)
    if (msm_cost(n, c, false) < msm_cost(n, best, false)) best = c;
  return best;
}
int pick_precompute_window(size_t n) {
  int best = 8;
  for (int c = 8; c <= 24; c++)
    if (msm_cost(n, c, true) < msm_cost(n, best, true)) best = c;
  return best;
}

// Segments of a streamed MSM.  The points are cut into S index ranges; the prep stream copies (host scalars), digit-
// extracts and sorts range s+1 while the main stream accumulates range s into its own copy of the bucket sets, so the
// PCIe copy and the HBM-bound sort hide behind the integer-bound accumulation.  Ranges grow geometrically (the first
// one is what stays exposed); the copies are added bucket by bucket before the reduction (msm_bucket_merge).
// QZ_MSM_SEGMENTS / QZ_MSM_SEGMENTS_DEV = comma-separated weights override the defaults for host / device scalars.
static int segment_weights(bool host_scalars, size_t n, double* w) {
  const char* env = getenv(host_scalars ? "QZ_MSM_SEGMENTS" : "QZ_MSM_SEGMENTS_DEV");
  if (env && *env) {
    int S = 0;
    const char* q = env;
    while (*q && S < qz_ctx::MAX_SEGMENTS) {
      char* e = nullptr;
      const double v = strtod(q, &e);
      if (e == q) break;
      if (v > 0) w[S++] = v;
      q = *e ? e + 1 : e;
    }
    if (S) return S;
  }
  if (host_scalars && n >= ((size_t)1 << 19)) {
    w[0] = 1, w[1] = 3, w[2] = 9;  // measured at 2^24 on B200: 47.4 ms unsegmented -> 40.0 ms (device-resident: 37.7)
    return 3;
  }
  w[0] = 1;
  return 1;
}

// Every choice of one MSM, made on the host before anything is allocated or enqueued.
struct MsmPlan {
  int c, Wd, W;             // window bits, digits per scalar, bucket sets (1 when collapsed)
  bool collapsed;           // all windows share one bucket set through the precomputed multiples srs->pre
  const uint8_t* bases;     // srs->pre when collapsed, else srs->bases
  uint64_t m;               // sorted entries: Wd per scalar
  int key_bits;             // bits the sort orders by: (segment, window, digit)
  uint32_t per_w, n_slots;  // buckets per set, buckets of one segment's W sets
  int pair_levels;
  int chunk_len;            // sorted entries per accumulate thread
  int S;                    // point ranges [seg_lo[s], seg_lo[s + 1]), each with its own copy of the bucket sets
  size_t seg_lo[qz_ctx::MAX_SEGMENTS + 1], max_seg;
  uint64_t chunk_base[qz_ctx::MAX_SEGMENTS + 1];  // range s accumulates chunks [chunk_base[s], chunk_base[s + 1])
  int seg;                  // buckets per bucket-reduce thread
  uint32_t red_threads, per_window_parts;
  // partial-run lists: level 0 has two slots per accumulate chunk, level k+1 two per PART_CHUNK slots of level k
  uint64_t n_part0, n_part1;
};

static int msm_plan(qz_ctx* ctx, const qz_srs* srs, size_t n, bool host_scalars, MsmPlan& p) {
  if (n >= ((size_t)1 << 31)) return ctx->fail(QZ_ERR_INVALID_ARG, "MSM size must be below 2^31");
  p.c = pick_window(n);
  p.collapsed = srs->pre && msm_cost(n, srs->pre_c, true) < msm_cost(n, p.c, false);
  if (p.collapsed) p.c = srs->pre_c;
  const int c = p.c;
  p.Wd = (256 + c - 1) / c;
  p.W = p.collapsed ? 1 : p.Wd;
  p.bases = p.collapsed ? srs->pre : srs->bases;
  p.m = (uint64_t)p.Wd * n;
  ctx->last_stat[0] = c;
  ctx->last_stat[1] = p.Wd;
  ctx->last_stat[2] = p.collapsed ? 1 : 0;
  ctx->last_stat[3] = (double)p.m;
  if (p.m >= ((uint64_t)1 << 32)) return ctx->fail(QZ_ERR_INVALID_ARG, "MSM too large for 32-bit positions");
  p.per_w = 1u << (c - 1);
  p.n_slots = (uint32_t)p.W * p.per_w;
  p.key_bits = c;
  while ((1u << (p.key_bits - c)) < (uint32_t)p.W) p.key_bits++;
  // pair levels ahead of the accumulation (QZ_MSM_PAIR_LEVELS = count; unset: none): values need bit 30 as the flag
  p.pair_levels = 0;
  const char* env = getenv("QZ_MSM_PAIR_LEVELS");
  if (env && *env) p.pair_levels = std::max(0, std::min(PAIR_MAX_LEVELS, atoi(env)));
  const uint64_t max_index = (p.collapsed ? (uint64_t)p.Wd * srs->n : (uint64_t)srs->n);
  if (p.m >= VAL_PAIR || max_index >= VAL_PAIR || p.m < 64) p.pair_levels = 0;
  // chunk length: at least ~16 chunks per resident accumulate thread, else the minimum.  The pair levels leave the
  // accumulation a list ~2^levels shorter: the chunks are sized for that list, so that enough of them fill the machine.
  p.chunk_len = (int)std::min<uint64_t>(ACC_CHUNK_MAX, (p.m >> p.pair_levels) / ((uint64_t)ctx->sm_count * 4 * ACC_THREADS * 16));
  p.chunk_len = std::max(ACC_CHUNK_MIN, p.chunk_len / 32 * 32);

  double weights[qz_ctx::MAX_SEGMENTS];
  const int S = segment_weights(host_scalars, n, weights);
  double total = 0, run = 0;
  for (int s = 0; s < S; s++) total += weights[s];
  p.S = 0;
  p.seg_lo[0] = 0;
  for (int s = 0; s < S; s++) {
    run += weights[s];
    size_t hi = s == S - 1 ? n : std::min(n, ((size_t)((double)n * run / total) + 255) & ~(size_t)255);
    if (hi > p.seg_lo[p.S]) p.seg_lo[++p.S] = hi;
  }
  if (((uint64_t)p.S * p.W) << c >= 0xffffffffull) {  // (segment, window, digit) must fit the 32-bit key below KEY_NONE
    p.S = 1;
    p.seg_lo[1] = n;
  }
  p.chunk_base[0] = 0;
  p.max_seg = 0;
  for (int s = 0; s < p.S; s++) {
    const uint64_t ms = (uint64_t)p.Wd * (p.seg_lo[s + 1] - p.seg_lo[s]);
    p.chunk_base[s + 1] = p.chunk_base[s] + (ms + p.chunk_len - 1) / p.chunk_len;
    p.max_seg = std::max(p.max_seg, p.seg_lo[s + 1] - p.seg_lo[s]);
  }
  p.n_part0 = 2 * p.chunk_base[p.S];
  p.n_part1 = 2 * ((p.n_part0 + PART_CHUNK - 1) / PART_CHUNK);
  // small problems are latency-bound: shorter running-sum segments (more threads, shorter dependent chains)
  // large bucket sets: one wave of threads (2^15 x 64 buckets at c = 22) beats two waves of shorter chains
  // (2^19 buckets, one rank's share of 2^24 points on 8 GPUs: 16K threads walking 32 buckets are latency-bound, 0.63 ms)
  const uint32_t n_slots = p.n_slots;
  const int seg_want = n_slots <= (1u << 17) ? 8 : n_slots <= (1u << 19) ? RED_SEG / 2 : n_slots >= (1u << 21) ? 2 * RED_SEG : RED_SEG;
  p.seg = p.per_w >= (uint32_t)seg_want ? seg_want : (int)p.per_w;
  p.red_threads = n_slots / p.seg;
  p.per_window_parts = p.per_w / p.seg;
  return QZ_OK;
}

// pair levels (msm_pair_*): scratch for the longest range, shared by the ranges (they run in turn on the main stream)
struct PairScratch {
  PairCtl* ctl;
  uint8_t *sums, *prefix, *codes;
  uint8_t *v[PAIR_TREE_MAX + 1], *pre[PAIR_TREE_MAX];  // inversion tree: elements / running products per depth
  unsigned long long *counts, *offs;
  void* scan_tmp;
  size_t scan_bytes;
};
struct MsmScratch {
  uint32_t *keys, *vals, *keys2, *vals2;  // the (key, value) list and the sort's second buffer
  uint8_t* buckets;                        // S copies of the bucket sets
  uint8_t *ppts_a, *ppts_b;                // partial-run lists (n_part0 / n_part1 slots) and their keys
  uint32_t *pkeys_a, *pkeys_b;
  uint8_t *fin_a, *fin_b;                  // msm_partials_finish's scan buffers
  uint8_t *partial, *partial2, *window_sums;
  void* sort_tmp;  // shared: the segments' sorts are serialised on the prep stream
  size_t sort_bytes;
  PairScratch pairs;                       // allocated only with pair levels
};

static int msm_scratch(qz_ctx* ctx, const MsmPlan& p, cudaStream_t ps, MsmScratch& sc) {
  bool ok = true;
  auto take = [&](size_t bytes) {
    void* q = ctx->arena_alloc(bytes);
    ok = ok && q;
    return q;
  };
  sc.keys = (uint32_t*)take(4 * p.m);
  sc.vals = (uint32_t*)take(4 * p.m);
  sc.keys2 = (uint32_t*)take(4 * p.m);
  sc.vals2 = (uint32_t*)take(4 * p.m);
  sc.buckets = (uint8_t*)take((size_t)p.S * p.n_slots * 128);
  sc.ppts_a = (uint8_t*)take(p.n_part0 * 128);
  sc.pkeys_a = (uint32_t*)take(p.n_part0 * 4);
  sc.ppts_b = (uint8_t*)take(p.n_part1 * 128);
  sc.pkeys_b = (uint32_t*)take(p.n_part1 * 4);
  sc.fin_a = (uint8_t*)take((size_t)FIN_SLOTS * 128);
  sc.fin_b = (uint8_t*)take((size_t)FIN_SLOTS * 128);
  sc.partial = (uint8_t*)take((size_t)p.red_threads * 128);
  sc.partial2 = (uint8_t*)take((size_t)p.W * ((p.per_window_parts + SUM_SPAN - 1) / SUM_SPAN) * 128);
  sc.window_sums = (uint8_t*)take((size_t)p.W * 128);
  cub::DoubleBuffer<uint32_t> dk(sc.keys, sc.keys2), dv(sc.vals, sc.vals2);
  cub::DeviceRadixSort::SortPairs(nullptr, sc.sort_bytes, dk, dv, (int64_t)((uint64_t)p.Wd * p.max_seg), 0, p.key_bits, ps);
  sc.sort_tmp = take(sc.sort_bytes);
  if (!ok) return ctx->fail(QZ_ERR_ALLOC, "MSM scratch");
  if (!p.pair_levels) return QZ_OK;

  PairScratch& pr = sc.pairs;
  const uint64_t mmax = (uint64_t)p.Wd * p.max_seg;
  const uint64_t tiles = (mmax + 2 * PAIR_TILE - 1) / (2 * PAIR_TILE);
  pr.ctl = (PairCtl*)take(sizeof(PairCtl));
  pr.sums = (uint8_t*)take(mmax * 64);
  pr.prefix = (uint8_t*)take(tiles * PAIR_TILE * 32);
  pr.codes = (uint8_t*)take(tiles * PAIR_TILE);
  uint64_t n = tiles * PAIR_THREADS;
  for (int k = 0; k <= PAIR_TREE_MAX; k++) {
    pr.v[k] = (uint8_t*)take(n * 32);
    if (n == 1) break;
    if (k == PAIR_TREE_MAX) {
      ok = false;
      break;
    }
    pr.pre[k] = (uint8_t*)take(n * 32);
    n = (n + PAIR_G - 1) / PAIR_G;
  }
  pr.counts = (unsigned long long*)take((tiles + 1) * 8);
  pr.offs = (unsigned long long*)take((tiles + 1) * 8);
  cub::DeviceScan::ExclusiveSum(nullptr, pr.scan_bytes, pr.counts, pr.offs, (int64_t)(tiles + 1), ctx->stream);
  pr.scan_tmp = take(pr.scan_bytes);
  if (!ok) return ctx->fail(QZ_ERR_ALLOC, "MSM pair-level scratch");
  return QZ_OK;
}

// On return dk / dv hold range s's sorted list in Current() and the sort's other buffer in Alternate().
static int prep_segment(qz_ctx* ctx, const qz_srs* srs, const MsmPlan& p, MsmScratch& sc, int s, cudaStream_t ps,
                        uint4* scalars_dev, const void* scalars_host, size_t first, cub::DoubleBuffer<uint32_t>& dk,
                        cub::DoubleBuffer<uint32_t>& dv) {
  QzRange nvtx("qz:msm:digits+sort");
  const size_t lo = p.seg_lo[s], ns = p.seg_lo[s + 1] - lo;
  const uint64_t off = (uint64_t)p.Wd * lo;
  if (scalars_host)
    QZ_CUDA(ctx, cudaMemcpyAsync(scalars_dev + 2 * lo, (const uint8_t*)scalars_host + 32 * lo, 32 * ns,
                                 cudaMemcpyHostToDevice, ps));
  QZ_LAUNCH_ON(ctx, ps, msm_digits, (unsigned)((ns + 255) / 256), 256, 0, scalars_dev + 2 * lo, (uint32_t)ns,
               (uint32_t)(first + lo), p.c, p.Wd, p.collapsed ? (uint32_t)srs->n : 0u, (uint32_t)(s * p.W), sc.keys + off,
               sc.vals + off, ctx->acc_ring_on ? ctx->acc_nonzero_dev : nullptr);
  dk = cub::DoubleBuffer<uint32_t>(sc.keys + off, sc.keys2 + off);
  dv = cub::DoubleBuffer<uint32_t>(sc.vals + off, sc.vals2 + off);
  QZ_CUDA(ctx, cub::DeviceRadixSort::SortPairs(sc.sort_tmp, sc.sort_bytes, dk, dv, (int64_t)((uint64_t)p.Wd * ns), 0,
                                               p.key_bits, ps));
  ctx->launches += 2 + (p.key_bits + 7) / 8;  // CUB: histogram + one onesweep pass per 8 key bits (approximate)
  if (p.S > 1) {
    QZ_CUDA(ctx, cudaEventRecord(ctx->ev_seg_ready[s], ps));
    QZ_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_seg_ready[s], 0));
  }
  return QZ_OK;
}

// Each level reads dk / dv's Current() buffers and writes their Alternate() ones, which then become Current().
static int pair_levels(qz_ctx* ctx, const MsmPlan& p, PairScratch& pr, uint64_t ms, cub::DoubleBuffer<uint32_t>& dk,
                       cub::DoubleBuffer<uint32_t>& dv) {
  const uint64_t tiles = (ms + 2 * PAIR_TILE - 1) / (2 * PAIR_TILE);  // of a level over the longest list possible
  uint64_t tree_n[PAIR_TREE_MAX + 1];  // elements per depth over the longest list possible, down to ONE root
  int tree_depth = 0;
  tree_n[0] = tiles * PAIR_THREADS;
  while (tree_n[tree_depth] > 1) {
    tree_n[tree_depth + 1] = (tree_n[tree_depth] + PAIR_G - 1) / PAIR_G;
    tree_depth++;
  }
  const uint32_t dmask = (1u << p.c) - 1;
  QZ_LAUNCH(ctx, msm_pair_init, 1, 1, 0, pr.ctl, ms, pr.counts + tiles);
  for (int l = 0; l < p.pair_levels; l++) {
    QZ_LAUNCH(ctx, msm_pair_scan, (unsigned)tiles, PAIR_THREADS, 0, dk.Current(), dv.Current(), pr.ctl, l, dmask, p.bases,
              pr.sums, pr.prefix, pr.v[0], pr.codes, pr.counts);
    QZ_CUDA(ctx, cub::DeviceScan::ExclusiveSum(pr.scan_tmp, pr.scan_bytes, pr.counts, pr.offs, (int64_t)(tiles + 1),
                                               ctx->stream));
    ctx->launches += 2;
    for (int k = 0; k < tree_depth; k++)
      QZ_LAUNCH(ctx, msm_pair_tree_up, (unsigned)((tree_n[k + 1] + 127) / 128), 128, 0, pr.ctl, l, k, pr.v[k], pr.pre[k],
                pr.v[k + 1]);
    QZ_LAUNCH(ctx, msm_pair_tree_root, 1, 1, 0, pr.ctl, l, pr.v[tree_depth]);
    for (int k = tree_depth - 1; k >= 0; k--)
      QZ_LAUNCH(ctx, msm_pair_tree_down, (unsigned)((tree_n[k + 1] + 127) / 128), 128, 0, pr.ctl, l, k, pr.v[k], pr.pre[k],
                pr.v[k + 1]);
    QZ_LAUNCH(ctx, msm_pair_apply, (unsigned)tiles, PAIR_THREADS, 0, dk.Current(), dv.Current(), pr.ctl, l, dmask, p.bases,
              pr.sums, pr.prefix, pr.v[0], pr.codes, pr.offs, (uint32_t)tiles, dk.Alternate(), dv.Alternate());
    dk.selector ^= 1;
    dv.selector ^= 1;
  }
  return QZ_OK;
}

// Merge the partial runs level by level until one chunk holds them all (one list: the segments' keys ascend).
static int reduce_partial_runs(qz_ctx* ctx, const MsmPlan& p, const MsmScratch& sc) {
  QzRange nvtx("qz:msm:partial-runs");
  uint32_t *kin = sc.pkeys_a, *kout = sc.pkeys_b;
  uint8_t *pin = sc.ppts_a, *pout = sc.ppts_b;
  uint64_t n_in = p.n_part0;
  while (true) {
    if (n_in <= (uint64_t)FIN_SLOTS && n_in > PART_CHUNK) {  // short list: scan it in one launch
      QZ_LAUNCH(ctx, msm_partials_finish, 1, FIN_THREADS, 0, kin, pin, (int)n_in, p.c, sc.buckets, sc.fin_a, sc.fin_b);
      return QZ_OK;
    }
    const uint64_t chunks = (n_in + PART_CHUNK - 1) / PART_CHUNK;
    const int last_level = chunks == 1;
    QZ_LAUNCH(ctx, msm_partials_reduce, (unsigned)((chunks + 127) / 128), 128, 0, kin, pin, n_in, p.c, sc.buckets, kout, pout,
              last_level);
    if (last_level) return QZ_OK;
    n_in = 2 * chunks;
    // the output of this level (<= n_part1 slots) becomes the input; the other buffer is large enough
    std::swap(kin, kout);
    std::swap(pin, pout);
  }
}

static int reduce_and_combine(qz_ctx* ctx, const MsmPlan& p, const MsmScratch& sc, uint8_t* out_xyzz_dev,
                              uint8_t* out_affine_dev) {
  QzRange nvtx("qz:msm:bucket-reduce+combine");
  if (p.S > 1) QZ_LAUNCH(ctx, msm_bucket_merge, (p.n_slots + 127) / 128, 128, 0, sc.buckets, p.n_slots, p.S);
  QZ_LAUNCH(ctx, msm_bucket_reduce, (p.red_threads + 127) / 128, 128, 0, sc.buckets, p.c, p.W, p.seg, sc.partial);
  uint8_t *in = sc.partial, *out = sc.partial2;  // per window: per_window_parts partial sums -> 1
  uint32_t per_in = p.per_window_parts;
  while (per_in > SUM_SPAN) {
    const uint32_t per_out = (per_in + SUM_SPAN - 1) / SUM_SPAN;
    QZ_LAUNCH(ctx, msm_block_sum, (unsigned)p.W * per_out, 128, 0, in, per_in, per_out, out);
    std::swap(in, out);
    per_in = per_out;
  }
  QZ_LAUNCH(ctx, msm_block_sum, (unsigned)p.W, 128, 0, in, per_in, 1u, sc.window_sums);
  QZ_LAUNCH(ctx, msm_combine, 1, 1, 0, sc.window_sums, p.c, p.W, out_xyzz_dev, out_affine_dev);
  return QZ_OK;
}

// `srs` supplies the bases and, when present and cheaper by the cost model, the precomputed window multiples.  Everything
// is ordered on ctx->stream when the call returns (the prep stream is joined before the last accumulation).
int msm_run(qz_ctx* ctx, const qz_srs* srs, uint4* scalars_dev, const void* scalars_host, size_t n,
            uint8_t* out_xyzz_dev, uint8_t* out_affine_dev, size_t first) {
  cudaStream_t st = ctx->stream;
  QzRange nvtx_call("qz:msm");
  ctx->acc_launches = 0;
  if (n == 0) {  // empty sum = identity (reachable: commit(&[]) for the quotient of a constant, mlpcs.rs:321-393)
    if (out_xyzz_dev) QZ_CUDA(ctx, cudaMemsetAsync(out_xyzz_dev, 0, 128, st));
    if (out_affine_dev) QZ_CUDA(ctx, cudaMemsetAsync(out_affine_dev, 0, 64, st));
    return QZ_OK;
  }
  MsmPlan p;
  int rc = msm_plan(ctx, srs, n, scalars_host != nullptr, p);
  if (rc) return rc;
  if (p.S > 1 && ctx->ensure_prep_stream()) return ctx->fail(QZ_ERR_CUDA, "prep stream");
  cudaStream_t ps = p.S > 1 ? ctx->prep_stream : st;
  auto mark = ctx->arena_mark();
  MsmScratch sc{};
  rc = msm_scratch(ctx, p, ps, sc);
  if (rc) return rc;

  if (p.S > 1) {  // the prep stream starts where the main stream stands (earlier users of the scratch, the scalars)
    QZ_CUDA(ctx, cudaEventRecord(ctx->ev_entry, st));
    QZ_CUDA(ctx, cudaStreamWaitEvent(ps, ctx->ev_entry, 0));
  }
  QZ_CUDA(ctx, cudaMemsetAsync(sc.buckets, 0, (size_t)p.S * p.n_slots * 128, st));
  const auto accumulate = p.pair_levels ? msm_accumulate<true> : msm_accumulate<false>;
  for (int s = 0; s < p.S; s++) {
    cub::DoubleBuffer<uint32_t> dk, dv;
    rc = prep_segment(ctx, srs, p, sc, s, ps, scalars_dev, scalars_host, first, dk, dv);
    if (rc) return rc;
    QzRange nvtx_acc("qz:msm:accumulate");
    const uint64_t ms = (uint64_t)p.Wd * (p.seg_lo[s + 1] - p.seg_lo[s]), chunks = p.chunk_base[s + 1] - p.chunk_base[s];
    cudaEvent_t ring0 = nullptr, ring1 = nullptr;
    const bool ring = ctx->acc_ring_next(&ring0, &ring1) == 0;
    if (ring) QZ_CUDA(ctx, cudaEventRecord(ring0, st));
    QZ_CUDA(ctx, cudaEventRecord(p.S > 1 ? ctx->ev_acc0[s] : ctx->ev_k0, st));
    rc = p.pair_levels ? pair_levels(ctx, p, sc.pairs, ms, dk, dv) : QZ_OK;
    if (rc) return rc;
    QZ_LAUNCH(ctx, accumulate, (unsigned)((chunks + ACC_THREADS - 1) / ACC_THREADS), ACC_THREADS, 0, dk.Current(),
              dv.Current(), p.pair_levels ? 0 : ms, p.pair_levels ? &sc.pairs.ctl->m[p.pair_levels] : nullptr, chunks,
              p.chunk_len, p.bases, sc.pairs.sums, p.c, sc.buckets, sc.ppts_a + p.chunk_base[s] * 256,
              sc.pkeys_a + 2 * p.chunk_base[s]);
    QZ_CUDA(ctx, cudaEventRecord(p.S > 1 ? ctx->ev_acc1[s] : ctx->ev_k1, st));
    if (ring) {
      QZ_CUDA(ctx, cudaEventRecord(ring1, st));
      ctx->acc_ring_adds += (double)ms;  // sorted entries; the additions executed are counted by msm_digits
    }
  }
  ctx->acc_launches = p.S > 1 ? p.S : 0;
  rc = reduce_partial_runs(ctx, p, sc);
  if (rc) return rc;
  rc = reduce_and_combine(ctx, p, sc, out_xyzz_dev, out_affine_dev);
  if (rc) return rc;
  ctx->arena_release(mark);  // stream order keeps the scratch valid for the kernels enqueued above
  return QZ_OK;
}

int msm_device(qz_ctx* ctx, const qz_srs* srs, const uint4* scalars_dev, size_t n, uint8_t* out_xyzz_dev,
               uint8_t* out_affine_dev) {
  return msm_run(ctx, srs, const_cast<uint4*>(scalars_dev), nullptr, n, out_xyzz_dev, out_affine_dev);
}

// KZG::open (kzg.rs:75-96) with everything on the device: x is read from device memory, y (32 B) and the affine proof
// (64 B) are written to device memory.  Asynchronous on ctx->stream; scratch is released on return (stream order keeps
// it valid for the kernels already enqueued).
int kzg_open_device(qz_ctx* ctx, const qz_srs* srs, const uint4* pdev, size_t n_coeffs, const Fr* x_dev,
                    Fr* y_dev, uint8_t* proof_affine_dev) {
  cudaStream_t st = ctx->stream;
  if (n_coeffs == 0) {  // zero polynomial: y = 0, quotient = 0, proof = identity
    QZ_CUDA(ctx, cudaMemsetAsync(y_dev, 0, 32, st));
    QZ_CUDA(ctx, cudaMemsetAsync(proof_affine_dev, 0, 64, st));
    return QZ_OK;
  }
  QzRange nvtx_call("qz:kzg_open");
  auto mark = ctx->arena_mark();
  const uint64_t n = n_coeffs, nchunks = (n + OPEN_CHUNK - 1) / OPEN_CHUNK;
  const int group = 64;
  const uint64_t ngroups = (nchunks + group - 1) / group;
  Fr* h = (Fr*)ctx->arena_alloc(32 * nchunks);
  Fr* carry = (Fr*)ctx->arena_alloc(32 * nchunks);
  Fr* gh = (Fr*)ctx->arena_alloc(32 * ngroups);
  Fr* gcarry = (Fr*)ctx->arena_alloc(32 * ngroups);
  Fr* pw = (Fr*)ctx->arena_alloc(64);
  uint4* q = (uint4*)ctx->arena_alloc(32 * std::max<uint64_t>(1, n - 1));
  if (!h || !carry || !gh || !gcarry || !pw || !q) return ctx->fail(QZ_ERR_ALLOC, "open scratch");
  QZ_LAUNCH(ctx, fr_pow_small, 1, 1, 0, x_dev, (uint32_t)OPEN_CHUNK, pw);
  QZ_LAUNCH(ctx, fr_pow_small, 1, 1, 0, x_dev, (uint32_t)(OPEN_CHUNK * group), pw + 1);
  QZ_LAUNCH(ctx, open_local, (unsigned)((nchunks + 127) / 128), 128, 0, pdev, n, x_dev, h);
  QZ_LAUNCH(ctx, open_carry_level, (unsigned)((ngroups + 255) / 256), 256, 0, h, nchunks, pw, group, gh);
  QZ_LAUNCH(ctx, open_carry_scan, 1, 256, 0, gh, ngroups, pw + 1, gcarry);
  QZ_LAUNCH(ctx, open_carry_expand, (unsigned)((ngroups + 255) / 256), 256, 0, h, nchunks, pw, group, gcarry, carry);
  QZ_LAUNCH(ctx, open_write, (unsigned)((nchunks + 127) / 128), 128, 0, pdev, n, x_dev, carry, q, y_dev);
  // commit(q): trailing zero coefficients contribute nothing, so trimming (DensePolynomial) is value-neutral
  const size_t qn = std::min<size_t>(n - 1, srs->n);
  int rc = msm_device(ctx, srs, q, qn, nullptr, proof_affine_dev);
  ctx->arena_release(mark);
  return rc;
}

int msm_sum_points_launch(qz_ctx* ctx, const uint8_t* pts_dev, int n, uint8_t* out_affine_dev) {
  QZ_LAUNCH(ctx, msm_sum_points, 1, 1, 0, pts_dev, n, out_affine_dev);
  return QZ_OK;
}

int msm_call(qz_ctx* ctx, const qz_srs* srs, const void* scalars, size_t n_scalars, int on_device, MsmMode mode,
             uint8_t out_xy[64]) {
  if (!ctx || !srs || !out_xy || (n_scalars && !scalars)) return QZ_ERR_INVALID_ARG;
  if (mode == MsmMode::split && n_scalars > srs->n) return ctx->fail(QZ_ERR_DEGREE, "Polynomial degree exceeds max degree");
  QZ_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->arena_reset();
  const int G = ctx->nranks > 0 ? ctx->nranks : 1;
  size_t lo = 0, n = std::min(n_scalars, srs->n);  // msm_unchecked zips to the shorter slice
  if (mode == MsmMode::split) {
    lo = n_scalars * (size_t)ctx->rank / G;
    n = n_scalars * ((size_t)ctx->rank + 1) / G - lo;
  }
  cudaStream_t st = ctx->stream;
  QZ_CUDA(ctx, cudaEventRecord(ctx->ev_call0, st));
  QZ_CUDA(ctx, cudaEventRecord(ctx->ev_k0, st));
  QZ_CUDA(ctx, cudaEventRecord(ctx->ev_k1, st));
  uint4* sdev = on_device ? (uint4*)scalars + 2 * lo : nullptr;
  const void* shost = nullptr;
  if (!on_device && n) {  // the copy is issued range by range inside msm_run, overlapped with the accumulation
    sdev = (uint4*)ctx->arena_alloc(32 * n);
    if (!sdev) return ctx->fail(QZ_ERR_ALLOC, "scalars");
    shost = (const uint8_t*)scalars + 32 * lo;
  }
  const bool exchange = mode != MsmMode::local;  // this rank's XYZZ partial sum `mine`, added to the other ranks' ones
  uint8_t* mine = exchange ? (uint8_t*)ctx->arena_alloc(128) : nullptr;
  uint8_t* all = exchange ? (uint8_t*)ctx->arena_alloc((size_t)128 * G) : nullptr;
  uint8_t* out_dev = (uint8_t*)ctx->arena_alloc(64);
  if ((exchange && (!mine || !all)) || !out_dev) return ctx->fail(QZ_ERR_ALLOC, "result");
  int rc = msm_run(ctx, srs, sdev, shost, n, mine, exchange ? nullptr : out_dev, lo);
  uint32_t* fault = nullptr;
  if (!rc && exchange) rc = msm_exchange_sum(ctx, mine, all, out_dev, &fault);
  if (rc) return rc;
  QZ_CUDA(ctx, cudaMemcpyAsync(out_xy, out_dev, 64, cudaMemcpyDeviceToHost, st));
  QZ_CUDA(ctx, cudaEventRecord(ctx->ev_call1, st));
  QZ_CUDA(ctx, cudaStreamSynchronize(st));
  if (fault && *fault) return ctx->fail(QZ_ERR_NCCL, "a peer did not deliver its partial sum (peer mailbox wait timed out)");
  cudaEventElapsedTime(&ctx->last_ms[0], ctx->ev_call0, ctx->ev_call1);
  float acc = 0.f;  // the msm_accumulate launches: between ev_k0 and ev_k1, or one event pair per range
  if (ctx->acc_launches == 0) cudaEventElapsedTime(&acc, ctx->ev_k0, ctx->ev_k1);
  for (int s = 0; s < ctx->acc_launches; s++) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev_acc0[s], ctx->ev_acc1[s]);
    acc += ms;
  }
  ctx->last_ms[1] = acc;
  return QZ_OK;
}

}  // namespace qz

extern "C" {

int qz_srs_upload(qz_ctx* ctx, const uint8_t* xy, size_t n, qz_srs** out) {
  if (!ctx || !out || (n && !xy)) return QZ_ERR_INVALID_ARG;
  QZ_CUDA(ctx, cudaSetDevice(ctx->device));
  qz_srs* s = new (std::nothrow) qz_srs{ctx, nullptr, n, nullptr, 0, 0};
  if (!s) return ctx->fail(QZ_ERR_ALLOC, "srs handle");
  cudaError_t e = cudaMalloc((void**)&s->bases, n ? n * 64 : 64);
  if (e != cudaSuccess) {
    delete s;
    return ctx->fail(QZ_ERR_ALLOC, "cudaMalloc(srs)", e);
  }
  if (n) {
    e = cudaMemcpyAsync(s->bases, xy, n * 64, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
      cudaFree(s->bases);
      delete s;
      return ctx->fail(QZ_ERR_CUDA, "srs upload", e);
    }
  }
  *out = s;
  return QZ_OK;
}

int qz_srs_generate(qz_ctx* ctx, const uint8_t g_xy[64], const uint8_t tau[32], size_t n, qz_srs** out) {
  if (!ctx || !out || !g_xy || !tau) return QZ_ERR_INVALID_ARG;
  QZ_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->arena_reset();
  qz_srs* s = new (std::nothrow) qz_srs{ctx, nullptr, n, nullptr, 0, 0};
  if (!s) return ctx->fail(QZ_ERR_ALLOC, "srs handle");
  cudaError_t e = cudaMalloc((void**)&s->bases, n ? n * 64 : 64);
  if (e != cudaSuccess) {
    delete s;
    return ctx->fail(QZ_ERR_ALLOC, "cudaMalloc(srs)", e);
  }
  uint8_t* pow_bases = (uint8_t*)ctx->arena_alloc(32 * 64);
  uint8_t* table = (uint8_t*)ctx->arena_alloc((size_t)32 * 255 * 64);
  if (!pow_bases || !table) {
    cudaFree(s->bases);
    delete s;
    return ctx->fail(QZ_ERR_ALLOC, "srs table");
  }
  Affine g;
  memcpy(g.x.v, g_xy, 32);
  memcpy(g.y.v, g_xy + 32, 32);
  Fr t;
  memcpy(t.v, tau, 32);
  *out = s;  // handed to the caller even on a later launch error so it can be freed
  QZ_LAUNCH(ctx, srs_table_bases, 1, 32, 0, g, pow_bases);
  QZ_LAUNCH(ctx, srs_table_fill, (32 * 255 + 127) / 128, 128, 0, pow_bases, table);
  if (n) {
    uint64_t threads = (n + SRS_CHUNK - 1) / SRS_CHUNK;
    QZ_LAUNCH(ctx, srs_generate, (unsigned)((threads + 127) / 128), 128, 0, table, t, (uint64_t)n, s->bases);
  }
  QZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return QZ_OK;
}

int qz_srs_precompute(qz_ctx* ctx, qz_srs* s, int window_bits) {
  if (!ctx || !s || window_bits < 0 || window_bits > 24 || (window_bits && window_bits < 4)) return QZ_ERR_INVALID_ARG;
  if (s->n == 0) return QZ_OK;
  QZ_CUDA(ctx, cudaSetDevice(ctx->device));
  const int c = window_bits ? window_bits : pick_precompute_window(s->n);
  const int W = (256 + c - 1) / c;
  if ((uint64_t)W * s->n >= ((uint64_t)1 << 31)) return ctx->fail(QZ_ERR_INVALID_ARG, "precomputed table index exceeds 31 bits");
  if (s->pre) {
    cudaFree(s->pre);
    s->pre = nullptr;
  }
  cudaError_t e = cudaMalloc((void**)&s->pre, (size_t)W * s->n * 64);
  if (e != cudaSuccess) {
    s->pre = nullptr;
    return ctx->fail(QZ_ERR_ALLOC, "precomputed window multiples", e);
  }
  s->pre_c = c;
  s->pre_W = W;
  QZ_LAUNCH(ctx, srs_precompute, (unsigned)((s->n + 127) / 128), 128, 0, s->bases, (uint64_t)s->n, c, W, s->pre);
  QZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return QZ_OK;
}

void qz_srs_free(qz_srs* s) {
  if (!s) return;
  cudaSetDevice(s->ctx->device);
  cudaFree(s->bases);
  if (s->pre) cudaFree(s->pre);
  delete s;
}
size_t qz_srs_len(const qz_srs* s) { return s ? s->n : 0; }

int qz_srs_download(qz_ctx* ctx, const qz_srs* s, size_t first, size_t count, uint8_t* out_xy) {
  if (!ctx || !s || !out_xy || first + count > s->n) return QZ_ERR_INVALID_ARG;
  if (!count) return QZ_OK;
  QZ_CUDA(ctx, cudaMemcpyAsync(out_xy, s->bases + first * 64, count * 64, cudaMemcpyDeviceToHost, ctx->stream));
  QZ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return QZ_OK;
}

int qz_msm(qz_ctx* ctx, const qz_srs* srs, const void* scalars, size_t n_scalars, int on_device, uint8_t out_xy[64]) {
  return msm_call(ctx, srs, scalars, n_scalars, on_device, MsmMode::local, out_xy);
}

int qz_kzg_commit(qz_ctx* ctx, const qz_srs* srs, const void* coeffs, size_t n_coeffs, int on_device,
                  uint8_t out_xy[64]) {
  if (!ctx || !srs) return QZ_ERR_INVALID_ARG;
  if (n_coeffs > srs->n) return ctx->fail(QZ_ERR_DEGREE, "Polynomial degree exceeds max degree");  // kzg.rs:62-65
  return qz_msm(ctx, srs, coeffs, n_coeffs, on_device, out_xy);
}

int qz_kzg_open(qz_ctx* ctx, const qz_srs* srs, const void* coeffs, size_t n_coeffs, int on_device, const uint8_t x[32],
                uint8_t out_y[32], uint8_t out_proof_xy[64]) {
  if (!ctx || !srs || !x || !out_y || !out_proof_xy || (n_coeffs && !coeffs)) return QZ_ERR_INVALID_ARG;
  // the quotient has n_coeffs - 1 coefficients; commit() asserts it fits the SRS (kzg.rs:62-65 via :89)
  if (n_coeffs > srs->n + 1) return ctx->fail(QZ_ERR_DEGREE, "Polynomial degree exceeds max degree");
  QZ_CUDA(ctx, cudaSetDevice(ctx->device));
  ctx->arena_reset();
  cudaStream_t st = ctx->stream;
  QZ_CUDA(ctx, cudaEventRecord(ctx->ev_call0, st));
  QZ_CUDA(ctx, cudaEventRecord(ctx->ev_k0, st));
  QZ_CUDA(ctx, cudaEventRecord(ctx->ev_k1, st));
  uint8_t* res = (uint8_t*)ctx->arena_alloc(192);  // y (32) ‖ x (32) ‖ proof (64)
  if (!res) return ctx->fail(QZ_ERR_ALLOC, "result");
  QZ_CUDA(ctx, cudaMemsetAsync(res, 0, 192, st));
  QZ_CUDA(ctx, cudaMemcpyAsync(res + 32, x, 32, cudaMemcpyHostToDevice, st));
  const uint4* pdev = (const uint4*)coeffs;
  if (!on_device && n_coeffs) {
    void* p = ctx->arena_alloc(32 * n_coeffs);
    if (!p) return ctx->fail(QZ_ERR_ALLOC, "coeffs");
    QZ_CUDA(ctx, cudaMemcpyAsync(p, coeffs, 32 * n_coeffs, cudaMemcpyHostToDevice, st));
    pdev = (const uint4*)p;
  }
  int rc = kzg_open_device(ctx, srs, pdev, n_coeffs, (const Fr*)(res + 32), (Fr*)res, res + 64);
  if (rc) return rc;
  uint8_t* pin = (uint8_t*)ctx->pinned_buf(192);
  if (!pin) return ctx->fail(QZ_ERR_ALLOC, "pinned");
  QZ_CUDA(ctx, cudaMemcpyAsync(pin, res, 192, cudaMemcpyDeviceToHost, st));
  QZ_CUDA(ctx, cudaEventRecord(ctx->ev_call1, st));
  QZ_CUDA(ctx, cudaStreamSynchronize(st));
  memcpy(out_y, pin, 32);
  memcpy(out_proof_xy, pin + 64, 64);
  cudaEventElapsedTime(&ctx->last_ms[0], ctx->ev_call0, ctx->ev_call1);
  cudaEventElapsedTime(&ctx->last_ms[1], ctx->ev_k0, ctx->ev_k1);
  return QZ_OK;
}

}  // extern "C"
