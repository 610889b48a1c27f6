// Fused codebook match on tcgen05 (AAE_PREC_TC_SPLIT): ONE kernel does
//     zq = z * rsqrt(max(sum z^2, 1e-12))          (tf.nn.l2_normalize,  auto_pose/ae/codebook.py:27)
//     cos = zq . E^T                                (tf.matmul,           codebook.py:50)
//     idx = argmax(cos), lowest index on ties       (np.argmax,           codebook.py:63-68)
// and never materialises the [B, N] cosine matrix.
//
// Layout: TMEM lanes = queries (M = 128 per block, up to two blocks for B <= 256), TMEM columns = codebook rows (128 per
// tile), so the arg-max over rows is a per-thread scan of its own lane -- no cross-thread reduction.
// The normalised queries are split into fp16 (hi, lo) in the kernel prologue and stay resident IN TENSOR MEMORY as the
// MMA's A operand (tcgen05.mma with A from TMEM), which leaves all of shared memory to the codebook: pre-split into
// (hi, lo) fp16 at create time -- the same 512 bytes per row as the fp32 table -- it streams through a 3-stage x 64 KB TMA
// ring, each row read from HBM exactly once.  Per (tile, query block) the issuer thread fires  hi*hi + hi*lo + lo*hi  into
// one fp32 accumulator (both operands pre-scaled by 64 so every lo term is a normal fp16; the 2^-12 unscale in the epilogue
// is exact).  Two accumulator stages alternate, so the epilogue scan of one block overlaps the MMAs of the next.  Per-CTA winners are merged with one 64-bit atomicMax per query on a
// (score, ~index) key -- max is order-independent, so the result is deterministic -- and the last CTA to finish writes
// the [B] score / index outputs and re-arms the scratch for the next launch (steady state: a single launch, no memset).
#include <stdlib.h>

#include "tc.cuh"
#include "tc_common.cuh"

namespace aae {

using namespace tc;

namespace {

constexpr int MT_ROWS = 128;                // codebook rows per tile (= MMA N)
constexpr int MT_STAGES = 3;
constexpr int MT_E_BYTES = MT_ROWS * 128;   // one K-half of one (hi|lo) array: 128 rows x 128 B
constexpr int MT_STAGE_BYTES = 4 * MT_E_BYTES;  // hi k0, hi k1, lo k0, lo k1  = 64 KB
constexpr float MT_SCALE = 64.f;
constexpr int MT_SMEM_TOTAL = MT_STAGES * MT_STAGE_BYTES + 1024 + 256;
// TMEM columns: per 128-query block mq: [mq*128, +64) Q_hi, [mq*128+64, +64) Q_lo  (fp16 pairs, K = 128 -> 64 columns);
// accumulators: two stages of 128 fp32 columns at 256 and 384.
constexpr int MT_TMEM_ACC0 = 256;

__device__ __forceinline__ unsigned long long pack_best(float s, int idx) {
  uint32_t b = __float_as_uint(s);
  b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return ((unsigned long long)b << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)idx);
}
__device__ __forceinline__ void unpack_best(unsigned long long k, float& s, int& idx) {
  uint32_t b = (uint32_t)(k >> 32);
  b = (b & 0x80000000u) ? (b & 0x7FFFFFFFu) : ~b;
  s = __uint_as_float(b);
  idx = (int)(0xFFFFFFFFu - (uint32_t)(k & 0xFFFFFFFFu));
}

// ------------------------------------------------------------------------------------------------------------------------
// Second generation of the fused match.  The first kernel (since removed) had the same arithmetic and operand layouts; what
// changed, each item aimed at the fixed costs that dominated it (20.5 us at B = 1 against a 7.2 us HBM floor):
//   * the codebook stream starts before anything else: thread 0 initialises the barriers, fences and issues the TMA loads
//     of the first tiles while the TMEM allocation, the query staging and the normalise/split prologue are still to come
//     (before: after the allocation and a block-wide barrier, and one tile only);
//   * B <= 128 stages its queries in ONE ring stage, so TWO tiles (128 KB per SM, 19 MB chip-wide = 40 % of the table) are in
//     flight during the prologue; B > 128 runs the prologue in two rounds of 128 queries and hands each staging stage to the
//     TMA producer as soon as its round is done;
//   * in every round all eight warps work: warps w and w+4 own the same 32 TMEM lanes (queries) and each converts one K
//     half of the row -- the fp32 -> fp16x2 conversions (the slow pipe) are what the prologue is bound by;
//   * top-k (k <= 8) and `upright` (codebook.py:64-71) run on this kernel too: a per-lane sorted list of K (score, index)
//     pairs in registers replaces the running best, per-CTA lists go through a scratch table and the last CTA merges them
//     ("score descending, ties to the lowest index" = the order of the packed 64-bit keys); upright is the same kernel on a
//     tensor map whose row stride is num_cyclo rows.
template <int K>
struct TopList {
  float s[K];
  int i[K];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int j = 0; j < K; ++j) { s[j] = -3.0e38f; i[j] = 0x7FFFFFFF; }
  }
  __device__ __forceinline__ float worst() const { return s[K - 1]; }
  // precondition: v > worst().  Replaces the worst entry and bubbles up past STRICTLY smaller scores only, so that among equal
  // scores the entry inserted first (lower row index: a CTA visits its rows in increasing order) stays ahead.
  __device__ __forceinline__ void insert(float v, int idx) {
    s[K - 1] = v; i[K - 1] = idx;
#pragma unroll
    for (int p = K - 1; p >= 1; --p) {
      if (s[p] > s[p - 1]) {
        const float ts = s[p]; s[p] = s[p - 1]; s[p - 1] = ts;
        const int ti = i[p]; i[p] = i[p - 1]; i[p - 1] = ti;
      }
    }
  }
};

template <int MQ, int K>
__global__ void __launch_bounds__(256, 1)
tc_match2_kernel(const __grid_constant__ CUtensorMap tm_e_hi, const __grid_constant__ CUtensorMap tm_e_lo, const float* __restrict__ z,
                 int B, int n_rows, int n_tiles, int idx_mul, long long row_offset, int k_out, unsigned long long* __restrict__ best,
                 unsigned long long* __restrict__ lists, unsigned int* __restrict__ counter, float* __restrict__ scores_out,
                 int* __restrict__ idx_out, long long* __restrict__ trace) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* e_smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* e_full = reinterpret_cast<uint64_t*>(e_smem + MT_STAGES * MT_STAGE_BYTES);
  uint64_t* e_empty = e_full + MT_STAGES;
  uint64_t* acc_full = e_empty + MT_STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_empty + 2);
  __shared__ int s_is_last;
  __shared__ float s_part[MQ][2][128];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool tr = trace != nullptr && blockIdx.x == 0;
  if (tr && threadIdx.x == 0) trace[0] = clock64();
  const int my_tiles = (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  // ring stage of this CTA's i-th tile.  MQ = 2 swaps stages 1 and 2: stage 2 is the staging area of the FIRST prologue round
  // and is free (and refilled) one round earlier than stage 1.
  auto stage_of = [](int i) -> int { const int r = i % MT_STAGES; return MQ == 1 ? r : (r == 0 ? 0 : MT_STAGES - r); };
  auto load_tile = [&](int i) {
    const int s = stage_of(i);
    const int row0 = ((int)blockIdx.x + i * (int)gridDim.x) * MT_ROWS;
    uint8_t* st = e_smem + s * MT_STAGE_BYTES;
    mbar_arrive_expect_tx(&e_full[s], MT_STAGE_BYTES);
    tma_load_2d(st, &tm_e_hi, &e_full[s], 0, row0);
    tma_load_2d(st + MT_E_BYTES, &tm_e_hi, &e_full[s], 64, row0);
    tma_load_2d(st + 2 * MT_E_BYTES, &tm_e_lo, &e_full[s], 0, row0);
    tma_load_2d(st + 3 * MT_E_BYTES, &tm_e_lo, &e_full[s], 64, row0);
  };
  constexpr int kPrefetch = MQ == 1 ? 2 : 1;   // tiles requested before the prologue

  if (threadIdx.x == 0) {
    for (int s = 0; s < MT_STAGES; ++s) { mbar_init(&e_full[s], 1); mbar_init(&e_empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], 4); }
    fence_barrier_init();
    for (int i = 0; i < kPrefetch && i < my_tiles; ++i) load_tile(i);     // the codebook stream starts here
  }
  if (warp == 2) tmem_alloc<512>(tmem_ptr);

  // ---- prologue: 128 queries per round.  Phase A (all warps, coalesced): cp.async the round's rows as fp32 into a staging
  //      stage (512 B per row, 16-byte chunks XOR-swizzled by the row: the row-wise writes here and the thread-per-row reads of
  //      phase B are both bank-conflict free).  Round 0 -> stage 2, round 1 (MQ = 2) -> stage 1.
#pragma unroll
  for (int mq = 0; mq < MQ; ++mq) {
    uint8_t* stg = e_smem + (2 - mq) * MT_STAGE_BYTES;
#pragma unroll 4
    for (int r = warp; r < 128; r += 8) {
      const int row = mq * 128 + r;
      cp_async_16(stg + r * 512 + ((lane ^ (r & 31)) << 4), z + (long long)(row < B ? row : 0) * 128 + lane * 4, row < B);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");      // one group per round: round 1's rows keep arriving while round 0 is converted
  }
  if (MQ == 2) asm volatile("cp.async.wait_group 1;" ::: "memory"); else asm volatile("cp.async.wait_group 0;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  if (tr && threadIdx.x == 0) trace[4] = clock64();
  // ---- phase B: warps w and w+4 own TMEM lanes 32*(w%4).. = queries r = 32*(w%4) + lane of the round's block; both read
  //      sum the squares of one K half each and exchange the partial sums (tf.nn.l2_normalize: z * rsqrt(max(sum z^2, 1e-12))),
  //      warp w < 4 converts K elements 0..63, warp w + 4 elements 64..127: scale by 64, split into fp16 (hi, lo), park in TMEM as the MMA's A operand
  //      (lane = query, column c = K elements 2c, 2c+1; Q_hi at columns [mq*128, +64), Q_lo at [mq*128+64, +64)).
#pragma unroll
  for (int mq = 0; mq < MQ; ++mq) {
    if (mq == 1) {                                   // round 1's rows: this thread's copies have landed; the barrier makes everybody's visible
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncthreads();
    }
    const int q = warp & 3, half = warp >> 2, r = q * 32 + lane;
    const uint8_t* src = e_smem + (2 - mq) * MT_STAGE_BYTES + r * 512;
    float4 mine[16];
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const float4 v = *reinterpret_cast<const float4*>(src + (((half * 16 + c) ^ (r & 31)) << 4));
      s0 = fmaf(v.x, v.x, s0); s1 = fmaf(v.y, v.y, s1); s2 = fmaf(v.z, v.z, s2); s3 = fmaf(v.w, v.w, s3);
      mine[c] = v;
    }
    s_part[mq][half][r] = (s0 + s1) + (s2 + s3);       // each thread sums its K half; the two halves meet through shared memory
    __syncthreads();
    const float ss = fmaxf(s_part[mq][0][r] + s_part[mq][1][r], 1e-12f);
    float y = rsqrtf(ss);
    y = y * (1.5f - 0.5f * ss * y * y);              // one Newton step: ~1 ulp
    const float inv = MT_SCALE * y;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(mq * 128 + half * 32);
#pragma unroll
    for (int g = 0; g < 4; ++g) {                    // 16 K elements -> 8 packed columns of Q_hi and of Q_lo
      uint32_t hi[8], lo[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 v = mine[g * 4 + j];
        split_f16x2(v.x * inv, v.y * inv, hi[2 * j], lo[2 * j]);
        split_f16x2(v.z * inv, v.w * inv, hi[2 * j + 1], lo[2 * j + 1]);
      }
      tmem_st_32x8(lane_base + (uint32_t)(g * 8), hi);
      tmem_st_32x8(lane_base + (uint32_t)(64 + g * 8), lo);
    }
    tmem_st_wait();
    fence_proxy_async_smem();   // the staging stage is about to be overwritten by TMA (async proxy)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // the round's staging stage is free: request the tile that lives there (MQ = 1: tile 2 -> stage 2; MQ = 2: tile 1 -> stage 2,
    // then tile 2 -> stage 1)
    if (threadIdx.x == 0 && kPrefetch + mq < my_tiles) load_tile(kPrefetch + mq);
  }
  if (tr && threadIdx.x == 0) trace[1] = clock64();
  constexpr int kIssued = kPrefetch + MQ;     // tiles requested so far (= MT_STAGES)

  if (warp == 0) {
    if (lane == 0) {
      for (int i = kIssued; i < my_tiles; ++i) {
        const int s = stage_of(i);
        mbar_wait(&e_empty[s], ((uint32_t)(i / MT_STAGES) & 1u) ^ 1u);
        load_tile(i);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(128, MT_ROWS, 0);
      for (int i = 0; i < my_tiles; ++i) {
        const int s = stage_of(i);
        mbar_wait(&e_full[s], (uint32_t)(i / MT_STAGES) & 1u);
        if (tr && i < 16) trace[16 + i * 8 + 0] = clock64();
        const uint32_t est = smem_u32(e_smem + s * MT_STAGE_BYTES);
#pragma unroll 1
        for (int mq = 0; mq < MQ; ++mq) {
          const int u = i * MQ + mq, as = u & 1;        // accumulator stage alternates per (tile, query block)
          mbar_wait(&acc_empty[as], ((uint32_t)(u >> 1) & 1u) ^ 1u);
          tc_fence_after();
          if (tr && i < 16) trace[16 + i * 8 + 1 + mq * 2] = clock64();
          const uint32_t d = tmem_base + (uint32_t)(MT_TMEM_ACC0 + as * MT_ROWS);
          const uint32_t q_hi = tmem_base + (uint32_t)(mq * 128), q_lo = q_hi + 64;
#pragma unroll 1
          for (int kh = 0; kh < 2; ++kh) {
            const uint64_t e_hi = make_sw128_kmajor_desc(est + kh * MT_E_BYTES);
            const uint64_t e_lo = make_sw128_kmajor_desc(est + (2 + kh) * MT_E_BYTES);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint32_t kc = (uint32_t)((kh * 4 + k) * 8);   // 16 fp16 K elements = 8 packed columns
              umma_f16_ts(d, q_lo + kc, desc_advance_k(e_hi, k), idesc, (kh > 0 || k > 0) ? 1u : 0u);
              umma_f16_ts(d, q_hi + kc, desc_advance_k(e_lo, k), idesc, 1u);
              umma_f16_ts(d, q_hi + kc, desc_advance_k(e_hi, k), idesc, 1u);
            }
          }
          umma_commit(&acc_full[as]);
          if (tr && i < 16) trace[16 + i * 8 + 2 + mq * 2] = clock64();
        }
        umma_commit(&e_empty[s]);
      }
    }
  } else if (warp >= 4) {
    const int q = warp & 3;
    TopList<K> l0, l1;                       // one list per query block (named objects: the mq loop is rolled)
    l0.init(); l1.init();
    for (int i = 0; i < my_tiles; ++i) {
      const int row0 = ((int)blockIdx.x + i * (int)gridDim.x) * MT_ROWS;
      const int nvalid = min(MT_ROWS, n_rows - row0);
#pragma unroll 1
      for (int mq = 0; mq < MQ; ++mq) {
        const int u = i * MQ + mq, as = u & 1;
        TopList<K> cur = mq ? l1 : l0;
        mbar_wait(&acc_full[as], (uint32_t)(u >> 1) & 1u);
        tc_fence_after();
        if (tr && warp == 4 && lane == 0 && i < 16) trace[16 + i * 8 + 5 + mq] = clock64();
#pragma unroll 1
        for (int c = 0; c < MT_ROWS / 64; ++c) {
          uint32_t v[32], w[32];
          const uint32_t col = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(MT_TMEM_ACC0 + as * MT_ROWS + c * 64);
          tmem_ld_32x32(col, v);
          tmem_ld_32x32(col + 32, w);
          tmem_ld_wait();
          if (nvalid < MT_ROWS) {                       // last tile only: padding rows must never win
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (c * 64 + j >= nvalid) v[j] = 0xFF800000u;        // -inf
              if (c * 64 + 32 + j >= nvalid) w[j] = 0xFF800000u;
            }
          }
          // log-depth max of the 64 scores; the (rare) list update only runs when this chunk beats the list's worst entry
          float m[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) m[j] = fmaxf(__uint_as_float(v[j]), __uint_as_float(w[j]));
#pragma unroll
          for (int st = 16; st >= 1; st >>= 1)
#pragma unroll
            for (int j = 0; j < st; ++j) m[j] = fmaxf(m[j], m[j + st]);
          const float mx = m[0];
          if (mx > cur.worst()) {                       // strict >: an equal score later in the table never displaces an earlier row
            if (K == 1) {
              int first = 63;
#pragma unroll
              for (int j = 31; j >= 0; --j)
                if (__uint_as_float(w[j]) == mx) first = 32 + j;
#pragma unroll
              for (int j = 31; j >= 0; --j)
                if (__uint_as_float(v[j]) == mx) first = j;          // lowest column holding the maximum
              cur.s[0] = mx;
              cur.i[0] = row0 + c * 64 + first;
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (__uint_as_float(v[j]) > cur.worst()) cur.insert(__uint_as_float(v[j]), row0 + c * 64 + j);
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (__uint_as_float(w[j]) > cur.worst()) cur.insert(__uint_as_float(w[j]), row0 + c * 64 + 32 + j);
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[as]);
        if (mq) l1 = cur; else l0 = cur;
      }
    }
    constexpr float kUnscale = 1.f / (MT_SCALE * MT_SCALE);
#pragma unroll
    for (int mq = 0; mq < MQ; ++mq) {
      const int qi = mq * 128 + q * 32 + lane;
      const TopList<K>& fin = mq ? l1 : l0;
      if (qi < B) {
        if (K == 1) {
          if (fin.i[0] != 0x7FFFFFFF) atomicMax(best + qi, pack_best(fin.s[0] * kUnscale, fin.i[0]));
        } else {
#pragma unroll
          for (int j = 0; j < K; ++j)
            lists[((size_t)blockIdx.x * B + qi) * K + j] = fin.i[j] != 0x7FFFFFFF ? pack_best(fin.s[j] * kUnscale, fin.i[j]) : 0ull;
        }
      }
    }
  }
  // ---- teardown + last-CTA finalisation ----
  if (tr && threadIdx.x == 128) trace[2] = clock64();
  tc_fence_before();
  __threadfence();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
  if (threadIdx.x == 0) {
    const unsigned int ticket = atomicAdd(counter, 1u);
    s_is_last = (ticket == gridDim.x - 1);
  }
  __syncthreads();
  if (s_is_last) {
    __threadfence();
    if (K == 1) {
      for (int qi = threadIdx.x; qi < B; qi += blockDim.x) {
        const unsigned long long k = atomicExch(best + qi, 0ull);   // read + re-arm
        float s;
        int idx;
        unpack_best(k, s, idx);
        scores_out[qi] = s;
        idx_out[qi] = (int)((long long)idx * idx_mul + row_offset);
      }
    } else {
      // one warp per query: the k_out largest of the gridDim.x * K packed keys (all distinct: the index is part of the key)
      constexpr int kPerLane = (148 * K + 31) / 32;
      const int total = (int)gridDim.x * K;
      for (int qi = warp; qi < B; qi += 8) {
        unsigned long long key[kPerLane];
#pragma unroll
        for (int t = 0; t < kPerLane; ++t) {
          const int e = lane + 32 * t;
          key[t] = e < total ? __ldcg(lists + ((size_t)(e / K) * B + qi) * K + (e % K)) : 0ull;
        }
        for (int j = 0; j < k_out; ++j) {
          unsigned long long mxk = 0ull;
#pragma unroll
          for (int t = 0; t < kPerLane; ++t) mxk = key[t] > mxk ? key[t] : mxk;
          unsigned long long wmax = mxk;
#pragma unroll
          for (int off = 16; off >= 1; off >>= 1) {
            const unsigned long long o = __shfl_xor_sync(0xFFFFFFFFu, wmax, off);
            wmax = o > wmax ? o : wmax;
          }
          if (wmax != 0ull) {
#pragma unroll
            for (int t = 0; t < kPerLane; ++t)
              if (key[t] == wmax) key[t] = 0ull;      // unique key: exactly one lane clears it
          }
          if (lane == 0) {
            float s = -INFINITY;
            int idx = -1;
            if (wmax != 0ull) {
              unpack_best(wmax, s, idx);
              idx = (int)((long long)idx * idx_mul + row_offset);
            }
            scores_out[(size_t)qi * k_out + j] = s;
            idx_out[(size_t)qi * k_out + j] = idx;
          }
        }
      }
    }
    if (threadIdx.x == 0) *counter = 0u;
  }
  if (tr && threadIdx.x == 0) trace[3] = clock64();
}

// Measurement aid (aae_launch_floor_probe): the fixed cost of launching a grid shaped like the match kernel -- one CTA per SM, the
// same dynamic shared memory (forces the same L1/shared carveout), optionally the same 512-column TMEM allocation -- that does nothing.
__global__ void __launch_bounds__(256, 1) launch_floor_kernel(int tmem, unsigned int* sink) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint32_t tmem_ptr;
  if (tmem) {
    if (threadIdx.x < 32) tmem_alloc<512>(&tmem_ptr);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (threadIdx.x < 32) tmem_dealloc<512>(tmem_ptr);
  }
  if (sink != nullptr && threadIdx.x == 0 && smem_raw[0] == 0xFF && blockIdx.x == 0xFFFFFFFFu) *sink = 1u;   // never true: keeps smem_raw referenced
}

// fp32 [n_rows][128] -> (hi, lo) fp16 [n_pad][128], scaled by 64; rows >= n_rows are zero
__global__ void pack_codebook_kernel(const float* __restrict__ E, long long n_rows, long long n_pad, __half* __restrict__ hi,
                                     __half* __restrict__ lo) {
  const long long total = n_pad * 128;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const float x = (i / 128 < n_rows) ? E[i] * MT_SCALE : 0.f;
    __half h, l;
    split_f16(x, h, l);
    hi[i] = h;
    lo[i] = l;
  }
}

}  // namespace

struct TcCodebook {
  int device;
  long long n_rows, n_pad;
  int n_tiles, max_batch, sm_count, num_cyclo;
  long long n_up;                 // rows of the `upright` view (every num_cyclo-th row)
  int n_tiles_up;
  __half *e_hi = nullptr, *e_lo = nullptr;
  CUtensorMap tm_hi, tm_lo, tm_hi_up, tm_lo_up;
  bool have_up = false;
  unsigned long long* best = nullptr;
  unsigned long long* lists = nullptr;   // [grid][max_batch][8] packed keys of the per-CTA top-k lists (k > 1)
  unsigned int* counter = nullptr;
  long long* trace = nullptr;   // optional clock64 trace of CTA 0 (AAE_MATCH_TRACE=1), diagnostics only
};

constexpr int MT_KMAX = 8;

int tc_codebook_max_k() { return MT_KMAX; }

int tc_launch_floor_probe(int device, int with_tmem, cudaStream_t s) {
  static bool attr_set = false;
  if (!attr_set) {
    AAE_CUDA_OK(cudaFuncSetAttribute(launch_floor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MT_SMEM_TOTAL));
    attr_set = true;
  }
  static int sms = 0;                                   // (cudaGetDeviceProperties costs milliseconds: never on a timed path)
  if (sms == 0) AAE_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  launch_floor_kernel<<<std::min(sms, 148), 256, MT_SMEM_TOTAL, s>>>(with_tmem, nullptr);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

int tc_codebook_create(int device, const float* E_dev, int64_t n_rows, int latent, int num_cyclo, int max_batch, TcCodebook** out) {
  *out = nullptr;
  AAE_REQUIRE(aae_device_supported(device), "AAE_PREC_TC_SPLIT needs a compute-capability 10.x device (tcgen05/TMEM)");
  AAE_REQUIRE(latent == 128, "AAE_PREC_TC_SPLIT codebook match is built for latent = 128 (got %d)", latent);
  TcCodebook* h = new TcCodebook();
  h->device = device;
  h->n_rows = n_rows;
  h->n_tiles = (int)ceil_div(n_rows, MT_ROWS);
  h->n_pad = (long long)h->n_tiles * MT_ROWS;
  h->max_batch = max_batch;
  h->num_cyclo = std::max(1, num_cyclo);
  h->n_up = ceil_div(n_rows, (int64_t)h->num_cyclo);
  h->n_tiles_up = (int)ceil_div(h->n_up, (int64_t)MT_ROWS);
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  h->sm_count = std::min(prop.multiProcessorCount, 148);
  const int cap_b = std::min(256, std::max(1, max_batch));
  cudaError_t e = cudaMalloc(&h->e_hi, (size_t)h->n_pad * 128 * sizeof(__half));
  if (e == cudaSuccess) e = cudaMalloc(&h->e_lo, (size_t)h->n_pad * 128 * sizeof(__half));
  if (e == cudaSuccess) e = cudaMalloc(&h->best, 256 * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMalloc(&h->lists, (size_t)h->sm_count * cap_b * MT_KMAX * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMalloc(&h->counter, sizeof(unsigned int));
  if (e != cudaSuccess) { set_error("tc codebook alloc failed: %s", cudaGetErrorString(e)); tc_codebook_destroy(h); return AAE_ERR_OOM; }
  cudaMemset(h->best, 0, 256 * sizeof(unsigned long long));
  cudaMemset(h->counter, 0, sizeof(unsigned int));
  if (getenv("AAE_MATCH_TRACE")) { cudaMalloc(&h->trace, 768 * sizeof(long long)); cudaMemset(h->trace, 0, 768 * sizeof(long long)); }
  pack_codebook_kernel<<<1024, 256>>>(E_dev, n_rows, h->n_pad, h->e_hi, h->e_lo);
  g_launches.fetch_add(1);
  e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { set_error("pack_codebook failed: %s", cudaGetErrorString(e)); tc_codebook_destroy(h); return AAE_ERR_CUDA; }
  const uint64_t dims[2] = {128, (uint64_t)h->n_pad};
  const uint64_t strides[1] = {256};
  const uint32_t box[2] = {64, MT_ROWS};
  int st = make_tmap_f16(&h->tm_hi, h->e_hi, 2, dims, strides, box);
  if (st == AAE_OK) st = make_tmap_f16(&h->tm_lo, h->e_lo, 2, dims, strides, box);
  if (st == AAE_OK && h->num_cyclo > 1) {
    // `upright` view (codebook.py:66 cos[::num_cyclo]): the same memory with a row stride of num_cyclo rows; boxes past
    // the last such row are zero-filled by TMA and masked by the kernel
    const uint64_t dims_u[2] = {128, (uint64_t)h->n_up};
    const uint64_t strides_u[1] = {(uint64_t)256 * (uint64_t)h->num_cyclo};
    st = make_tmap_f16(&h->tm_hi_up, h->e_hi, 2, dims_u, strides_u, box);
    if (st == AAE_OK) st = make_tmap_f16(&h->tm_lo_up, h->e_lo, 2, dims_u, strides_u, box);
    h->have_up = st == AAE_OK;
  }
  if (st != AAE_OK) { tc_codebook_destroy(h); return st; }
  auto attr = [&](const void* fn) { return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, MT_SMEM_TOTAL); };
  e = attr((const void*)tc_match2_kernel<1, 1>);
  if (e == cudaSuccess) e = attr((const void*)tc_match2_kernel<2, 1>);
  if (e == cudaSuccess) e = attr((const void*)tc_match2_kernel<1, MT_KMAX>);
  if (e == cudaSuccess) e = attr((const void*)tc_match2_kernel<2, MT_KMAX>);
  if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(match kernels) failed: %s", cudaGetErrorString(e)); tc_codebook_destroy(h); return AAE_ERR_CUDA; }
  *out = h;
  return AAE_OK;
}

void tc_codebook_destroy(TcCodebook* h) {
  if (!h) return;
  cudaFree(h->e_hi); cudaFree(h->e_lo); cudaFree(h->best); cudaFree(h->lists); cudaFree(h->counter); cudaFree(h->trace);
  delete h;
}

static void print_trace(TcCodebook* h, cudaStream_t s) {
  long long t[768];
  cudaStreamSynchronize(s);
  cudaMemcpy(t, h->trace, sizeof(t), cudaMemcpyDeviceToHost);
  fprintf(stderr, "[match2 trace, CTA 0, clocks from kernel entry] queries staged + TMEM allocated %lld | prologue done %lld | loops done %lld | end %lld\n",
          t[4] - t[0], t[1] - t[0], t[2] - t[0], t[3] - t[0]);
  for (int i = 0; i < 6; ++i)
    fprintf(stderr, "  tile %d: e_full %lld | mq0 acc_empty %lld issued %lld | mq1 acc_empty %lld issued %lld | epi acc_full mq0 %lld mq1 %lld\n", i,
            t[16 + i * 8] - t[0], t[16 + i * 8 + 1] - t[0], t[16 + i * 8 + 2] - t[0], t[16 + i * 8 + 3] - t[0], t[16 + i * 8 + 4] - t[0],
            t[16 + i * 8 + 5] - t[0], t[16 + i * 8 + 6] - t[0]);
}

// k in [1, 8]; upright != 0 searches rows (row_offset + r * num_cyclo) only -- needs row_offset % num_cyclo == 0 (shard_bounds aligns shards so)
int tc_codebook_match(TcCodebook* h, const float* z_dev, int B, int64_t row_offset, int k, int upright, float* scores_out, int32_t* idx_out,
                      cudaStream_t s) {
  AAE_REQUIRE(k >= 1 && k <= MT_KMAX, "tc match: k=%d outside [1, %d]", k, MT_KMAX);
  AAE_REQUIRE(!upright || (h->have_up || h->num_cyclo == 1), "tc match: no upright view");
  AAE_REQUIRE(!upright || row_offset % h->num_cyclo == 0, "tc match: upright needs a shard offset that is a multiple of num_cyclo");
  AAE_REQUIRE(B <= h->max_batch || k == 1, "tc match: batch %d > max_batch %d", B, h->max_batch);
  const bool up = upright && h->num_cyclo > 1;
  const int n_tiles = up ? h->n_tiles_up : h->n_tiles;
  const int n_rows = (int)(up ? h->n_up : h->n_rows);
  const int idx_mul = up ? h->num_cyclo : 1;
  const CUtensorMap& th = up ? h->tm_hi_up : h->tm_hi;
  const CUtensorMap& tl = up ? h->tm_lo_up : h->tm_lo;
  const int grid = std::min(h->sm_count, n_tiles);
  for (int a = 0; a < B; a += 256) {
    const int nb = std::min(256, B - a);
    const float* z = z_dev + (size_t)a * 128;
    float* so = scores_out + (size_t)a * k;
    int32_t* io = idx_out + (size_t)a * k;
    if (k == 1) {
      if (nb > 128) tc_match2_kernel<2, 1><<<grid, 256, MT_SMEM_TOTAL, s>>>(th, tl, z, nb, n_rows, n_tiles, idx_mul, (long long)row_offset, 1, h->best, h->lists, h->counter, so, io, h->trace);
      else tc_match2_kernel<1, 1><<<grid, 256, MT_SMEM_TOTAL, s>>>(th, tl, z, nb, n_rows, n_tiles, idx_mul, (long long)row_offset, 1, h->best, h->lists, h->counter, so, io, h->trace);
    } else {
      if (nb > 128) tc_match2_kernel<2, MT_KMAX><<<grid, 256, MT_SMEM_TOTAL, s>>>(th, tl, z, nb, n_rows, n_tiles, idx_mul, (long long)row_offset, k, h->best, h->lists, h->counter, so, io, h->trace);
      else tc_match2_kernel<1, MT_KMAX><<<grid, 256, MT_SMEM_TOTAL, s>>>(th, tl, z, nb, n_rows, n_tiles, idx_mul, (long long)row_offset, k, h->best, h->lists, h->counter, so, io, h->trace);
    }
    AAE_LAUNCH_OK();
  }
  if (h->trace) print_trace(h, s);
  return AAE_OK;
}

}  // namespace aae
