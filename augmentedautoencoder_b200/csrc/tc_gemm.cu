// tcgen05 implicit-GEMM for the encoder's dense contractions (AAE_PREC_TC_SPLIT).
//
//   D[128 output pixels x N_TILE channels] (fp32, TMEM) += A[128 x 64] * W[N_TILE x 64]^T   per K chunk of 64 input channels
//
// Replaces tf.layers.conv2d(k=5, stride 2, padding='same') + ReLU and tf.layers.dense of
// auto_pose/ae/encoder.py:43-50,62-66 for every layer with Cin % 64 == 0 (conv2..conv4, dense).
//
// fp32-grade arithmetic on fp16 tensor cores: every fp32 operand x is stored as two fp16 terms, hi = rn(x) and
// lo = rn(x - hi) (22 significant bits; operands pre-scaled by a power of two so lo stays a normal fp16), and each
// K chunk issues three MMAs  hi*hi + hi*lo + lo*hi  into the same fp32 TMEM accumulator.
//
// Data movement: activations live in HBM in a space-to-depth layout  Xs[b, h/2, w/2, (h%2, w%2, c)]  written by the
// producing layer's epilogue, so that tap (kh, kw) of the stride-2 / asymmetric-SAME(1,2) convolution is a plain
// unit-stride 4-D TMA box  [64 ch, BW, BH, BB]  at offset (di, dj) with zero fill outside the image -- no im2col
// buffer, no stride-2 gathers.  Weights are pre-packed [Cout][25*Cin] K-major.  Both operands land in shared memory in
// the 128-byte-swizzle canonical layout tcgen05.mma consumes directly.
//
// Warp roles (512 threads): warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM allocator, warps 4-15 epilogue, three per TMEM lane
// quadrant (TMEM -> registers -> bias/ReLU -> hi/lo split -> global, in the next layer's space-to-depth layout).
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "tc.cuh"
#include "tc_common.cuh"
#include "tc_plan.cuh"

namespace aae {

using namespace tc;

// ------------------------------------------------------------------------------------------------- host helpers
PFN_tmapEncodeTiled get_tmap_encoder() {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  }
  return fn;
}

int make_tmap_f16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
                  int swizzle_bytes) {
  PFN_tmapEncodeTiled enc = get_tmap_encoder();
  if (!enc) { set_error("cuTensorMapEncodeTiled is unavailable in this driver"); return AAE_ERR_CUDA; }
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d)", (int)r, rank); return AAE_ERR_CUDA; }
  return AAE_OK;
}

// ------------------------------------------------------------------------------------------------- kernel
template <int N_TILE, int STAGES, int KCH = 64>
struct TcSmem {
  static constexpr int A_BYTES = 128 * KCH * 2;        // 128 rows x KCH fp16
  static constexpr int W_BYTES = N_TILE * KCH * 2;
  static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * W_BYTES;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

template <int N_TILE, int STAGES, int KCH>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
               const __grid_constant__ CUtensorMap tm_w_hi, const __grid_constant__ CUtensorMap tm_w_lo, const TcGemmParams p) {
  using S = TcSmem<N_TILE, STAGES, KCH>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * S::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * 128;
  const int n0 = blockIdx.y * N_TILE;
  const int total_iters = p.taps * p.chunks_per_tap;
  const int it_begin = blockIdx.z * p.iters_per_split;
  const int it_end = min(total_iters, it_begin + p.iters_per_split);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tm_a_hi); prefetch_tmap(&tm_a_lo); prefetch_tmap(&tm_w_hi); prefetch_tmap(&tm_w_lo);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<2 * N_TILE>(tmem_ptr);   // [0,N) main hi*hi accumulator, [N,2N) cross-term accumulator
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      const int hw = p.OH * p.OW;
      const int b0 = m0 / hw, rem = m0 - b0 * hw;
      const int oh0 = rem / p.OW, ow0 = rem - oh0 * p.OW;
      for (int it = it_begin, i = 0; it < it_end; ++it, ++i) {
        const int s = i % STAGES;
        const uint32_t ph = (uint32_t)(i / STAGES) & 1u;
        mbar_wait(&empty_bar[s], ph ^ 1u);
        const int tap = it / p.chunks_per_tap, cc = it - tap * p.chunks_per_tap;
        uint8_t* st = smem + s * S::STAGE_BYTES;
        mbar_arrive_expect_tx(&full_bar[s], S::STAGE_BYTES);
        const int c0 = p.tap_ch[tap] + cc * KCH;
        const int x = ow0 + p.tap_dj[tap], y = oh0 + p.tap_di[tap];
        tma_load_4d(st, &tm_a_hi, &full_bar[s], c0, x, y, b0);
        tma_load_4d(st + S::A_BYTES, &tm_a_lo, &full_bar[s], c0, x, y, b0);
        const int kcol = it * KCH;
        tma_load_2d(st + 2 * S::A_BYTES, &tm_w_hi, &full_bar[s], kcol, n0);
        tma_load_2d(st + 2 * S::A_BYTES + S::W_BYTES, &tm_w_lo, &full_bar[s], kcol, n0);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(128, N_TILE, 0);
      for (int it = it_begin, i = 0; it < it_end; ++it, ++i) {
        const int s = i % STAGES;
        const uint32_t ph = (uint32_t)(i / STAGES) & 1u;
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        const uint32_t st = smem_u32(smem + s * S::STAGE_BYTES);
        const uint64_t a_hi = KCH == 64 ? make_sw128_kmajor_desc(st) : make_sw64_kmajor_desc(st);
        const uint64_t a_lo = KCH == 64 ? make_sw128_kmajor_desc(st + S::A_BYTES) : make_sw64_kmajor_desc(st + S::A_BYTES);
        const uint64_t w_hi = KCH == 64 ? make_sw128_kmajor_desc(st + 2 * S::A_BYTES) : make_sw64_kmajor_desc(st + 2 * S::A_BYTES);
        const uint64_t w_lo = KCH == 64 ? make_sw128_kmajor_desc(st + 2 * S::A_BYTES + S::W_BYTES) : make_sw64_kmajor_desc(st + 2 * S::A_BYTES + S::W_BYTES);
#pragma unroll
        for (int k = 0; k < KCH / 16; ++k) {
          // The tensor core truncates when it adds into a large fp32 accumulator, so the 2^-11-sized cross terms get an
          // accumulator of their own (small magnitude -> negligible truncation) and are folded in by the epilogue in RN fp32.
          const uint32_t first = (i > 0 || k > 0) ? 1u : 0u;
          umma_f16(tmem_base, desc_advance_k(a_hi, k), desc_advance_k(w_hi, k), idesc, first);
          umma_f16(tmem_base + N_TILE, desc_advance_k(a_lo, k), desc_advance_k(w_hi, k), idesc, first);
          umma_f16(tmem_base + N_TILE, desc_advance_k(a_hi, k), desc_advance_k(w_lo, k), idesc, 1u);
        }
        umma_commit(&empty_bar[s]);  // frees the smem stage once these MMAs have read it
      }
      umma_commit(tmem_full_bar);    // accumulator complete
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int q = warp & 3, grp = (warp - 4) >> 2;   // TC_EPI_GROUPS warps per TMEM lane quadrant, interleaved 32-column chunks
    const TcRow row = tc_decode_row(p, m0 + q * 32 + lane);
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    const bool has_work = it_end > it_begin;
    const float unscale = p.amax_bits ? p.unscale * tc_dyn_unscale(__ldg(p.amax_bits)) : p.unscale;
#pragma unroll 1
    for (int c = grp; c < N_TILE / 32; c += TC_EPI_GROUPS) {
      uint32_t v[32], x[32];
      tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), v);
      tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(N_TILE + c * 32), x);
      tmem_ld_wait();
      const int n = n0 + c * 32;
      if (!row.valid || n >= p.N) continue;
      float f[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) f[j] = has_work ? (__uint_as_float(v[j]) + __uint_as_float(x[j])) * unscale : 0.f;
      tc_store_chunk(p, row, n, f, (int)blockIdx.z);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<2 * N_TILE>(tmem_base);
  }
}


// ------------------------------------------------------------------------------------------------- persistent 2-CTA kernel
// The same computation with CTA pairs (cta_group::2): two 128-pixel tiles that share a 256-channel weight tile run as ONE
// M = 256 MMA.  Each CTA stages its own pixels plus only HALF of the weight tile (128 channels), so per K chunk it moves
// 2/3 of the bytes of the single-CTA kernel through L2 -> smem and the tensor core reads 2/3 as much shared memory per
// MMA -- the single-CTA version is shared-memory-bandwidth bound (operand reads + TMA writes > 128 B/clk/SM).  Both CTAs'
// TMA loads complete on the leader's (even rank) barrier; the leader's issuer thread fires the MMAs and multicasts the
// stage-free / accumulator-ready commits to both CTAs; each CTA drains its own 128 TMEM lanes.
struct TcSmem2 {
  static constexpr int STAGES = 6;
  static constexpr int KCH = 32;                          // K chunk per stage (64-byte swizzle)
  static constexpr int T_BYTES = 128 * KCH * 2;          // 128 rows x KCH fp16: A tile and W half tile have the same size
  static constexpr int STAGE_BYTES = 4 * T_BYTES;        // A_hi, A_lo, W_hi(half), W_lo(half)
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 + 256;
};

// One CTA pair per SM pair walks over the output tiles (m pair fastest, so that concurrently running pairs share the weight
// tile in L2).  Barrier setup, TMEM allocation and the launch of a fresh CTA are paid once, and the TMA producer runs ahead
// through the shared-memory ring while the epilogue of the previous tile drains TMEM, so the next tile's MMAs start on full
// stages: per tile only the epilogue itself is exposed (the accumulators occupy all 512 TMEM columns, so it is not
// double-buffered).  tmem_empty (leader CTA) collects one arrival per epilogue warp of BOTH CTAs before the issuer
// overwrites the accumulators.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}

struct TcTileSched {
  int m_pairs, n_tiles, splits;   // tiles = m_pairs * n_tiles * splits, each tile = 256 rows x 256 columns x one K range
  int tma_out;                    // > 0: tm_o_hi / tm_o_lo describe the output and each epilogue warp owns 4 KB of staging behind the ring:
                                  // 1 space-to-depth (hi, lo), 2 plain (hi, lo), 3 depth-to-space (hi, lo), 4 fp32 [M, N] (tm_o_hi only)
  long long* trace;               // AAE_TC_TRACE: clock64 of CTA 0 for its first 96 chunks: [g*4+0] TMA issued, +1 full barrier seen by the MMA thread, +2 MMAs issued, +3 stage seen empty again
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
tc_gemm2p_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                 const __grid_constant__ CUtensorMap tm_w_hi, const __grid_constant__ CUtensorMap tm_w_lo,
                 const __grid_constant__ CUtensorMap tm_o_hi, const __grid_constant__ CUtensorMap tm_o_lo, const TcGemmParams p,
                 const TcTileSched sch) {
  using S = TcSmem2;
  constexpr int STAGES = S::STAGES, KCH = S::KCH;
  constexpr int N_TILE = 256;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * S::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint64_t* tmem_empty_bar = tmem_full_bar + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int n_epi_warps = ((int)blockDim.x >> 5) - 4;
  const int total_iters = p.taps * p.chunks_per_tap;
  const int n_tiles_total = sch.m_pairs * sch.n_tiles * sch.splits;
  const int first_tile = (int)(blockIdx.x >> 1), tile_step = (int)(gridDim.x >> 1);

  if (sch.trace && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    sch.trace[384] = clock64(); sch.trace[385] = (long long)gt;
  }
  if (warp == 0 && lane == 0) { prefetch_tmap(&tm_a_hi); prefetch_tmap(&tm_a_lo); prefetch_tmap(&tm_w_hi); prefetch_tmap(&tm_w_lo); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(tmem_full_bar, 1);
    mbar_init(tmem_empty_bar, 2 * n_epi_warps);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2sm<512>(tmem_ptr);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      const int hw = p.OH * p.OW;
      int g = 0;                                               // ring position, continues across tiles
      for (int t = first_tile; t < n_tiles_total; t += tile_step) {
        const int mp = t % sch.m_pairs, r = t / sch.m_pairs, ny = r % sch.n_tiles, z = r / sch.n_tiles;
        const int m0 = (mp * 2 + (int)rank) * 128, n0 = ny * N_TILE;
        const int b0 = m0 / hw, rem = m0 - b0 * hw;
        const int oh0 = rem / p.OW, ow0 = rem - oh0 * p.OW;
        const int it_begin = z * p.iters_per_split, it_end = min(total_iters, it_begin + p.iters_per_split);
        for (int it = it_begin; it < it_end; ++it, ++g) {
          const int s = g % STAGES;
          mbar_wait(&empty_bar[s], (((uint32_t)(g / STAGES)) & 1u) ^ 1u);
          if (sch.trace && blockIdx.x == 0 && g >= STAGES && g - STAGES < 96) sch.trace[(g - STAGES) * 4 + 3] = clock64();
          const int tap = it / p.chunks_per_tap, cc = it - tap * p.chunks_per_tap;
          uint8_t* st = smem + s * S::STAGE_BYTES;
          if (leader) mbar_arrive_expect_tx(&full_bar[s], 2 * S::STAGE_BYTES);
          const uint32_t lb = leader_bar_addr(&full_bar[s]);
          const int c0 = p.tap_ch[tap] + cc * KCH;
          const int x = ow0 + p.tap_dj[tap], y = oh0 + p.tap_di[tap];
          tma_load_4d_2sm(st, &tm_a_hi, lb, c0, x, y, b0);
          tma_load_4d_2sm(st + S::T_BYTES, &tm_a_lo, lb, c0, x, y, b0);
          const int kcol = it * KCH;
          tma_load_2d_2sm(st + 2 * S::T_BYTES, &tm_w_hi, lb, kcol, n0 + (int)rank * 128);
          tma_load_2d_2sm(st + 3 * S::T_BYTES, &tm_w_lo, lb, kcol, n0 + (int)rank * 128);
          if (sch.trace && blockIdx.x == 0 && g < 96) sch.trace[g * 4 + 0] = clock64();
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(256, N_TILE, 0);
      int g = 0, tl = 0;
      for (int t = first_tile; t < n_tiles_total; t += tile_step, ++tl) {
        const int z = (t / sch.m_pairs) / sch.n_tiles;
        const int it_begin = z * p.iters_per_split, it_end = min(total_iters, it_begin + p.iters_per_split);
        if (tl > 0) {                                           // both CTAs' epilogues have drained the previous accumulators
          if (sch.trace && blockIdx.x == 0 && tl < 16) sch.trace[392 + tl * 4 + 0] = clock64();
          mbar_wait(tmem_empty_bar, (uint32_t)(tl - 1) & 1u);
          tc_fence_after();
          if (sch.trace && blockIdx.x == 0 && tl < 16) sch.trace[392 + tl * 4 + 1] = clock64();
        }
        for (int it = it_begin, i = 0; it < it_end; ++it, ++i, ++g) {
          const int s = g % STAGES;
          mbar_wait(&full_bar[s], ((uint32_t)(g / STAGES)) & 1u);
          tc_fence_after();
          if (sch.trace && blockIdx.x == 0 && g < 96) sch.trace[g * 4 + 1] = clock64();
          const uint32_t st = smem_u32(smem + s * S::STAGE_BYTES);
          const uint64_t a_hi = make_sw64_kmajor_desc(st);
          const uint64_t a_lo = make_sw64_kmajor_desc(st + S::T_BYTES);
          const uint64_t w_hi = make_sw64_kmajor_desc(st + 2 * S::T_BYTES);
          const uint64_t w_lo = make_sw64_kmajor_desc(st + 3 * S::T_BYTES);
#pragma unroll
          for (int k = 0; k < KCH / 16; ++k) {
            const uint32_t first = (i > 0 || k > 0) ? 1u : 0u;
            umma_f16_2sm(tmem_base, desc_advance_k(a_hi, k), desc_advance_k(w_hi, k), idesc, first);
            umma_f16_2sm(tmem_base + N_TILE, desc_advance_k(a_lo, k), desc_advance_k(w_hi, k), idesc, first);
            umma_f16_2sm(tmem_base + N_TILE, desc_advance_k(a_hi, k), desc_advance_k(w_lo, k), idesc, 1u);
          }
          umma_commit_2sm(&empty_bar[s]);
          if (sch.trace && blockIdx.x == 0 && g < 96) sch.trace[g * 4 + 2] = clock64();
        }
        umma_commit_2sm(tmem_full_bar);
      }
    }
  } else if (warp >= 4) {
    const int q = warp & 3, grp = (warp - 4) >> 2, epi_groups = n_epi_warps >> 2;
    const float unscale = p.amax_bits ? p.unscale * tc_dyn_unscale(__ldg(p.amax_bits)) : p.unscale;
    const uint32_t empty_addr = leader_bar_addr(tmem_empty_bar);
    const bool lean = tc_lean_epilogue_ok(p);
    uint8_t* stage_out = smem + STAGES * S::STAGE_BYTES + 1024;   // behind the barriers; 4 KB per epilogue warp when sch.tma_out
    const float floor_v = p.relu == 1 ? 0.f : -INFINITY;
    int tl = 0;
    for (int t = first_tile; t < n_tiles_total; t += tile_step, ++tl) {
      const int mp = t % sch.m_pairs, r = t / sch.m_pairs, ny = r % sch.n_tiles, z = r / sch.n_tiles;
      const int m0 = (mp * 2 + (int)rank) * 128, n0 = ny * N_TILE;
      const TcRow row = tc_decode_row(p, m0 + q * 32 + lane);
      mbar_wait(tmem_full_bar, (uint32_t)tl & 1u);
      tc_fence_after();
      if (sch.trace && blockIdx.x == 0 && threadIdx.x == 128 && tl < 16) sch.trace[392 + tl * 4 + 2] = clock64();
      bool released = false;
      if ((lean && sch.tma_out >= 1 && sch.tma_out <= 3) || sch.tma_out == 4) {
        // TMA-store epilogue: the warp parks its 32 pixels x 32 columns (hi and lo with 64-byte rows and 64-byte swizzle, or fp32
        // with 128-byte rows and 128-byte swizzle) in its own 4 KB of shared memory and one lane ships the box(es) with tensor
        // stores, so the LSU sees 8 conflict-free STS.128 per thread instead of 8 STG.128 that each touch 32 different lines.
        // The stores drain while the next chunk is computed (and while the next tile's MMAs run); the buffer is reused once the
        // engine has READ it.
        uint8_t* sbuf = stage_out + (warp - 4) * 4096;
        const int mw = m0 + q * 32;                              // the warp's first pixel: its 32 pixels lie in one image
        const TcRow r0 = tc_decode_row(p, mw);
        const int rsw = (lane >> 1) & 3;
#pragma unroll 1
        for (int c = grp; c < N_TILE / 32; c += epi_groups) {
          uint32_t v[32], x[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), v);
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(N_TILE + c * 32), x);
          tmem_ld_wait();
          if (c + epi_groups >= N_TILE / 32) {                      // last chunk of this warp: its accumulator words are in registers,
            tc_fence_before();                                         // the issuer may overwrite TMEM while the warp finishes the chunk
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(empty_addr);
            released = true;
          }
          const int n = n0 + c * 32;
          if (mw >= p.M || n >= p.N) continue;
          if (sch.tma_out == 4) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __float_as_uint((__uint_as_float(v[j]) + __uint_as_float(x[j])) * unscale);
            if (lane == 0) bulk_wait_read_all();                  // the previous chunk's store has read the buffer
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 8; ++j)
              *reinterpret_cast<uint4*>(sbuf + lane * 128 + ((j ^ (lane & 7)) << 4)) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          } else {
            uint32_t hi[16], lo[16];
            tc_lean_chunk(p, n, v, x, unscale, floor_v, hi, lo);
            if (lane == 0) bulk_wait_read_all();
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int ch = (j ^ rsw) << 4;
              *reinterpret_cast<uint4*>(sbuf + lane * 64 + ch) = make_uint4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
              *reinterpret_cast<uint4*>(sbuf + 2048 + lane * 64 + ch) = make_uint4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
            }
          }
          fence_proxy_async_smem();                               // generic-proxy writes -> visible to the TMA engine
          __syncwarp();
          if (lane == 0) {
            if (sch.tma_out == 4) {
              tma_store_2d(&tm_o_hi, sbuf, 2 * n, mw);            // fp32 column n = fp16 column 2n of the map
            } else if (sch.tma_out == 2) {
              tma_store_2d(&tm_o_hi, sbuf, n, mw);
              tma_store_2d(&tm_o_lo, sbuf + 2048, n, mw);
            } else if (sch.tma_out == 1) {                        // {channel, column parity, column / 2, row parity, image * OH/2 + row / 2}
              const int c4 = r0.b * (p.OH >> 1) + (r0.i >> 1);
              tma_store_5d(&tm_o_hi, sbuf, n, 0, r0.j >> 1, r0.i & 1, c4);
              tma_store_5d(&tm_o_lo, sbuf + 2048, n, 0, r0.j >> 1, r0.i & 1, c4);
            } else {                                              // depth-to-space: {channel, x parity, column, y parity, image * OH + row}
              const int cq = p.N >> 2, cls = n / cq, co = n - cls * cq;
              tma_store_5d(&tm_o_hi, sbuf, co, cls & 1, r0.j, cls >> 1, r0.b * p.OH + r0.i);
              tma_store_5d(&tm_o_lo, sbuf + 2048, co, cls & 1, r0.j, cls >> 1, r0.b * p.OH + r0.i);
            }
            bulk_commit_group();
          }
        }
      } else if (lean) {
#pragma unroll 1
        for (int c = grp; c < N_TILE / 32; c += epi_groups) {
          uint32_t v[32], x[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), v);
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(N_TILE + c * 32), x);
          tmem_ld_wait();
          const int n = n0 + c * 32;
          if (!row.valid || n >= p.N) continue;
          tc_store_chunk_lean(p, row, n, v, x, unscale, floor_v);
        }
      } else {
#pragma unroll 1
        for (int c = grp; c < N_TILE / 32; c += epi_groups) {
          uint32_t v[32], x[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), v);
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(N_TILE + c * 32), x);
          tmem_ld_wait();
          const int n = n0 + c * 32;
          if (!row.valid || n >= p.N) continue;
          float f[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = (__uint_as_float(v[j]) + __uint_as_float(x[j])) * unscale;
          tc_store_chunk(p, row, n, f, z);
        }
      }
      if (!released) {
        tc_fence_before();                                      // this warp's TMEM reads are complete
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(empty_addr);
      }
      if (sch.trace && blockIdx.x == 0 && threadIdx.x == 128 && tl < 16) sch.trace[392 + tl * 4 + 3] = clock64();
    }
    if (lane == 0) bulk_wait_all();                               // this warp's tensor stores have landed before the CTA exits
  }
  if (sch.trace && blockIdx.x == 0 && threadIdx.x == 128) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    sch.trace[386] = clock64(); sch.trace[387] = (long long)gt;
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2sm<512>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------- packing kernels
namespace {

// W fp32 [taps][Cin][Cout] (HWIO flattened) -> Wp_{hi,lo} fp16 [Cout][taps*Cin], value scaled by `scale`
__global__ void pack_weights_kernel(const float* __restrict__ w, int taps, int cin, int cout, float scale, __half* __restrict__ hi,
                                    __half* __restrict__ lo, unsigned* __restrict__ range_flag, unsigned range_bit) {
  __shared__ float tile[32][33];
  const int tap = blockIdx.z;
  const int ci0 = blockIdx.y * 32, co0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int ci = ci0 + i, co = co0 + threadIdx.x;
    tile[i][threadIdx.x] = (ci < cin && co < cout) ? w[((long long)tap * cin + ci) * cout + co] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int co = co0 + i, ci = ci0 + threadIdx.x;
    if (co < cout && ci < cin) {
      __half h, l;
      const float v = tile[threadIdx.x][i] * scale;
      if (range_flag != nullptr && !(fabsf(v) < TC_F16_OVERFLOW)) atomicOr(range_flag, range_bit);
      split_f16(v, h, l);
      const long long o = (long long)co * taps * cin + (long long)tap * cin + ci;
      hi[o] = h;
      lo[o] = l;
    }
  }
}

// (hi, lo) fp16 activations -> fp32 NHWC (undoing the space-to-depth layout and the scale); debug / test visibility only
__global__ void unpack_act_kernel(const __half* __restrict__ hi, const __half* __restrict__ lo, int B, int H, int W, int C, int s2d,
                                  float inv_scale, float* __restrict__ out) {
  const long long total = (long long)B * H * W * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    long long r = i / C;
    const int w = (int)(r % W); r /= W;
    const int h = (int)(r % H);
    const int b = (int)(r / H);
    long long src = i;
    if (s2d) src = ((long long)(b * (H >> 1) + (h >> 1)) * (W >> 1) + (w >> 1)) * (4LL * C) + (((h & 1) << 1) | (w & 1)) * C + c;
    out[i] = (__half2float(hi[src]) + __half2float(lo[src])) * inv_scale;
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------- encoder plan
namespace {

// Split-K forward of a conv layer at small batch: the GEMM leaves fp32 partial sums [splits][M][N] (OUT_F32); this kernel folds
// them in a fixed order and applies the layer's real epilogue -- bias, ReLU, range guard, (hi, lo) split, store in the next
// layer's layout (tc_store_chunk's OUT_S2D_SPLIT / OUT_PLAIN_SPLIT branch).  One thread per (row, 8 columns).
__global__ void __launch_bounds__(256) splitk_forward_finish_kernel(const float* __restrict__ partials, int splits, const TcGemmParams p) {
  const long long groups = (long long)p.M * (p.N >> 3);
  for (long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x; gi < groups; gi += (long long)gridDim.x * blockDim.x) {
    const int m = (int)(gi / (p.N >> 3)), n = (int)(gi - (long long)m * (p.N >> 3)) << 3;
    float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const float* src = partials + (long long)m * p.N + n;
    for (int sp = 0; sp < splits; ++sp, src += (long long)p.M * p.N) {
      const float4 a = *reinterpret_cast<const float4*>(src), b = *reinterpret_cast<const float4*>(src + 4);
      f[0] += a.x; f[1] += a.y; f[2] += a.z; f[3] += a.w; f[4] += b.x; f[5] += b.y; f[6] += b.z; f[7] += b.w;
    }
    float amax = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = f[j] + (p.bias ? __ldg(p.bias + n + j) : 0.f);
      if (p.relu == 1) v = fmaxf(v, 0.f);
      amax = fmaxf(amax, fabsf(v));
      f[j] = v * p.out_scale;
    }
    if (p.range_flag != nullptr && !(amax * p.out_scale < TC_F16_OVERFLOW)) atomicOr(p.range_flag, p.range_bit);
    const TcRow r = tc_decode_row(p, m);
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) split_f16x2(f[2 * j], f[2 * j + 1], hi[j], lo[j]);
    *reinterpret_cast<uint4*>(p.out_hi + r.row_off + n) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(p.out_lo + r.row_off + n) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

int launch_tc_gemm2(const TcLayer& L, dim3 grid, cudaStream_t s) {
  using S = TcSmem2;
  TcTileSched sch;
  sch.m_pairs = (int)((grid.x + 1) / 2); sch.n_tiles = (int)grid.y; sch.splits = (int)grid.z;
  static long long* trace_dev = nullptr;
  sch.trace = nullptr;
  if (getenv("AAE_TC_TRACE")) {
    if (!trace_dev) { cudaMalloc(&trace_dev, (96 * 4 + 8 + 64 + 64) * sizeof(long long)); }
    cudaMemsetAsync(trace_dev, 0, (96 * 4 + 8 + 64 + 64) * sizeof(long long), s);
    sch.trace = trace_dev;
  }
  const int tiles = sch.m_pairs * sch.n_tiles * sch.splits;
  auto pk = tc_gemm2p_kernel;
  // TMA-store epilogue: 4 KB of staging per epilogue warp behind the ring.  With six 32 KB stages that leaves room for eight
  // epilogue warps (384 threads); the branch-free epilogue is no longer issue-bound, so eight are enough.
  // AAE_TC_NO_TMA_OUT=1 (read per launch) selects the plain-store epilogue: the reference the TMA-store epilogue is tested against
  const char* no_tma = getenv("AAE_TC_NO_TMA_OUT");
  const bool tma_out_on = !(no_tma && no_tma[0] == '1');
  constexpr int EPI_TMA = 8;                                     // epilogue warps the staging has room for
  static_assert(S::STAGES * S::STAGE_BYTES + 2048 + EPI_TMA * 4096 <= 232448, "TMA-store staging does not fit behind the ring");
  const bool f32_target_ok = L.gp.out_mode != OUT_F32 || (sch.splits == 1 && L.gp.out_f32 == L.tma_f32_base);
  const bool tma_out = tma_out_on && L.tma_out && f32_target_ok;
  const int threads = tma_out ? 128 + 32 * EPI_TMA : TC_THREADS;
  const int smem_bytes = tma_out ? S::STAGES * S::STAGE_BYTES + 2048 + EPI_TMA * 4096 : S::TOTAL;
  sch.tma_out = !tma_out ? 0 : L.gp.out_mode == OUT_S2D_SPLIT ? 1 : L.gp.out_mode == OUT_PLAIN_SPLIT ? 2 : L.gp.out_mode == OUT_D2S_SPLIT ? 3 : 4;
  AAE_CUDA_OK(cudaFuncSetAttribute(pk, cudaFuncAttributeMaxDynamicSharedMemorySize, std::max(smem_bytes, (int)S::TOTAL)));
  static int pair_slots = 0;                       // CTA pairs that can be resident at once (asked from the driver: pairs cannot straddle GPCs)
  if (pair_slots == 0) {
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(2u * (unsigned)std::max(1, sms / 2));
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = (size_t)std::max(smem_bytes, (int)S::TOTAL);
    cudaLaunchAttribute at;
    at.id = cudaLaunchAttributeClusterDimension;
    at.val.clusterDim.x = 2; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
    cfg.attrs = &at; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, pk, &cfg) != cudaSuccess || n <= 0) { cudaGetLastError(); n = std::max(1, sms / 2); }
    pair_slots = std::min(n, std::max(1, sms / 2));
    if (getenv("AAE_TC_VERBOSE")) fprintf(stderr, "[tc] CTA pairs resident at once: %d (of %d SMs / 2 = %d)\n", n, sms, sms / 2);
  }
  pk<<<dim3(2u * (unsigned)std::min(tiles, pair_slots)), threads, smem_bytes, s>>>(L.tm_a_hi, L.tm_a_lo, L.tm_w2_hi, L.tm_w2_lo,
                                                                                 tma_out ? L.tm_o_hi : L.tm_a_hi, tma_out ? L.tm_o_lo : L.tm_a_lo, L.gp, sch);
  AAE_LAUNCH_OK();
  if (sch.trace) {
    long long t[96 * 4 + 8 + 64 + 64];
    cudaStreamSynchronize(s);
    cudaMemcpy(t, sch.trace, sizeof(t), cudaMemcpyDeviceToHost);
    fprintf(stderr, "[gemm2p trace] N=%d taps=%d chunks/tap=%d: chunk: issue | +full seen | +mma issued | next-use empty seen (clocks, relative to chunk 0 issue)\n", L.gp.N, L.gp.taps, L.gp.chunks_per_tap);
    fprintf(stderr, "  CTA 0 (epilogue warp 4): %lld cycles in %lld ns -> SM clock %.0f MHz during this kernel\n", t[386] - t[384], t[387] - t[385],
            1e3 * (double)(t[386] - t[384]) / (double)(t[387] - t[385]));
    for (int k = 0; k < 4; ++k)
      fprintf(stderr, "  tile 1, warp 4, chunk round %d: tcgen05.ld %lld | math %lld | wait for buffer %lld | STS + proxy fence %lld | TMA issue %lld | (next round starts +%lld)\n", k,
              t[456 + k * 8 + 1] - t[456 + k * 8], t[456 + k * 8 + 2] - t[456 + k * 8 + 1], t[456 + k * 8 + 3] - t[456 + k * 8 + 2],
              t[456 + k * 8 + 4] - t[456 + k * 8 + 3], t[456 + k * 8 + 5] - t[456 + k * 8 + 4], k < 3 ? t[456 + (k + 1) * 8] - t[456 + k * 8 + 5] : 0LL);
    for (int tl = 0; tl < 15; ++tl)
      fprintf(stderr, "  tile %2d: epilogue warp 4 sees accumulators at %8lld, done +%6lld | issuer waits for drained TMEM from %8lld for %6lld\n", tl,
              t[392 + tl * 4 + 2] - t[384], t[392 + tl * 4 + 3] - t[392 + tl * 4 + 2], t[392 + tl * 4 + 0] - t[384], t[392 + tl * 4 + 1] - t[392 + tl * 4 + 0]);
    for (int g = 0; g < 96; g += (g < 8 ? 1 : 16))
      fprintf(stderr, "  g=%2d issue %7lld | full +%5lld | mma issued +%5lld | empty seen +%5lld\n", g, t[g * 4] - t[0], t[g * 4 + 1] - t[g * 4], t[g * 4 + 2] - t[g * 4],
              t[g * 4 + 3] - t[g * 4]);
  }
  return AAE_OK;
}

template <int N_TILE, int STAGES, int KCH>
int launch_tc_gemm(const TcLayer& L, dim3 grid, cudaStream_t s) {
  using S = TcSmem<N_TILE, STAGES, KCH>;
  auto kern = tc_gemm_kernel<N_TILE, STAGES, KCH>;
  AAE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
  kern<<<grid, TC_THREADS, S::TOTAL, s>>>(L.tm_a_hi, L.tm_a_lo, L.tm_w_hi, L.tm_w_lo, L.gp);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

int dev_alloc(void** p, size_t bytes) { return tc_dev_alloc(p, bytes); }

bool pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

}  // namespace

int tc_dev_alloc(void** p, size_t bytes) {
  cudaError_t e = cudaMalloc(p, bytes);
  if (e != cudaSuccess) { *p = nullptr; set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); return AAE_ERR_OOM; }
  cudaMemset(*p, 0, bytes);
  return AAE_OK;
}

int tc_launch_layer(const TcLayer& T, dim3 grid, cudaStream_t s) {
  if (T.pair && T.kch == 32) return launch_tc_gemm2(T, grid, s);
  if (T.n_tile == 256 && T.kch == 32) return launch_tc_gemm<256, 4, 32>(T, grid, s);
  if (T.n_tile == 128 && T.kch == 64) return launch_tc_gemm<128, 3, 64>(T, grid, s);
  if (T.n_tile == 32 && T.kch == 32) return launch_tc_gemm<32, 6, 32>(T, grid, s);
  set_error("tc_launch_layer: no kernel for n_tile=%d kch=%d", T.n_tile, T.kch);
  return AAE_ERR_UNSUPPORTED;
}

int tc_layer_setup_out_maps(TcLayer& T, long long out_rows_pad) {
  const TcGemmParams& g = T.gp;
  const uint64_t OH = (uint64_t)g.OH, OW = (uint64_t)g.OW, R = (uint64_t)out_rows_pad;
  T.tma_out = false;
  if (OH * OW < 32 && g.out_mode != OUT_F32) return AAE_OK;
  const uint32_t rows = OW >= 32 ? 1u : (uint32_t)(32 / std::max<uint64_t>(OW, 1));   // image rows covered by 32 consecutive pixels
  if (g.out_mode == OUT_F32) {                       // fp32 [rows, N] seen as fp16 [rows, 2N]: box = 32 rows x 32 floats (128-byte rows)
    const uint64_t dims[2] = {2ull * g.N, R};
    const uint64_t strides[1] = {4ull * g.N};
    const uint32_t box[2] = {64, 32};
    AAE_TRY(make_tmap_f16(&T.tm_o_hi, g.out_f32, 2, dims, strides, box, 128));
    T.tm_o_lo = T.tm_o_hi;
    T.tma_f32_base = g.out_f32;
  } else if (g.out_mode == OUT_PLAIN_SPLIT) {
    const uint64_t C = (uint64_t)g.N;
    const uint64_t dims[2] = {C, R * OH * OW};
    const uint64_t strides[1] = {C * 2};
    const uint32_t box[2] = {32, 32};
    AAE_TRY(make_tmap_f16(&T.tm_o_hi, g.out_hi, 2, dims, strides, box, 64));
    AAE_TRY(make_tmap_f16(&T.tm_o_lo, g.out_lo, 2, dims, strides, box, 64));
  } else if (g.out_mode == OUT_S2D_SPLIT) {
    // [image, row/2, column/2, (row parity, column parity), channel] seen as {channel, column parity, column/2, row parity, image*OH/2 + row/2}
    const uint64_t C = (uint64_t)g.N;
    if (OW < 2 || (rows > 1 && ((rows & 1) || OH % rows != 0))) return AAE_OK;
    const uint64_t dims[5] = {C, 2, OW / 2, 2, R * (OH / 2)};
    const uint64_t strides[4] = {C * 2, 4 * C * 2, 2 * C * 2, (OW / 2) * 4 * C * 2};
    const uint32_t box[5] = {32, 2, (uint32_t)std::min<uint64_t>(16, OW / 2), rows > 1 ? 2u : 1u, rows > 1 ? rows / 2 : 1u};
    AAE_TRY(make_tmap_f16(&T.tm_o_hi, g.out_hi, 5, dims, strides, box, 64));
    AAE_TRY(make_tmap_f16(&T.tm_o_lo, g.out_lo, 5, dims, strides, box, 64));
  } else if (g.out_mode == OUT_D2S_SPLIT) {
    // [image, 2 row + y parity, 2 column + x parity, channel] seen as {channel, x parity, column, y parity, image*OH + row}
    const uint64_t cq = (uint64_t)g.N / 4;
    if (cq < 32 || cq % 32 != 0 || OH % rows != 0) return AAE_OK;
    const uint64_t dims[5] = {cq, 2, OW, 2, R * OH};
    const uint64_t strides[4] = {cq * 2, 2 * cq * 2, 2 * OW * cq * 2, 4 * OW * cq * 2};
    const uint32_t box[5] = {32, 1, (uint32_t)std::min<uint64_t>(32, OW), 1, rows};
    AAE_TRY(make_tmap_f16(&T.tm_o_hi, g.out_hi, 5, dims, strides, box, 64));
    AAE_TRY(make_tmap_f16(&T.tm_o_lo, g.out_lo, 5, dims, strides, box, 64));
  } else {
    return AAE_OK;
  }
  T.tma_out = true;
  return AAE_OK;
}

int tc_encoder_create(int device, const aae_net_cfg* cfg, TcEncoder** out) {
  *out = nullptr;
  const int L = cfg->num_layers;
  AAE_REQUIRE(aae_device_supported(device), "AAE_PREC_TC_SPLIT needs a compute-capability 10.x device (tcgen05/TMEM)");
  AAE_REQUIRE(L >= 2, "AAE_PREC_TC_SPLIT: at least two conv layers expected");
  TcEncoder* h = new TcEncoder();
  h->device = device;
  h->cfg = *cfg;
  int ih = (cfg->in_h + cfg->strides[0] - 1) / cfg->strides[0], iw = (cfg->in_w + cfg->strides[0] - 1) / cfg->strides[0], ic = cfg->filters[0];
  const int B = cfg->max_batch;
  int st = AAE_OK;
  for (int l = 1; l <= L && st == AAE_OK; ++l) {
    TcLayer T;
    memset(&T.gp, 0, sizeof(T.gp));
    const bool dense = (l == L);
    if (!dense) {
      if (cfg->strides[l] != 2 || cfg->kernel_size != 5 || (ih & 1) || (iw & 1) || ic % 64 != 0 || cfg->filters[l] % 32 != 0) {
        set_error("AAE_PREC_TC_SPLIT: layer %d unsupported (needs k=5, stride 2, even dims, Cin %% 64 == 0, Cout %% 32 == 0)", l);
        st = AAE_ERR_UNSUPPORTED;
        break;
      }
      T.in_h = ih; T.in_w = iw; T.in_c = ic;
      T.out_h = ih / 2; T.out_w = iw / 2; T.out_c = cfg->filters[l];
      T.taps = 25;
      if (!pow2(T.out_w) || !pow2(T.out_h) || T.out_w > 128) { set_error("AAE_PREC_TC_SPLIT: output dims must be powers of two <= 128"); st = AAE_ERR_UNSUPPORTED; break; }
      T.BW = T.out_w;
      T.BH = std::min(T.out_h, 128 / T.BW);
      T.BB = 128 / (T.BW * T.BH);
    } else {
      T.in_h = T.in_w = 1; T.in_c = ih * iw * ic;
      T.out_h = T.out_w = 1; T.out_c = cfg->latent;
      T.taps = 1; T.BW = 1; T.BH = 1; T.BB = 128;
      h->flat = T.in_c;
      if (T.in_c % 64 != 0 || T.out_c % 32 != 0) { set_error("AAE_PREC_TC_SPLIT: dense layer needs flat %% 64 == 0 and latent %% 32 == 0"); st = AAE_ERR_UNSUPPORTED; break; }
    }
    T.n_tile = T.out_c >= 256 ? 256 : 128;
    T.kch = T.n_tile == 256 ? 32 : 64;
    // batch dimension padded to a whole number of TMA boxes, so a tile never addresses rows outside the tensor map
    const int B_pad = (int)ceil_div(B, T.BB) * T.BB;
    const size_t act_alloc = (size_t)B_pad * T.in_h * T.in_w * T.in_c;
    if ((st = dev_alloc((void**)&T.in_hi, act_alloc * sizeof(__half))) != AAE_OK) break;
    if ((st = dev_alloc((void**)&T.in_lo, act_alloc * sizeof(__half))) != AAE_OK) break;
    const size_t w_elems = (size_t)T.out_c * T.taps * T.in_c;
    if ((st = dev_alloc((void**)&T.w_hi, w_elems * sizeof(__half))) != AAE_OK) break;
    if ((st = dev_alloc((void**)&T.w_lo, w_elems * sizeof(__half))) != AAE_OK) break;
    // ---- tensor maps ----
    if (!dense) {
      const uint64_t C4 = 4ull * T.in_c, W2 = T.in_w / 2, H2 = T.in_h / 2;
      const uint64_t dims[4] = {C4, W2, H2, (uint64_t)B_pad};
      const uint64_t strides[3] = {C4 * 2, W2 * C4 * 2, H2 * W2 * C4 * 2};
      const uint32_t box[4] = {(uint32_t)T.kch, (uint32_t)T.BW, (uint32_t)T.BH, (uint32_t)T.BB};
      const int swz = 2 * T.kch;
      if ((st = make_tmap_f16(&T.tm_a_hi, T.in_hi, 4, dims, strides, box, swz)) != AAE_OK) break;
      if ((st = make_tmap_f16(&T.tm_a_lo, T.in_lo, 4, dims, strides, box, swz)) != AAE_OK) break;
    } else {
      const uint64_t dims[4] = {(uint64_t)T.in_c, 1, 1, (uint64_t)B_pad};
      const uint64_t strides[3] = {(uint64_t)T.in_c * 2, (uint64_t)T.in_c * 2, (uint64_t)T.in_c * 2};
      const uint32_t box[4] = {(uint32_t)T.kch, 1, 1, 128};
      if ((st = make_tmap_f16(&T.tm_a_hi, T.in_hi, 4, dims, strides, box, 2 * T.kch)) != AAE_OK) break;
      if ((st = make_tmap_f16(&T.tm_a_lo, T.in_lo, 4, dims, strides, box, 2 * T.kch)) != AAE_OK) break;
    }
    {
      const uint64_t K = (uint64_t)T.taps * T.in_c;
      const uint64_t dims[2] = {K, (uint64_t)T.out_c};
      const uint64_t strides[1] = {K * 2};
      const uint32_t box[2] = {(uint32_t)T.kch, (uint32_t)std::min(T.n_tile, T.out_c)};
      if ((st = make_tmap_f16(&T.tm_w_hi, T.w_hi, 2, dims, strides, box, 2 * T.kch)) != AAE_OK) break;
      if ((st = make_tmap_f16(&T.tm_w_lo, T.w_lo, 2, dims, strides, box, 2 * T.kch)) != AAE_OK) break;
      T.pair = !dense && T.n_tile == 256 && T.out_c % 256 == 0;
      if (T.pair) {
        const uint32_t box2[2] = {(uint32_t)T.kch, 128};
        const int swz2 = 2 * T.kch;
        if ((st = make_tmap_f16(&T.tm_w2_hi, T.w_hi, 2, dims, strides, box2, swz2)) != AAE_OK) break;
        if ((st = make_tmap_f16(&T.tm_w2_lo, T.w_lo, 2, dims, strides, box2, swz2)) != AAE_OK) break;
      }
    }
    // ---- static GEMM parameters ----
    TcGemmParams& g = T.gp;
    g.N = T.out_c; g.OH = T.out_h; g.OW = T.out_w; g.BW = T.BW; g.BH = T.BH;
    g.taps = T.taps; g.chunks_per_tap = T.in_c / T.kch;
    g.iters_per_split = g.taps * g.chunks_per_tap;
    for (int t = 0; t < T.taps; ++t) {
      if (dense) { g.tap_di[t] = 0; g.tap_dj[t] = 0; g.tap_ch[t] = 0; continue; }
      const int kh = t / 5, kw = t % 5;
      // input row 2*oh + kh - 1 (TF SAME pads 1 before): block offset (kh+1)/2 - 1, parity (kh+1) % 2
      g.tap_di[t] = (int8_t)((kh + 1) / 2 - 1);
      g.tap_dj[t] = (int8_t)((kw + 1) / 2 - 1);
      g.tap_ch[t] = ((((kh + 1) & 1) << 1) | ((kw + 1) & 1)) * T.in_c;
    }
    g.unscale = 1.f / (ACT_SCALE * W_SCALE);
    g.out_scale = ACT_SCALE;
    g.relu = dense ? 0 : 1;
    h->layers.push_back(T);
    if (!dense) { ih = T.out_h; iw = T.out_w; ic = T.out_c; }
  }
  if (st == AAE_OK) {
    // wire outputs: layer i writes the input buffers of layer i+1; the last conv writes plain NHWC (the flatten order)
    for (size_t i = 0; i + 1 < h->layers.size(); ++i) {
      TcGemmParams& g = h->layers[i].gp;
      g.out_hi = h->layers[i + 1].in_hi;
      g.out_lo = h->layers[i + 1].in_lo;
      g.out_mode = (i + 2 == h->layers.size()) ? OUT_PLAIN_SPLIT : OUT_S2D_SPLIT;
      if (h->layers[i].pair && (st = tc_layer_setup_out_maps(h->layers[i], (long long)ceil_div(B, h->layers[i + 1].BB) * h->layers[i + 1].BB)) != AAE_OK) break;
    }
    TcLayer& D = h->layers.back();
    const int total = D.gp.taps * D.gp.chunks_per_tap;
    h->dense_splits = std::min(total, 74);
    D.gp.iters_per_split = (total + h->dense_splits - 1) / h->dense_splits;
    h->dense_splits = (total + D.gp.iters_per_split - 1) / D.gp.iters_per_split;
    D.gp.out_mode = OUT_F32;
    st = dev_alloc((void**)&h->partials, (size_t)h->dense_splits * (B + 128) * cfg->latent * sizeof(float));
    D.gp.out_f32 = h->partials;
  }
  if (st == AAE_OK) st = dev_alloc((void**)&h->range_flag, sizeof(unsigned));
  if (st == AAE_OK)
    for (size_t i = 0; i + 1 < h->layers.size(); ++i) {   // layers[i] writes the activation of conv layer i + 1 (0-based); the dense layer writes fp32
      h->layers[i].gp.range_flag = h->range_flag;
      h->layers[i].gp.range_bit = 1u << (i + 1);
    }
  if (st == AAE_OK && tc_conv1_supported(cfg)) st = tc_conv1_create(device, cfg, &h->conv1);
  if (st != AAE_OK) { tc_encoder_destroy(h); return st; }
  *out = h;
  return AAE_OK;
}

void tc_encoder_destroy(TcEncoder* h) {
  if (!h) return;
  for (auto& T : h->layers) { cudaFree(T.in_hi); cudaFree(T.in_lo); cudaFree(T.w_hi); cudaFree(T.w_lo); }
  cudaFree(h->partials);
  cudaFree(h->fwd_partials);
  cudaFree(h->dbg);
  cudaFree(h->range_flag);
  tc_conv1_destroy(h->conv1);
  for (auto e : h->ev) cudaEventDestroy(e);
  delete h;
}

int tc_encoder_pack_weights(TcEncoder* h, int layer, const float* w_dev, cudaStream_t s) {
  if (layer == 0) {
    if (h->conv1) return tc_conv1_pack(h->conv1, w_dev, h->cfg.kernel_size * h->cfg.kernel_size * h->cfg.in_c, W_SCALE, h->range_flag, 1u << 16, s);
    return AAE_OK;  // conv1 on the fp32 SIMT kernel
  }
  AAE_REQUIRE(layer >= 1 && layer <= (int)h->layers.size(), "tc pack: layer %d out of range", layer);
  TcLayer& T = h->layers[layer - 1];
  dim3 grid((unsigned)ceil_div(T.out_c, 32), (unsigned)ceil_div(T.in_c, 32), (unsigned)T.taps), block(32, 8);
  pack_weights_kernel<<<grid, block, 0, s>>>(w_dev, T.taps, T.in_c, T.out_c, W_SCALE, T.w_hi, T.w_lo, h->range_flag, 1u << (16 + layer));
  AAE_LAUNCH_OK();
  return AAE_OK;
}

unsigned* tc_encoder_range_flag(TcEncoder* h) { return h->range_flag; }
unsigned* tc_decoder_range_flag(TcDecoder* h) { return h->range_flag; }

void tc_encoder_enable_timer(TcEncoder* h, bool on) { h->timer_on = on; }

static void tc_mark(TcEncoder* h, cudaStream_t s) {
  if (!h->timer_on) return;
  if (h->ev_used == (int)h->ev.size()) { cudaEvent_t e; if (cudaEventCreate(&e) != cudaSuccess) return; h->ev.push_back(e); }
  cudaEventRecord(h->ev[h->ev_used++], s);
}

int tc_encoder_read_timer(TcEncoder* h, float* ms, int cap) {
  int n = 0;
  if (h->ev_used >= 2) {
    cudaEventSynchronize(h->ev[h->ev_used - 1]);
    for (int i = 0; i + 1 < h->ev_used && n < cap; ++i, ++n) cudaEventElapsedTime(&ms[n], h->ev[i], h->ev[i + 1]);
  }
  return n;
}

int tc_encoder_forward(TcEncoder* h, const void* crops, int src_u8, int B, const float* w0, const float* b0, const float* dense_b,
                       float* z_out, cudaStream_t s) {
  const aae_net_cfg& cfg = h->cfg;
  h->ev_used = 0;
  tc_mark(h, s);
  if (h->conv1) {
    AAE_TRY(tc_conv1_forward(h->conv1, &cfg, crops, src_u8, B, b0, ACT_SCALE, W_SCALE, h->layers[0].in_hi, h->layers[0].in_lo, h->range_flag, s));
  } else {  // conv1 (Cin = 3, K = 75): fp32 SIMT implicit GEMM, epilogue writes conv2's space-to-depth (hi, lo) input directly
    IGemmParams p;
    memset(&p, 0, sizeof(p));
    p.src = crops; p.src_u8 = src_u8;
    p.B = B; p.SH = cfg.in_h; p.SW = cfg.in_w; p.SC = cfg.in_c;
    p.PH = h->layers[0].in_h; p.PW = h->layers[0].in_w;
    p.KH = p.KW = cfg.kernel_size; p.stride = cfg.strides[0];
    const int tot_h = std::max((p.PH - 1) * p.stride + p.KH - cfg.in_h, 0), tot_w = std::max((p.PW - 1) * p.stride + p.KW - cfg.in_w, 0);
    p.pad_t = tot_h / 2; p.pad_l = tot_w / 2;
    p.Bm = w0; p.N = cfg.filters[0]; p.bias = b0; p.act = ACT_RELU;
    p.M = B * p.PH * p.PW; p.K = p.KH * p.KW * p.SC;
    p.k_per_split = (int)ceil_div(p.K, 16) * 16;
    p.split_hi = h->layers[0].in_hi; p.split_lo = h->layers[0].in_lo; p.split_scale = ACT_SCALE; p.split_s2d = 1;
    AAE_TRY(launch_igemm(p, GATHER_FWD, s));
  }
  tc_mark(h, s);
  for (size_t i = 0; i < h->layers.size(); ++i) {
    TcLayer& T = h->layers[i];
    const bool dense = (i + 1 == h->layers.size());
    T.gp.M = dense ? B : B * T.out_h * T.out_w;
    dim3 grid((unsigned)ceil_div(T.gp.M, 128), (unsigned)ceil_div(T.out_c, T.n_tile), dense ? (unsigned)h->dense_splits : 1u);
    // Small batches leave most SM pairs idle (conv4 at 32 crops: 16 tiles of 400 K iterations for 74 pairs): split K so that the
    // persistent grid is covered, fold the fp32 partials and apply the real epilogue in splitk_forward_finish_kernel.
    int splits = 1;
    if (!dense && T.pair && T.gp.out_mode != OUT_F32) {
      const int tiles = (int)((grid.x + 1) / 2) * (int)grid.y, total_iters = T.gp.taps * T.gp.chunks_per_tap;
      if (tiles * 2 <= 74) {
        splits = std::min(74 / tiles, std::max(1, total_iters / 24));
        const size_t per_split = (size_t)T.gp.M * T.gp.N;
        if (per_split * (size_t)splits > h->fwd_partial_floats) {
          const size_t want = std::min<size_t>(per_split * (size_t)splits, (size_t)32 << 20);     // at most 128 MB of partials
          if (want > h->fwd_partial_floats) {
            cudaFree(h->fwd_partials);
            h->fwd_partials = nullptr; h->fwd_partial_floats = 0;
            AAE_TRY(dev_alloc((void**)&h->fwd_partials, want * sizeof(float)));
            h->fwd_partial_floats = want;
          }
          splits = (int)std::min<size_t>((size_t)splits, h->fwd_partial_floats / per_split);
        }
        splits = std::max(splits, 1);
      }
    }
    if (splits > 1) {
      TcLayer S = T;                                   // same operands and maps, partial sums out
      const int total_iters = T.gp.taps * T.gp.chunks_per_tap;
      S.gp.iters_per_split = (int)ceil_div(total_iters, splits);
      splits = (int)ceil_div(total_iters, S.gp.iters_per_split);
      S.gp.out_mode = OUT_F32;
      S.gp.out_f32 = h->fwd_partials;
      grid.z = (unsigned)splits;
      AAE_TRY(tc_launch_layer(S, grid, s));
      const long long groups = (long long)T.gp.M * (T.gp.N >> 3);
      splitk_forward_finish_kernel<<<(unsigned)std::min<long long>(148 * 8, ceil_div(groups, 256)), 256, 0, s>>>(h->fwd_partials, splits, T.gp);
      AAE_LAUNCH_OK();
    } else {
      AAE_TRY(tc_launch_layer(T, grid, s));
    }
    if (dense) AAE_TRY(launch_splitk_reduce(h->partials, h->dense_splits, (int64_t)B * cfg.latent, cfg.latent, dense_b, ACT_NONE, z_out, s));
    tc_mark(h, s);
  }
  return AAE_OK;
}

int tc_encoder_set_bias(TcEncoder* h, int layer, const float* bias_dev) {
  if (layer >= 1 && layer < (int)h->layers.size()) h->layers[layer - 1].gp.bias = bias_dev;
  return AAE_OK;
}

int tc_encoder_activation(TcEncoder* h, int layer, int B, const float** ptr, int64_t* count, cudaStream_t s) {
  // layer l's output is the input of TcLayer[l] (layers[] starts at conv index 1)
  AAE_REQUIRE(layer >= 0 && layer < (int)h->layers.size(), "tc activation: layer %d out of range", layer);
  const TcLayer& T = h->layers[layer];
  const bool plain = (layer + 1 == (int)h->layers.size());
  int H, W, C;
  if (plain) { const TcLayer& P = h->layers[layer - 1]; H = P.out_h; W = P.out_w; C = P.out_c; }
  else { H = T.in_h; W = T.in_w; C = T.in_c; }
  const size_t n = (size_t)B * H * W * C;
  if (h->dbg_floats < n) {
    cudaFree(h->dbg);
    h->dbg = nullptr;
    AAE_TRY(dev_alloc((void**)&h->dbg, n * sizeof(float)));
    h->dbg_floats = n;
  }
  unpack_act_kernel<<<1024, 256, 0, s>>>(T.in_hi, T.in_lo, B, H, W, C, plain ? 0 : 1, 1.f / ACT_SCALE, h->dbg);
  AAE_LAUNCH_OK();
  AAE_CUDA_OK(cudaStreamSynchronize(s));
  *ptr = h->dbg;
  *count = (int64_t)n;
  return AAE_OK;
}


// ================================================================================================= decoder plan
// Decoder.x (auto_pose/ae/decoder.py:36-84) on the tensor cores, in the sub-pixel form: dense 128 -> 8*8*512 (+ReLU), then
// every "nearest x2 upsample + conv5x5 (+ReLU)" as ONE GEMM  [B*h*w pixels] x [9*Cin] x [4*Cout]  over the LOW-resolution
// activation (plain NHWC (hi, lo) fp16, 3x3 taps as unit-stride TMA boxes) with the taps of the 5x5 kernel pre-summed per
// output parity; the epilogue scatters column (parity, co) of pixel (i, j) to pixel (2i+py, 2j+px) of the next layer's input
// (depth-to-space).  The output layer (Cout = 3 -> N = 12, padded to 32) applies the sigmoid and writes fp32 NHWC.
namespace {

__global__ void split_scale_kernel(const float* __restrict__ x, long long n, float scale, __half* __restrict__ hi, __half* __restrict__ lo,
                                   unsigned* __restrict__ range_flag, unsigned range_bit) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    __half h, l;
    if (range_flag != nullptr && !(fabsf(x[i] * scale) < TC_F16_OVERFLOW)) atomicOr(range_flag, range_bit);
    split_f16(x[i] * scale, h, l);
    hi[i] = h;
    lo[i] = l;
  }
}

// merged weights Wm [9][cin][n4] -> operand of the tap-separable output layer: row (tap * n4 + m) = Wm[tap][:, m], rows >= 9*n4 zero
__global__ void pack_out_sep_kernel(const float* __restrict__ wm, int cin, int n4, float scale, __half* __restrict__ hi, __half* __restrict__ lo,
                                    unsigned* __restrict__ range_flag, unsigned range_bit) {
  const int total = 128 * cin;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int ci = i % cin, n = i / cin;
    const int tap = n / n4, m = n - tap * n4;
    const float v = tap < 9 ? wm[((long long)tap * cin + ci) * n4 + m] * scale : 0.f;
    if (range_flag != nullptr && !(fabsf(v) < TC_F16_OVERFLOW)) atomicOr(range_flag, range_bit);
    __half a, d;
    split_f16(v, a, d);
    hi[i] = a;
    lo[i] = d;
  }
}

// x[b, 2i+py, 2j+px, co] = sigmoid(bias[co] + sum_{tap=(ty,tx)} P[(b, i+ty-1, j+tx-1)][tap*4c + (py*2+px)*c + co]); one thread per output value
__global__ void outlayer_gather_kernel(const float* __restrict__ P, const float* __restrict__ bias, int B, int h, int w, int c,
                                       float* __restrict__ x) {
  const int n4 = 4 * c;
  const long long total = (long long)B * h * w * n4;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int m = (int)(t % n4);
    long long r = t / n4;
    const int j = (int)(r % w); r /= w;
    const int i = (int)(r % h);
    const long long b = r / h;
    const int cls = m / c, co = m - cls * c;
    float s = bias ? __ldg(bias + co) : 0.f;
#pragma unroll
    for (int ty = 0; ty < 3; ++ty) {
      const int ii = i + ty - 1;
      if (ii < 0 || ii >= h) continue;
#pragma unroll
      for (int tx = 0; tx < 3; ++tx) {
        const int jj = j + tx - 1;
        if (jj < 0 || jj >= w) continue;
        s += P[((b * h + ii) * w + jj) * 128 + (ty * 3 + tx) * n4 + m];
      }
    }
    x[((b * 2 * h + 2 * i + (cls >> 1)) * (2LL * w) + 2 * j + (cls & 1)) * c + co] = 1.f / (1.f + expf(-s));
  }
}

__global__ void tile_bias_kernel(const float* __restrict__ b, int cout, int n_pad, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_pad) out[i] = i < 4 * cout ? b[i % cout] : 0.f;
}

}  // namespace

int tc_layer_setup_plain(TcLayer& T, int B, bool pair_ok, bool alloc_input) {
  int st;
  const int B_pad = (int)ceil_div(B, T.BB) * T.BB;
  const size_t act = (size_t)B_pad * T.in_h * T.in_w * T.in_c;
  if (alloc_input) {
    if ((st = dev_alloc((void**)&T.in_hi, act * sizeof(__half))) != AAE_OK) return st;
    if ((st = dev_alloc((void**)&T.in_lo, act * sizeof(__half))) != AAE_OK) return st;
  }
  const uint64_t K = (uint64_t)T.taps * T.in_c;
  const int rows = (int)ceil_div(T.gp.N, T.n_tile) * T.n_tile;
  if ((st = dev_alloc((void**)&T.w_hi, (size_t)rows * K * sizeof(__half))) != AAE_OK) return st;
  if ((st = dev_alloc((void**)&T.w_lo, (size_t)rows * K * sizeof(__half))) != AAE_OK) return st;
  {
    const uint64_t dims[4] = {(uint64_t)T.in_c, (uint64_t)T.in_w, (uint64_t)T.in_h, (uint64_t)B_pad};
    const uint64_t strides[3] = {(uint64_t)T.in_c * 2, (uint64_t)T.in_w * T.in_c * 2, (uint64_t)T.in_h * T.in_w * T.in_c * 2};
    const uint32_t box[4] = {(uint32_t)T.kch, (uint32_t)T.BW, (uint32_t)T.BH, (uint32_t)T.BB};
    if ((st = make_tmap_f16(&T.tm_a_hi, T.in_hi, 4, dims, strides, box, 2 * T.kch)) != AAE_OK) return st;
    if ((st = make_tmap_f16(&T.tm_a_lo, T.in_lo, 4, dims, strides, box, 2 * T.kch)) != AAE_OK) return st;
  }
  {
    const uint64_t dims[2] = {K, (uint64_t)rows};
    const uint64_t strides[1] = {K * 2};
    const uint32_t box[2] = {(uint32_t)T.kch, (uint32_t)T.n_tile};
    if ((st = make_tmap_f16(&T.tm_w_hi, T.w_hi, 2, dims, strides, box, 2 * T.kch)) != AAE_OK) return st;
    if ((st = make_tmap_f16(&T.tm_w_lo, T.w_lo, 2, dims, strides, box, 2 * T.kch)) != AAE_OK) return st;
    T.pair = pair_ok && T.n_tile == 256 && T.gp.N % 256 == 0;
    if (T.pair) {
      const uint32_t box2[2] = {(uint32_t)T.kch, 128};
      if ((st = make_tmap_f16(&T.tm_w2_hi, T.w_hi, 2, dims, strides, box2, 2 * T.kch)) != AAE_OK) return st;
      if ((st = make_tmap_f16(&T.tm_w2_lo, T.w_lo, 2, dims, strides, box2, 2 * T.kch)) != AAE_OK) return st;
    }
  }
  return AAE_OK;
}

int tc_decoder_create(int device, const aae_net_cfg* cfg, TcDecoder** out) {
  *out = nullptr;
  AAE_REQUIRE(aae_device_supported(device), "AAE_PREC_TC_SPLIT needs a compute-capability 10.x device (tcgen05/TMEM)");
  const int L = cfg->num_layers;
  AAE_REQUIRE(cfg->kernel_size == 5 && cfg->in_h == cfg->in_w, "AAE_PREC_TC_SPLIT decoder: kernel 5, square crops");
  TcDecoder* h = new TcDecoder();
  h->device = device;
  h->cfg = *cfg;
  const int B = cfg->max_batch;
  int h0 = cfg->in_h;
  for (int i = 0; i < L; ++i) h0 /= 2;
  std::vector<int> nf(L);
  for (int i = 0; i < L; ++i) nf[i] = cfg->filters[L - 1 - i];
  int st = AAE_OK;
  for (int l = 0; l <= L && st == AAE_OK; ++l) {
    TcLayer T;
    memset(&T.gp, 0, sizeof(T.gp));
    TcGemmParams& g = T.gp;
    T.kch = 32;
    if (l == 0) {                                   // dense_1: [B, latent] x [latent, h0*h0*f0]
      T.in_h = T.in_w = 1; T.in_c = cfg->latent; T.out_h = T.out_w = 1; T.out_c = h0 * h0 * nf[0];
      T.taps = 1; T.BW = 1; T.BH = 1; T.BB = 128; T.n_tile = 256;
      g.N = T.out_c; g.OH = g.OW = 1; g.relu = 1; g.out_mode = OUT_PLAIN_SPLIT;
      if (cfg->latent % 32 != 0 || T.out_c % 256 != 0) { set_error("tc decoder: latent %% 32 and dense width %% 256 required"); st = AAE_ERR_UNSUPPORTED; break; }
    } else {                                        // sub-pixel conv on the (h x w x C) low-resolution activation
      const int hh = h0 << (l - 1);
      T.in_h = T.in_w = hh; T.in_c = nf[l - 1];
      const int cout = l < L ? nf[l] : cfg->in_c;
      T.out_h = T.out_w = 2 * hh; T.out_c = cout;
      T.taps = 9;
      if (hh > 128 || (hh & (hh - 1)) || T.in_c % 32 != 0 || (l < L && cout % 64 != 0)) {
        set_error("tc decoder: layer %d unsupported (power-of-two size <= 128, Cin %% 32, Cout %% 64)", l); st = AAE_ERR_UNSUPPORTED; break;
      }
      T.BW = hh; T.BH = std::min(hh, 128 / T.BW); T.BB = 128 / (T.BW * T.BH);
      g.OH = g.OW = hh;
      if (l < L) { g.N = 4 * cout; T.n_tile = 256; g.relu = 1; g.out_mode = OUT_D2S_SPLIT; }
      else if (36 * cout <= 128 && T.in_c % 64 == 0) {
        h->sep_out = true;                          // 1x1 GEMM into P, neighbourhood sum in outlayer_gather_kernel
        T.taps = 1; T.kch = 64; g.N = 128; T.n_tile = 128; g.relu = 0; g.out_mode = OUT_F32; g.cout_real = cout;
        st = dev_alloc((void**)&h->out_p, (size_t)ceil_div((int64_t)B * hh * hh, 128) * 128 * 128 * sizeof(float));
        if (st != AAE_OK) break;
      } else { g.N = 32; T.n_tile = 32; g.relu = 2; g.out_mode = OUT_D2S_F32; g.cout_real = cout;
             if (4 * cout > 32) { set_error("tc decoder: output channels > 8 unsupported"); st = AAE_ERR_UNSUPPORTED; break; } }
    }
    g.BW = T.BW; g.BH = T.BH; g.taps = T.taps; g.chunks_per_tap = T.in_c / T.kch;
    g.iters_per_split = g.taps * g.chunks_per_tap;
    for (int t = 0; t < T.taps; ++t) {
      g.tap_di[t] = (int8_t)(T.taps == 1 ? 0 : t / 3 - 1);
      g.tap_dj[t] = (int8_t)(T.taps == 1 ? 0 : t % 3 - 1);
      g.tap_ch[t] = 0;
    }
    g.unscale = 1.f / (ACT_SCALE * W_SCALE);
    g.out_scale = ACT_SCALE;
    if ((st = tc_layer_setup_plain(T, B, /*pair_ok=*/l > 0, /*alloc_input=*/true)) != AAE_OK) { h->layers.push_back(T); break; }
    h->layers.push_back(T);
    float* bz = nullptr;
    if (l > 0) st = dev_alloc((void**)&bz, (size_t)std::max(g.N, 32) * sizeof(float));
    h->bias_dev.push_back(bz);
    h->wm_floats = std::max(h->wm_floats, (size_t)9 * T.in_c * 4 * T.out_c);
  }
  if (st == AAE_OK) st = dev_alloc((void**)&h->wm_tmp, h->wm_floats * sizeof(float));
  if (st == AAE_OK) st = dev_alloc((void**)&h->range_flag, sizeof(unsigned));
  if (st == AAE_OK) {
    for (size_t i = 0; i + 1 < h->layers.size(); ++i) {
      h->layers[i].gp.out_hi = h->layers[i + 1].in_hi;
      h->layers[i].gp.out_lo = h->layers[i + 1].in_lo;
      h->layers[i].gp.range_flag = h->range_flag;       // bit i: the activation written by layer i (0 = dense_1)
      h->layers[i].gp.range_bit = 1u << i;
      if (h->layers[i].pair && h->layers[i].gp.out_mode == OUT_D2S_SPLIT &&
          (st = tc_layer_setup_out_maps(h->layers[i], (long long)ceil_div(B, h->layers[i + 1].BB) * h->layers[i + 1].BB)) != AAE_OK)
        break;
    }
  }
  if (st != AAE_OK) { tc_decoder_destroy(h); return st; }
  *out = h;
  return AAE_OK;
}

void tc_decoder_destroy(TcDecoder* h) {
  if (!h) return;
  for (auto& T : h->layers) { cudaFree(T.in_hi); cudaFree(T.in_lo); cudaFree(T.w_hi); cudaFree(T.w_lo); }
  for (auto b : h->bias_dev) cudaFree(b);
  cudaFree(h->wm_tmp);
  cudaFree(h->out_p);
  cudaFree(h->range_flag);
  delete h;
}

// layer 0: dense_1 kernel [latent, h0*w0*f0]; layers 1..L: conv kernels HWIO [5,5,cin,cout]; biases in the reference layout
int tc_decoder_pack_weights(TcDecoder* h, int layer, const float* w_dev, const float* b_dev, cudaStream_t s) {
  AAE_REQUIRE(layer >= 0 && layer < (int)h->layers.size(), "tc decoder pack: layer %d out of range", layer);
  TcLayer& T = h->layers[layer];
  dim3 block(32, 8);
  if (layer == 0) {
    if (w_dev) {
      dim3 grid((unsigned)ceil_div(T.out_c, 32), (unsigned)ceil_div(T.in_c, 32), 1);
      pack_weights_kernel<<<grid, block, 0, s>>>(w_dev, 1, T.in_c, T.out_c, W_SCALE, T.w_hi, T.w_lo, h->range_flag, 1u << 16);
      AAE_LAUNCH_OK();
    }
    if (b_dev) T.gp.bias = b_dev;      // device pointer owned by the decoder handle
    return AAE_OK;
  }
  const bool sep = h->sep_out && layer + 1 == (int)h->layers.size();
  if (w_dev) {
    AAE_TRY(launch_merge_subpixel_weights(w_dev, T.in_c, T.out_c, h->wm_tmp, s));
    if (sep) {
      pack_out_sep_kernel<<<64, 256, 0, s>>>(h->wm_tmp, T.in_c, 4 * T.out_c, W_SCALE, T.w_hi, T.w_lo, h->range_flag, 1u << (16 + layer));
    } else {
      dim3 grid((unsigned)ceil_div(4 * T.out_c, 32), (unsigned)ceil_div(T.in_c, 32), 9);
      pack_weights_kernel<<<grid, block, 0, s>>>(h->wm_tmp, 9, T.in_c, 4 * T.out_c, W_SCALE, T.w_hi, T.w_lo, h->range_flag, 1u << (16 + layer));
    }
    AAE_LAUNCH_OK();
  }
  if (sep) {
    if (b_dev) h->out_bias = b_dev;
    return AAE_OK;
  }
  if (b_dev) {
    const int n_pad = std::max(T.gp.N, 32);
    tile_bias_kernel<<<(unsigned)ceil_div(n_pad, 128), 128, 0, s>>>(b_dev, T.out_c, n_pad, h->bias_dev[layer]);
    AAE_LAUNCH_OK();
    T.gp.bias = h->bias_dev[layer];
  }
  return AAE_OK;
}

const float* tc_decoder_merged_weights(const TcDecoder* h) { return h->wm_tmp; }

int tc_decoder_forward(TcDecoder* h, const float* z_dev, int B, float* x_out, cudaStream_t s) {
  TcLayer& D = h->layers[0];
  split_scale_kernel<<<(unsigned)std::min<int64_t>(1024, ceil_div((int64_t)B * D.in_c, 256)), 256, 0, s>>>(z_dev, (long long)B * D.in_c, ACT_SCALE,
                                                                                                          D.in_hi, D.in_lo, h->range_flag, 1u << 15);
  AAE_LAUNCH_OK();
  for (size_t i = 0; i < h->layers.size(); ++i) {
    TcLayer& T = h->layers[i];
    T.gp.M = i == 0 ? B : B * T.in_h * T.in_w;
    const bool last = i + 1 == h->layers.size();
    if (last) T.gp.out_f32 = h->sep_out ? h->out_p : x_out;
    dim3 grid((unsigned)ceil_div(T.gp.M, 128), (unsigned)ceil_div(T.gp.N, T.n_tile), 1u);
    AAE_TRY(tc_launch_layer(T, grid, s));
    if (last && h->sep_out) {
      const long long total = (long long)T.gp.M * 4 * T.gp.cout_real;
      outlayer_gather_kernel<<<(unsigned)std::min<long long>(148 * 16, ceil_div(total, 256)), 256, 0, s>>>(h->out_p, h->out_bias, B, T.in_h, T.in_w,
                                                                                                         T.gp.cout_real, x_out);
      AAE_LAUNCH_OK();
    }
  }
  return AAE_OK;
}

}  // namespace aae
