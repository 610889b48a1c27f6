// Backward pass of the AAE training step on the tensor cores (AAE_PREC_TC_SPLIT trainer).
//
// Replaces the gradient sub-graph TensorFlow derives for auto_pose/ae/ae_factory.py:79-95 (build_train_op) over
// auto_pose/ae/encoder.py:37-68 and auto_pose/ae/decoder.py:36-84, for the conv layers with Cin >= 128.  Every such layer is
// one "unit" with two GEMMs, both in the same split-fp16 x3 arithmetic as the forward pass:
//
//   dgrad  dX = G (*) W'      a 3x3 unit-stride conv over the pre-activation gradient G of the layer's GEMM output
//                             (plain NHWC (hi, lo) fp16): the forward GEMM kernels (tc_gemm.cu) with re-packed weights.
//                               decoder sub-pixel layer: W'[ci][(tap', (cls,co))] = Wm[8 - tap'][ci][(cls,co)]
//                               encoder 5x5/s2 layer   : W'[(py,px,ci)][(tap', co)] = W[3 - 2ty + py][3 - 2tx + px][ci][co]  (0 outside 5x5)
//                             i.e. the transposed stride-2 conv is a 3x3 conv producing the space-to-depth form of dX.
//   wgrad  dW = X^T G         contraction over pixels: both operands are read straight from their NHWC tensors as
//                             MN-major tcgen05 operands (channels contiguous), no transposed copies (tc_wgrad_kernel).
//
// Gradients have no a-priori range, so every G tensor is stored as (hi, lo) fp16 of  G * 2^k  with k chosen per tensor and
// per step from its largest magnitude (tc_dyn_scale): dgrad/wgrad results are written as raw fp32, a small elementwise
// pass applies the ReLU mask of the forward activation, finds the maximum and re-splits into the next unit's layout.
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "tc.cuh"
#include "tc_common.cuh"
#include "tc_plan.cuh"

namespace aae {

using namespace tc;

// ------------------------------------------------------------------------------------------------- wgrad kernel
struct TcWgradParams {
  int cin_blocks;          // X channels / 128: blockIdx.x = tap * cin_blocks + channel block
  int OH, OW;              // pixel grid of the contraction (G's spatial dims)
  int BWk, BHk;            // pixel box of one K chunk (BWk * BHk = 32)
  int chunks_per_image;    // OH * OW / 32
  int total_chunks;        // B * chunks_per_image
  int chunks_per_split;    // K chunks per blockIdx.z
  int8_t tap_di[32], tap_dj[32];
  int tap_ch[32];          // channel offset of the tap's parity plane in X
  int m_tiles;             // taps * cin_blocks (the CTA-pair kernel pads an odd count with an idle CTA)
  TcGemmParams ep;         // epilogue: OUT_F32 partials [splits][taps*Cin][N]
};

template <int N_TILE, int STAGES>
struct WgSmem {
  static constexpr int KP = 32;                          // pixels per K chunk
  static constexpr int X_BYTES = 128 * KP * 2;           // two 64-channel boxes of KP rows x 128 B
  static constexpr int G_BYTES = N_TILE * KP * 2;
  static constexpr int STAGE_BYTES = 2 * X_BYTES + 2 * G_BYTES;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 + 256;
};

// MN-major operand in the 128-byte-swizzle canonical layout: K rows (pixels) of 128 B = 64 fp16 channels, 8-row groups SBO
// apart, successive 64-channel atoms LBO apart (cute::UMMA canonical ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units).
__device__ __forceinline__ uint64_t make_sw128_mnmajor_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

template <int N_TILE, int STAGES>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_wgrad_kernel(const __grid_constant__ CUtensorMap tm_x_hi, const __grid_constant__ CUtensorMap tm_x_lo,
                const __grid_constant__ CUtensorMap tm_g_hi, const __grid_constant__ CUtensorMap tm_g_lo, const TcWgradParams p) {
  using S = WgSmem<N_TILE, STAGES>;
  constexpr int BOX_BYTES = 64 * S::KP * 2;   // one TMA box: 64 channels x KP pixels
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * S::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tap = blockIdx.x / p.cin_blocks, cb = blockIdx.x - tap * p.cin_blocks;
  const int m0 = blockIdx.x * 128;
  const int n0 = blockIdx.y * N_TILE;
  const int q_begin = blockIdx.z * p.chunks_per_split;
  const int q_end = min(p.total_chunks, q_begin + p.chunks_per_split);

  if (warp == 0 && lane == 0) { prefetch_tmap(&tm_x_hi); prefetch_tmap(&tm_x_lo); prefetch_tmap(&tm_g_hi); prefetch_tmap(&tm_g_lo); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<2 * N_TILE>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      const int cols = p.OW / p.BWk;
      const int cx = p.tap_ch[tap] + cb * 128;
      const int di = p.tap_di[tap], dj = p.tap_dj[tap];
      for (int q = q_begin, i = 0; q < q_end; ++q, ++i) {
        const int s = i % STAGES;
        mbar_wait(&empty_bar[s], (((uint32_t)(i / STAGES)) & 1u) ^ 1u);
        const int b = q / p.chunks_per_image, r = q - b * p.chunks_per_image;
        const int y0 = (r / cols) * p.BHk, x0 = (r - (r / cols) * cols) * p.BWk;
        uint8_t* st = smem + s * S::STAGE_BYTES;
        mbar_arrive_expect_tx(&full_bar[s], S::STAGE_BYTES);
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          tma_load_4d(st + g * BOX_BYTES, &tm_x_hi, &full_bar[s], cx + 64 * g, x0 + dj, y0 + di, b);
          tma_load_4d(st + S::X_BYTES + g * BOX_BYTES, &tm_x_lo, &full_bar[s], cx + 64 * g, x0 + dj, y0 + di, b);
        }
#pragma unroll
        for (int g = 0; g < N_TILE / 64; ++g) {
          tma_load_4d(st + 2 * S::X_BYTES + g * BOX_BYTES, &tm_g_hi, &full_bar[s], n0 + 64 * g, x0, y0, b);
          tma_load_4d(st + 2 * S::X_BYTES + S::G_BYTES + g * BOX_BYTES, &tm_g_lo, &full_bar[s], n0 + 64 * g, x0, y0, b);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(128, N_TILE, 0) | (1u << 15) | (1u << 16);   // both operands MN-major
      for (int q = q_begin, i = 0; q < q_end; ++q, ++i) {
        const int s = i % STAGES;
        mbar_wait(&full_bar[s], ((uint32_t)(i / STAGES)) & 1u);
        tc_fence_after();
        const uint32_t st = smem_u32(smem + s * S::STAGE_BYTES);
#pragma unroll
        for (int k = 0; k < S::KP / 16; ++k) {
          const uint32_t ko = (uint32_t)k * 16u * 128u;   // 16 pixel rows of 128 B
          const uint64_t x_hi = make_sw128_mnmajor_desc(st + ko, BOX_BYTES, 1024);
          const uint64_t x_lo = make_sw128_mnmajor_desc(st + S::X_BYTES + ko, BOX_BYTES, 1024);
          const uint64_t g_hi = make_sw128_mnmajor_desc(st + 2 * S::X_BYTES + ko, BOX_BYTES, 1024);
          const uint64_t g_lo = make_sw128_mnmajor_desc(st + 2 * S::X_BYTES + S::G_BYTES + ko, BOX_BYTES, 1024);
          const uint32_t first = (i > 0 || k > 0) ? 1u : 0u;
          umma_f16(tmem_base, x_hi, g_hi, idesc, first);
          umma_f16(tmem_base + N_TILE, x_lo, g_hi, idesc, first);
          umma_f16(tmem_base + N_TILE, x_hi, g_lo, idesc, 1u);
        }
        umma_commit(&empty_bar[s]);
      }
      umma_commit(tmem_full_bar);
    }
  } else if (warp >= 4) {
    const int q4 = warp & 3, grp = (warp - 4) >> 2;   // TC_EPI_GROUPS warps per TMEM lane quadrant, interleaved 32-column chunks
    const TcRow row = tc_decode_row(p.ep, m0 + q4 * 32 + lane);
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    const bool has_work = q_end > q_begin;
    const float unscale = p.ep.amax_bits ? p.ep.unscale * tc_dyn_unscale(__ldg(p.ep.amax_bits)) : p.ep.unscale;
#pragma unroll 1
    for (int c = grp; c < N_TILE / 32; c += TC_EPI_GROUPS) {
      uint32_t v[32], x[32];
      tmem_ld_32x32(tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(c * 32), v);
      tmem_ld_32x32(tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(N_TILE + c * 32), x);
      tmem_ld_wait();
      const int n = n0 + c * 32;
      if (!row.valid || n >= p.ep.N) continue;
      float f[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) f[j] = has_work ? (__uint_as_float(v[j]) + __uint_as_float(x[j])) * unscale : 0.f;
      tc_store_chunk(p.ep, row, n, f, (int)blockIdx.z);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<2 * N_TILE>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------- wgrad on CTA pairs
// Same contraction with cta_group::2: two M tiles (consecutive (tap, channel-block) pairs) share one 256-column G tile and
// run as ONE M = 256 MMA; each CTA stages its own X tile and only HALF of the G tile (128 columns), i.e. 32 KB instead of
// 48 KB per K chunk, which is what bounds the single-CTA kernel (shared-memory bandwidth, see the pair kernel in tc_gemm.cu).
template <int STAGES>
struct WgSmem2 {
  static constexpr int KP = 32;
  static constexpr int T_BYTES = 128 * KP * 2;            // X tile and G half tile: 128 channels x KP pixels
  static constexpr int STAGE_BYTES = 4 * T_BYTES;         // X_hi, X_lo, G_hi(half), G_lo(half)
  static constexpr int TOTAL = STAGES * STAGE_BYTES + 1024 + 256;
};

template <int STAGES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
tc_wgrad2_kernel(const __grid_constant__ CUtensorMap tm_x_hi, const __grid_constant__ CUtensorMap tm_x_lo,
                 const __grid_constant__ CUtensorMap tm_g_hi, const __grid_constant__ CUtensorMap tm_g_lo, const TcWgradParams p) {
  using S = WgSmem2<STAGES>;
  constexpr int N_TILE = 256;
  constexpr int BOX_BYTES = 64 * S::KP * 2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * S::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  // an odd number of M tiles is padded to whole pairs: the extra CTA repeats the last tile's loads and writes nothing
  const int mt = min((int)blockIdx.x, p.m_tiles - 1);
  const int tap = mt / p.cin_blocks, cb = mt - tap * p.cin_blocks;
  const int m0 = blockIdx.x * 128;
  const int n0 = blockIdx.y * N_TILE;
  const int q_begin = blockIdx.z * p.chunks_per_split;
  const int q_end = min(p.total_chunks, q_begin + p.chunks_per_split);

  if (warp == 0 && lane == 0) { prefetch_tmap(&tm_x_hi); prefetch_tmap(&tm_x_lo); prefetch_tmap(&tm_g_hi); prefetch_tmap(&tm_g_lo); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2sm<512>(tmem_ptr);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      const int cols = p.OW / p.BWk;
      const int cx = p.tap_ch[tap] + cb * 128;
      const int di = p.tap_di[tap], dj = p.tap_dj[tap];
      const int gn = n0 + (int)rank * 128;
      for (int q = q_begin, i = 0; q < q_end; ++q, ++i) {
        const int s = i % STAGES;
        mbar_wait(&empty_bar[s], (((uint32_t)(i / STAGES)) & 1u) ^ 1u);
        const int b = q / p.chunks_per_image, r = q - b * p.chunks_per_image;
        const int y0 = (r / cols) * p.BHk, x0 = (r - (r / cols) * cols) * p.BWk;
        uint8_t* st = smem + s * S::STAGE_BYTES;
        if (leader) mbar_arrive_expect_tx(&full_bar[s], 2 * S::STAGE_BYTES);
        const uint32_t lb = leader_bar_addr(&full_bar[s]);
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          tma_load_4d_2sm(st + g * BOX_BYTES, &tm_x_hi, lb, cx + 64 * g, x0 + dj, y0 + di, b);
          tma_load_4d_2sm(st + S::T_BYTES + g * BOX_BYTES, &tm_x_lo, lb, cx + 64 * g, x0 + dj, y0 + di, b);
          tma_load_4d_2sm(st + 2 * S::T_BYTES + g * BOX_BYTES, &tm_g_hi, lb, gn + 64 * g, x0, y0, b);
          tma_load_4d_2sm(st + 3 * S::T_BYTES + g * BOX_BYTES, &tm_g_lo, lb, gn + 64 * g, x0, y0, b);
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(256, N_TILE, 0) | (1u << 15) | (1u << 16);
      for (int q = q_begin, i = 0; q < q_end; ++q, ++i) {
        const int s = i % STAGES;
        mbar_wait(&full_bar[s], ((uint32_t)(i / STAGES)) & 1u);
        tc_fence_after();
        const uint32_t st = smem_u32(smem + s * S::STAGE_BYTES);
#pragma unroll
        for (int k = 0; k < S::KP / 16; ++k) {
          const uint32_t ko = (uint32_t)k * 16u * 128u;
          const uint64_t x_hi = make_sw128_mnmajor_desc(st + ko, BOX_BYTES, 1024);
          const uint64_t x_lo = make_sw128_mnmajor_desc(st + S::T_BYTES + ko, BOX_BYTES, 1024);
          const uint64_t g_hi = make_sw128_mnmajor_desc(st + 2 * S::T_BYTES + ko, BOX_BYTES, 1024);
          const uint64_t g_lo = make_sw128_mnmajor_desc(st + 3 * S::T_BYTES + ko, BOX_BYTES, 1024);
          const uint32_t first = (i > 0 || k > 0) ? 1u : 0u;
          umma_f16_2sm(tmem_base, x_hi, g_hi, idesc, first);
          umma_f16_2sm(tmem_base + N_TILE, x_lo, g_hi, idesc, first);
          umma_f16_2sm(tmem_base + N_TILE, x_hi, g_lo, idesc, 1u);
        }
        umma_commit_2sm(&empty_bar[s]);
      }
      umma_commit_2sm(tmem_full_bar);
    }
  } else if (warp >= 4) {
    const int q4 = warp & 3, grp = (warp - 4) >> 2;   // TC_EPI_GROUPS warps per TMEM lane quadrant, interleaved 32-column chunks
    const TcRow row = tc_decode_row(p.ep, m0 + q4 * 32 + lane);
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    const float unscale = p.ep.amax_bits ? p.ep.unscale * tc_dyn_unscale(__ldg(p.ep.amax_bits)) : p.ep.unscale;
#pragma unroll 1
    for (int c = grp; c < N_TILE / 32; c += TC_EPI_GROUPS) {
      uint32_t v[32], x[32];
      tmem_ld_32x32(tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(c * 32), v);
      tmem_ld_32x32(tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(N_TILE + c * 32), x);
      tmem_ld_wait();
      const int n = n0 + c * 32;
      if (!row.valid || n >= p.ep.N) continue;
      float f[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) f[j] = (__uint_as_float(v[j]) + __uint_as_float(x[j])) * unscale;
      tc_store_chunk(p.ep, row, n, f, (int)blockIdx.z);
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2sm<512>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------- elementwise kernels
namespace {

enum RemapMode : int { REMAP_SAME = 0, REMAP_PLAIN_TO_S2D = 1, REMAP_S2D_TO_PLAIN = 2 };

// element offset i (first of 8 consecutive channels) of the source layout -> offset in the destination layout
//   PLAIN_TO_S2D: src [B, h, w, C]            -> dst [B, h/2, w/2, (py, px, C)]
//   S2D_TO_PLAIN: src [B, h, w, (py, px, C)]  -> dst [B, 2h, 2w, C]
__device__ __forceinline__ long long remap_offset(long long i, int mode, int h, int w, int C) {
  if (mode == REMAP_SAME) return i;
  if (mode == REMAP_PLAIN_TO_S2D) {
    const int c = (int)(i % C);
    long long r = i / C;
    const int x = (int)(r % w); r /= w;
    const int y = (int)(r % h);
    const long long b = r / h;
    return ((b * (h >> 1) + (y >> 1)) * (w >> 1) + (x >> 1)) * (4LL * C) + (((y & 1) << 1) | (x & 1)) * C + c;
  }
  const int c = (int)(i % C);
  long long r = i / C;
  const int cls = (int)(r & 3); r >>= 2;
  const int x = (int)(r % w); r /= w;
  const int y = (int)(r % h);
  const long long b = r / h;
  return ((b * 2 * h + 2 * y + (cls >> 1)) * (2LL * w) + 2 * x + (cls & 1)) * C + c;
}

__device__ __forceinline__ void load8(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void store8(float* p, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void apply_mask8(const __half* mask, float (&v)[8]) {
  const uint4 m = *reinterpret_cast<const uint4*>(mask);
  const __half2* mh = reinterpret_cast<const __half2*>(&m);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 f = __half22float2(mh[j]);
    if (!(f.x > 0.f)) v[2 * j] = 0.f;
    if (!(f.y > 0.f)) v[2 * j + 1] = 0.f;
  }
}

// slot = max(slot, max |x * (mask > 0)|) as fp32 bits (non-negative floats order like unsigned integers)
__global__ void amax_kernel(const float* __restrict__ x, const __half* __restrict__ mask, long long groups, unsigned* __restrict__ slot) {
  float m = 0.f;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (long long)gridDim.x * blockDim.x) {
    float v[8];
    load8(x + g * 8, v);
    if (mask) apply_mask8(mask + g * 8, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) m = fmaxf(m, fabsf(v[j]));
  }
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ float wm[8];
  if ((threadIdx.x & 31) == 0) wm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) m = fmaxf(m, wm[i]);
    if (m > 0.f) atomicMax(slot, __float_as_uint(m));
  }
}

// raw (fp32 dgrad result, source layout) -> ReLU mask of the forward activation (same layout as raw) -> (hi, lo) fp16 of
// value * tc_dyn_scale(amax) and/or fp32 in the remapped layout; optionally the masked fp32 back in place (fp32 consumers)
// and the per-column sums of the masked values (bias gradient): a thread always meets the same 8-column group because
// 256 % groups_per_row == 0, so it sums in registers and the block folds the threads of a group in fixed order.
__global__ void __launch_bounds__(256) finish_kernel(float* __restrict__ raw, const __half* __restrict__ mask, long long groups, int mode, int h, int w,
                                                     int C, const unsigned* __restrict__ amax, __half* __restrict__ hi, __half* __restrict__ lo,
                                                     float* __restrict__ out_f32, int write_masked, float* __restrict__ colsum, int groups_per_row) {
  __shared__ float red[256 * 8];
  const float scale = amax ? tc_dyn_scale(__ldg(amax)) : 1.f;
  float cs[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) cs[j] = 0.f;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (long long)gridDim.x * blockDim.x) {
    const long long i = g * 8;
    float v[8];
    load8(raw + i, v);
    if (mask) {
      apply_mask8(mask + i, v);
      if (write_masked) store8(raw + i, v);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) cs[j] += v[j];
    const long long j = remap_offset(i, mode, h, w, C);
    if (out_f32) store8(out_f32 + j, v);
    if (hi) {
      uint32_t hh[4], ll[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) split_f16x2(v[2 * t] * scale, v[2 * t + 1] * scale, hh[t], ll[t]);
      *reinterpret_cast<uint4*>(hi + j) = make_uint4(hh[0], hh[1], hh[2], hh[3]);
      *reinterpret_cast<uint4*>(lo + j) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
    }
  }
  if (colsum) {
#pragma unroll
    for (int j = 0; j < 8; ++j) red[threadIdx.x * 8 + j] = cs[j];
    __syncthreads();
    if ((int)threadIdx.x < groups_per_row) {
      for (int k = 1; k < 256 / groups_per_row; ++k)
#pragma unroll
        for (int j = 0; j < 8; ++j) cs[j] += red[(threadIdx.x + k * groups_per_row) * 8 + j];
      store8(colsum + ((long long)blockIdx.x * groups_per_row + threadIdx.x) * 8, cs);
    }
  }
}

// db[c] = sum over blocks and over the `reps` column blocks (space-to-depth parity classes) of partial[block][rep * C + c]:
// block = 32 columns x 32 row lanes (fixed assignment and fold order, so the result is deterministic)
__global__ void __launch_bounds__(1024) colsum_final_kernel(const float* __restrict__ partial, int blocks, int reps, int C, float* __restrict__ db) {
  __shared__ float red[32][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  float s0 = 0.f, s1 = 0.f;
  if (c < C) {
    const int rows = blocks * reps;
    float s2 = 0.f, s3 = 0.f;
    int r = threadIdx.y;
    for (; r + 96 < rows; r += 128) {
      s0 += partial[(long long)r * C + c];
      s1 += partial[(long long)(r + 32) * C + c];
      s2 += partial[(long long)(r + 64) * C + c];
      s3 += partial[(long long)(r + 96) * C + c];
    }
    for (; r < rows; r += 32) s0 += partial[(long long)r * C + c];
    s0 += s2; s1 += s3;
  }
  red[threadIdx.y][threadIdx.x] = s0 + s1;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float s = 0.f;
    for (int j = 0; j < 32; ++j) s += red[j][threadIdx.x];
    db[c] = s;
  }
}

// amax over a tensor whose size is not a multiple of 8 (the [B,H,W,3] loss gradient)
__global__ void amax_scalar_kernel(const float* __restrict__ x, long long n, unsigned* __restrict__ slot) {
  float m = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) m = fmaxf(m, fabsf(x[i]));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(slot, __float_as_uint(m));
}

// pre-sigmoid gradient g [B, 2h, 2w, c] (c <= 4) -> G of the output layer's GEMM: [B, h, w, gN] with channel (cls * c + co), rest zero
__global__ void pack_loss_grad_kernel(const float* __restrict__ g, int B, int h, int w, int c, int gN, const unsigned* __restrict__ amax,
                                      __half* __restrict__ hi, __half* __restrict__ lo) {
  const float scale = tc_dyn_scale(__ldg(amax));
  const long long total = (long long)B * h * w * 4 * c;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i % (4 * c));
    long long r = i / (4 * c);
    const int x = (int)(r % w); r /= w;
    const int y = (int)(r % h);
    const long long b = r / h;
    const int cls = n / c, co = n - cls * c;
    const float v = g[((b * 2 * h + 2 * y + (cls >> 1)) * (2LL * w) + 2 * x + (cls & 1)) * c + co] * scale;
    __half a, d;
    split_f16(v, a, d);
    const long long o = ((b * h + y) * w + x) * gN + n;
    hi[o] = a;
    lo[o] = d;
  }
}

// tap-separable output layer: G[pixel (b,y,x)][tap * n4 + m] = gs[(b, y - (ty-1), x - (tx-1))][m], gs = space-to-depth of the
// pre-sigmoid gradient g [B, 2h, 2w, c] (m = cls * c + co); columns >= 9 * n4 stay zero.  With this im2col both the dgrad
// (K = 128) and the wgrad (N = 128) of the layer read the big activation tensor exactly once.
__global__ void pack_loss_grad_sep_kernel(const float* __restrict__ g, int B, int h, int w, int c, const unsigned* __restrict__ amax,
                                          __half* __restrict__ hi, __half* __restrict__ lo) {
  const float scale = tc_dyn_scale(__ldg(amax));
  const int n4 = 4 * c;
  const long long total = (long long)B * h * w * 9;       // one thread per (pixel, tap): n4 consecutive columns
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int tap = (int)(i % 9);
    long long r = i / 9;
    const int x = (int)(r % w); r /= w;
    const int y = (int)(r % h);
    const long long b = r / h;
    const int ys = y - (tap / 3 - 1), xs = x - (tap % 3 - 1);
    const bool in = ys >= 0 && ys < h && xs >= 0 && xs < w;
    const long long o = ((b * h + y) * w + x) * 128 + tap * n4;
    // n4 = 4c values -> c groups of 4 halves (8 bytes) each for hi and lo
    for (int q = 0; q < c; ++q) {
      float v[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int m = q * 4 + e, cls = m / c, co = m - cls * c;
        v[e] = in ? g[((b * 2 * h + 2 * ys + (cls >> 1)) * (2LL * w) + 2 * xs + (cls & 1)) * c + co] * scale : 0.f;
      }
      uint32_t h0, l0, h1, l1;
      split_f16x2(v[0], v[1], h0, l0);
      split_f16x2(v[2], v[3], h1, l1);
      *reinterpret_cast<uint2*>(hi + o + q * 4) = make_uint2(h0, h1);
      *reinterpret_cast<uint2*>(lo + o + q * 4) = make_uint2(l0, l1);
    }
  }
}

// tap-separable output layer: dgrad operand [cin][128], column (tap * n4 + m) = Wm[tap][ci][m]
__global__ void pack_dec_dgrad_sep_kernel(const float* __restrict__ wm, int cin, int n4, float scale, __half* __restrict__ hi,
                                          __half* __restrict__ lo) {
  const int total = cin * 128;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int k = i & 127, ci = i >> 7;
    const int tap = k / n4, m = k - tap * n4;
    const float v = tap < 9 ? wm[((long long)tap * cin + ci) * n4 + m] * scale : 0.f;
    __half a, d;
    split_f16(v, a, d);
    hi[i] = a;
    lo[i] = d;
  }
}

// wgrad result of the tap-separable layer [cin][128] (column = tap * n4 + m) -> merged-gradient layout [9][cin][n4]
__global__ void rearrange_sep_wgrad_kernel(const float* __restrict__ in, int cin, int n4, float* __restrict__ out) {
  const int total = 9 * cin * n4;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int m = i % n4, ci = (i / n4) % cin, tap = i / (n4 * cin);
    out[i] = in[ci * 128 + tap * n4 + m];
  }
}

// 8 consecutive fp32 -> (hi, lo) fp16, one 16-byte store each
__device__ __forceinline__ void split_store8(const float (&v)[8], float scale, __half* hi, __half* lo) {
  uint32_t hh[4], ll[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) split_f16x2(v[2 * t] * scale, v[2 * t + 1] * scale, hh[t], ll[t]);
  *reinterpret_cast<uint4*>(hi) = make_uint4(hh[0], hh[1], hh[2], hh[3]);
  *reinterpret_cast<uint4*>(lo) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
}

// decoder unit: merged weights Wm [9][cin][n4] -> dgrad operand [cin][9 * gN] with the taps flipped, columns >= n4 zero.
// One thread per 8 consecutive columns (n4 % 8 == 0) or per column (the padded output layer).
__global__ void pack_dec_dgrad_kernel(const float* __restrict__ wm, int cin, int n4, int gN, float scale, __half* __restrict__ hi,
                                      __half* __restrict__ lo) {
  if (n4 % 8 == 0 && gN == n4) {
    const int g8 = gN / 8;
    const long long total = (long long)cin * 9 * g8;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const int n = (int)(i % g8) * 8;
      long long r = i / g8;
      const int t = (int)(r % 9);
      const int ci = (int)(r / 9);
      float v[8];
      load8(wm + ((long long)(8 - t) * cin + ci) * n4 + n, v);
      split_store8(v, scale, hi + i * 8, lo + i * 8);
    }
    return;
  }
  const long long total = (long long)cin * 9 * gN;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i % gN);
    long long r = i / gN;
    const int t = (int)(r % 9);
    const int ci = (int)(r / 9);
    const float v = n < n4 ? wm[((long long)(8 - t) * cin + ci) * n4 + n] * scale : 0.f;
    __half a, d;
    split_f16(v, a, d);
    hi[i] = a;
    lo[i] = d;
  }
}

// encoder unit: W HWIO [5][5][cin][cout] -> dgrad operand [(py,px,ci)][9 * cout]; tap (ty,tx) of the 3x3 window over dY
// carries kernel element (3 - 2ty + py, 3 - 2tx + px) when that lies inside the 5x5 kernel.  8 output channels per thread.
__global__ void pack_enc_dgrad_kernel(const float* __restrict__ w, int cin, int cout, float scale, __half* __restrict__ hi,
                                      __half* __restrict__ lo) {
  const int c8 = cout / 8;
  const long long total = 4LL * cin * 9 * c8;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(i % c8) * 8;
    long long r = i / c8;
    const int t = (int)(r % 9); r /= 9;
    const int ci = (int)(r % cin);
    const int cls = (int)(r / cin);
    const int kh = 3 - 2 * (t / 3) + (cls >> 1), kw = 3 - 2 * (t % 3) + (cls & 1);
    float v[8];
    if (kh >= 0 && kh < 5 && kw >= 0 && kw < 5) {
      load8(w + (((long long)kh * 5 + kw) * cin + ci) * cout + co, v);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
    }
    split_store8(v, scale, hi + i * 8, lo + i * 8);
  }
}

__global__ void unpack_plain_kernel(const __half* __restrict__ hi, const __half* __restrict__ lo, long long n, float inv_scale,
                                    float* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = (__half2float(hi[i]) + __half2float(lo[i])) * inv_scale;
}

__global__ void compact_cols_kernel(const float* __restrict__ in, long long rows, int ld, int n, float* __restrict__ out) {
  const long long total = rows * n;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
    out[i] = in[(i / n) * ld + (i % n)];
}

inline unsigned ew_grid(long long n, int threads = 256) {
  long long b = (n + threads - 1) / threads;
  return (unsigned)std::max<long long>(1, std::min<long long>(b, 148 * 16));
}

// First encoder layer (Cin = 3, K = 75): its weight gradient is a 1x1 wgrad GEMM over the im2col matrix of the input image.
// x fp32 [B, H, W, 3] -> A (hi, lo) fp16 [B*OH*OW][128]: column k = (kh*5 + kw)*3 + c < 75 holds scale * x[b, 2oh - pad_t + kh, 2ow - pad_l + kw, c]
// (zero outside the image), columns 75..127 are zero.  One thread per (pixel, 8-column group): 16-byte stores.
__global__ void conv1_im2col_kernel(const float* __restrict__ x, long long pixels, int H, int W, int OH, int OW, int pad_t, int pad_l, float scale,
                                    __half* __restrict__ hi, __half* __restrict__ lo) {
  const long long total = pixels * 16;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long pix = idx >> 4;
    const int g = (int)(idx & 15);
    const int ow = (int)(pix % OW), oh = (int)((pix / OW) % OH);
    const long long b = pix / ((long long)OW * OH);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = g * 8 + j;
      v[j] = 0.f;
      if (k < 75) {
        const int kh = k / 15, r = k - kh * 15, kw = r / 3, c = r - kw * 3;
        const int ih = 2 * oh - pad_t + kh, iw = 2 * ow - pad_l + kw;
        if (ih >= 0 && ih < H && iw >= 0 && iw < W) v[j] = __ldg(x + ((b * H + ih) * W + iw) * 3 + c) * scale;
      }
    }
    uint32_t hh[4], ll[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) split_f16x2(v[2 * t], v[2 * t + 1], hh[t], ll[t]);
    *reinterpret_cast<uint4*>(hi + pix * 128 + g * 8) = make_uint4(hh[0], hh[1], hh[2], hh[3]);
    *reinterpret_cast<uint4*>(lo + pix * 128 + g * 8) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
  }
}

template <int N_TILE, int STAGES>
int launch_wgrad(const CUtensorMap& xh, const CUtensorMap& xl, const CUtensorMap& gh, const CUtensorMap& gl, const TcWgradParams& p, dim3 grid,
                 cudaStream_t s) {
  using S = WgSmem<N_TILE, STAGES>;
  auto kern = tc_wgrad_kernel<N_TILE, STAGES>;
  AAE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
  kern<<<grid, TC_THREADS, S::TOTAL, s>>>(xh, xl, gh, gl, p);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

template <int STAGES>
int launch_wgrad2(const CUtensorMap& xh, const CUtensorMap& xl, const CUtensorMap& gh, const CUtensorMap& gl, const TcWgradParams& p, dim3 grid,
                  cudaStream_t s) {
  using S = WgSmem2<STAGES>;
  auto kern = tc_wgrad2_kernel<STAGES>;
  AAE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
  grid.x = (grid.x + 1) & ~1u;
  kern<<<grid, TC_THREADS, S::TOTAL, s>>>(xh, xl, gh, gl, p);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------- plan
struct TcUnit {
  bool enc;                 // encoder 5x5/s2 layer (X in space-to-depth form) or decoder sub-pixel layer
  int cin, cout;            // the layer's real channel counts
  int gh, gw, gN;           // G = pre-activation gradient of the layer's GEMM output: plain [B, gh, gw, gN]
  int n_real;               // real columns of G (4*cout for the decoder output layer whose gN is padded)
  int taps_w;               // taps of the wgrad (25 / 9; 1 for the tap-separable output layer)
  int dg_taps;              // taps of the dgrad conv over G (9; 1 for the tap-separable output layer)
  bool sep;                 // decoder output layer in tap-separable form: G is the im2col [pixel][(tap, cls, co)] of the loss gradient
  TcLayer dg;               // dgrad GEMM: A = G (dg.in_hi / in_lo are the G buffers), B = re-packed weights
  int nd;                   // dgrad output columns (decoder: cin, encoder: 4*cin)
  const __half *x_hi, *x_lo;  // the layer's forward input (owned by the encoder / decoder plan)
  const __half* mask_hi;    // forward activation whose ReLU masks this unit's dgrad result (same layout as the result)
  CUtensorMap tm_x_hi, tm_x_lo, tm_g_hi, tm_g_lo;   // wgrad operand maps (64-channel x 32-pixel boxes)
  TcWgradParams wp;
  int wg_n_tile;
};

struct TcTrainPlan {
  int device, max_batch;
  TcEncoder* enc;
  TcDecoder* dec;
  std::vector<TcUnit> units;      // backward order: decoder L..1, encoder L-1..1
  int n_dec;                      // number of decoder units
  unsigned* amax = nullptr;       // one slot per unit (largest |G|, fp32 bits)
  float* raw = nullptr;           // fp32 dgrad result of the current unit
  size_t raw_floats = 0;
  float* f32_out = nullptr;       // fp32 gradient handed to the SIMT conv1 wgrad (plain NHWC)
  float* partials = nullptr;      // split-K partials of the wgrad GEMMs
  size_t partial_floats = 0;
  float* wm = nullptr;            // fp32 merged sub-pixel weights / padded merged gradient scratch
  size_t wm_floats = 0;
  // conv1 (Cin = 3): wgrad-only unit appended after the encoder units (index c1, -1 = SIMT wgrad): X = im2col of the input image
  int c1 = -1;
  __half *c1_x_hi = nullptr, *c1_x_lo = nullptr;
};

static int make_wgrad_maps(TcUnit& U, int x_c_total, int x_bpad, int g_bpad) {
  const int bw = std::min(U.gw, 32), bh = 32 / bw;
  {
    const uint64_t dims[4] = {(uint64_t)x_c_total, (uint64_t)U.gw, (uint64_t)U.gh, (uint64_t)x_bpad};
    const uint64_t str[3] = {(uint64_t)x_c_total * 2, (uint64_t)U.gw * x_c_total * 2, (uint64_t)U.gh * U.gw * x_c_total * 2};
    const uint32_t box[4] = {64, (uint32_t)bw, (uint32_t)bh, 1};
    AAE_TRY(make_tmap_f16(&U.tm_x_hi, U.x_hi, 4, dims, str, box, 128));
    AAE_TRY(make_tmap_f16(&U.tm_x_lo, U.x_lo, 4, dims, str, box, 128));
  }
  {
    const uint64_t dims[4] = {(uint64_t)U.gN, (uint64_t)U.gw, (uint64_t)U.gh, (uint64_t)g_bpad};
    const uint64_t str[3] = {(uint64_t)U.gN * 2, (uint64_t)U.gw * U.gN * 2, (uint64_t)U.gh * U.gw * U.gN * 2};
    const uint32_t box[4] = {64, (uint32_t)bw, (uint32_t)bh, 1};
    AAE_TRY(make_tmap_f16(&U.tm_g_hi, U.dg.in_hi, 4, dims, str, box, 128));
    AAE_TRY(make_tmap_f16(&U.tm_g_lo, U.dg.in_lo, 4, dims, str, box, 128));
  }
  TcWgradParams& w = U.wp;
  memset(&w, 0, sizeof(w));
  w.cin_blocks = U.cin / 128;
  w.OH = U.gh; w.OW = U.gw; w.BWk = bw; w.BHk = bh;
  w.chunks_per_image = U.gh * U.gw / 32;
  w.ep.out_mode = OUT_F32;
  w.ep.M = U.taps_w * U.cin;
  w.ep.N = U.gN;
  w.ep.OH = w.ep.OW = 1;
  w.ep.unscale = 1.f / ACT_SCALE;
  w.m_tiles = U.taps_w * w.cin_blocks;
  U.wg_n_tile = U.gN >= 256 ? 256 : 64;
  return AAE_OK;
}

int tc_train_create(TcEncoder* enc, TcDecoder* dec, int max_batch, TcTrainPlan** out) {
  *out = nullptr;
  AAE_REQUIRE(enc && dec && enc->conv1, "tensor-core trainer: needs the tensor-core encoder (incl. conv1) and decoder plans");
  TcTrainPlan* h = new TcTrainPlan();
  h->device = enc->device; h->max_batch = max_batch; h->enc = enc; h->dec = dec;
  const int B = max_batch;
  int st = AAE_OK;
  const int Ld = (int)dec->layers.size() - 1;       // decoder conv layers 1..Ld
  const int Le = (int)enc->layers.size() - 1;       // encoder TC conv layers (conv2..): enc->layers[0..Le-1]
  size_t raw_max = 0, part_max = 0, wm_max = 0;
  auto add_unit = [&](TcUnit& U, const TcLayer& F, int x_c_total) -> int {
    TcLayer& T = U.dg;
    memset(&T.gp, 0, sizeof(T.gp));
    T.in_h = U.gh; T.in_w = U.gw; T.in_c = U.gN;
    T.out_h = U.gh; T.out_w = U.gw; T.out_c = U.nd;
    T.taps = U.dg_taps;
    T.BW = U.gw; T.BH = std::min(U.gh, 128 / T.BW); T.BB = 128 / (T.BW * T.BH);
    T.n_tile = U.nd >= 256 ? 256 : 128;
    T.kch = T.n_tile == 256 ? 32 : 64;
    if (U.gw > 128 || (U.gw & (U.gw - 1)) || (U.gh & (U.gh - 1)) || U.gN % T.kch != 0 || U.nd % T.n_tile != 0 || U.cin % 128 != 0 ||
        U.gN % 64 != 0 || (U.gh * U.gw) % 32 != 0) {
      set_error("tensor-core trainer: layer geometry unsupported (G %dx%dx%d, dgrad N %d, Cin %d)", U.gh, U.gw, U.gN, U.nd, U.cin);
      return AAE_ERR_UNSUPPORTED;
    }
    TcGemmParams& g = T.gp;
    g.N = U.nd; g.OH = U.gh; g.OW = U.gw; g.BW = T.BW; g.BH = T.BH;
    g.taps = T.taps; g.chunks_per_tap = U.gN / T.kch; g.iters_per_split = g.taps * g.chunks_per_tap;
    for (int t = 0; t < T.taps; ++t) {
      g.tap_di[t] = (int8_t)(T.taps == 1 ? 0 : t / 3 - 1);
      g.tap_dj[t] = (int8_t)(T.taps == 1 ? 0 : t % 3 - 1);
      g.tap_ch[t] = 0;
    }
    g.unscale = 1.f / W_SCALE;
    g.out_mode = OUT_F32;
    AAE_TRY(tc_layer_setup_plain(T, B, /*pair_ok=*/true, /*alloc_input=*/true));
    U.x_hi = F.in_hi; U.x_lo = F.in_lo;
    const int x_bpad = (int)ceil_div(B, F.BB) * F.BB, g_bpad = (int)ceil_div(B, T.BB) * T.BB;
    AAE_TRY(make_wgrad_maps(U, x_c_total, x_bpad, g_bpad));
    for (int t = 0; t < U.taps_w; ++t) { U.wp.tap_di[t] = F.gp.tap_di[t]; U.wp.tap_dj[t] = F.gp.tap_dj[t]; U.wp.tap_ch[t] = F.gp.tap_ch[t]; }
    raw_max = std::max(raw_max, (size_t)B * U.gh * U.gw * U.nd);
    wm_max = std::max(wm_max, (size_t)U.taps_w * U.cin * U.gN);
    return AAE_OK;
  };
  for (int l = Ld; l >= 1 && st == AAE_OK; --l) {          // decoder units
    const TcLayer& F = dec->layers[l];
    TcUnit U;
    U.enc = false; U.cin = F.in_c; U.cout = F.out_c;
    U.gh = F.in_h; U.gw = F.in_w;
    U.sep = l == Ld && dec->sep_out;
    U.n_real = U.sep ? 36 * F.out_c : 4 * F.out_c;
    U.gN = U.sep ? 128 : (l == Ld ? 64 : 4 * F.out_c);
    U.taps_w = U.sep ? 1 : 9; U.dg_taps = U.sep ? 1 : 9; U.nd = F.in_c;
    U.mask_hi = F.in_hi;                                   // dgrad result = gradient wrt this layer's input activation
    if (l == Ld && U.n_real > U.gN) { set_error("tensor-core trainer: output channels > 16 unsupported"); st = AAE_ERR_UNSUPPORTED; break; }
    h->units.push_back(U);
    st = add_unit(h->units.back(), F, F.in_c);
  }
  h->n_dec = (int)h->units.size();
  for (int i = Le - 1; i >= 0 && st == AAE_OK; --i) {      // encoder units (enc->layers[i] = conv i+2)
    const TcLayer& F = enc->layers[i];
    TcUnit U;
    U.enc = true; U.cin = F.in_c; U.cout = F.out_c;
    U.gh = F.out_h; U.gw = F.out_w; U.gN = F.out_c; U.n_real = F.out_c;
    U.taps_w = 25; U.dg_taps = 9; U.sep = false; U.nd = 4 * F.in_c;
    U.mask_hi = F.in_hi;                                   // space-to-depth activation, same layout as the dgrad result
    h->units.push_back(U);
    st = add_unit(h->units.back(), F, 4 * F.in_c);
  }
  if (st == AAE_OK && Le >= 1 && enc->cfg.in_c == 3 && enc->cfg.kernel_size == 5 && enc->layers[0].in_c == 128) {
    // dW1[75, 128] = sum over pixels of im2col(x)[pixel, :75]^T G1[pixel, :]: the same 1x1 wgrad GEMM as the tap-separable output layer
    const TcLayer& F2 = enc->layers[0];                    // conv2: in_h x in_w x in_c are the dims of conv1's output (stored space-to-depth)
    const size_t n = (size_t)B * F2.in_h * F2.in_w * 128;
    st = tc_dev_alloc((void**)&h->c1_x_hi, n * sizeof(__half));
    if (st == AAE_OK) st = tc_dev_alloc((void**)&h->c1_x_lo, n * sizeof(__half));
    if (st == AAE_OK) {
      TcLayer Fx;                                          // stands for "the layer whose input is X": only in_hi/in_lo, BB and the tap tables are read
      memset(&Fx.gp, 0, sizeof(Fx.gp));
      Fx.in_hi = h->c1_x_hi; Fx.in_lo = h->c1_x_lo; Fx.BB = 1;
      TcUnit U;
      U.enc = true; U.cin = 128; U.cout = F2.in_c;
      U.gh = F2.in_h; U.gw = F2.in_w; U.gN = F2.in_c; U.n_real = F2.in_c;
      U.taps_w = 1; U.dg_taps = 1; U.sep = false; U.nd = 128;   // (no dgrad is ever run for this unit: the input image needs no gradient)
      U.mask_hi = nullptr;
      h->units.push_back(U);
      st = add_unit(h->units.back(), Fx, 128);
      if (st == AAE_OK) h->c1 = (int)h->units.size() - 1;
    }
  }
  part_max = (size_t)40 << 20;   // 160 MB of fp32 partials; wgrad split counts are clamped to fit
  if (st == AAE_OK) st = tc_dev_alloc((void**)&h->amax, 64 * sizeof(unsigned));
  if (st == AAE_OK) st = tc_dev_alloc((void**)&h->raw, raw_max * sizeof(float));
  if (st == AAE_OK) st = tc_dev_alloc((void**)&h->f32_out, raw_max * sizeof(float));
  if (st == AAE_OK) st = tc_dev_alloc((void**)&h->partials, part_max * sizeof(float));
  if (st == AAE_OK) st = tc_dev_alloc((void**)&h->wm, wm_max * sizeof(float));
  h->raw_floats = raw_max; h->partial_floats = part_max; h->wm_floats = wm_max;
  // the persistent pair kernel ships unsplit dgrad results to `raw` with tensor stores
  for (size_t u = 0; u < h->units.size() && st == AAE_OK; ++u) {
    TcLayer& T = h->units[u].dg;
    if (!T.pair) continue;
    T.gp.out_f32 = h->raw;
    st = tc_layer_setup_out_maps(T, (long long)(raw_max / (size_t)T.gp.N));
  }
  if (st != AAE_OK) { tc_train_destroy(h); return st; }
  *out = h;
  return AAE_OK;
}

void tc_train_destroy(TcTrainPlan* h) {
  if (!h) return;
  for (auto& U : h->units) { cudaFree(U.dg.in_hi); cudaFree(U.dg.in_lo); cudaFree(U.dg.w_hi); cudaFree(U.dg.w_lo); }
  cudaFree(h->amax); cudaFree(h->raw); cudaFree(h->f32_out); cudaFree(h->partials); cudaFree(h->wm);
  cudaFree(h->c1_x_hi); cudaFree(h->c1_x_lo);
  delete h;
}

int tc_train_num_units(const TcTrainPlan* h) { return (int)h->units.size() - (h->c1 >= 0 ? 1 : 0); }   // conv units with a dgrad
int tc_train_conv1_unit(const TcTrainPlan* h) { return h->c1; }
int tc_train_num_decoder_units(const TcTrainPlan* h) { return h->n_dec; }
float* tc_train_raw(TcTrainPlan* h) { return h->raw; }
float* tc_train_f32_out(TcTrainPlan* h) { return h->f32_out; }

int tc_train_begin_step(TcTrainPlan* h, cudaStream_t s) {
  AAE_CUDA_OK(cudaMemsetAsync(h->amax, 0, 64 * sizeof(unsigned), s));
  return AAE_OK;
}

// dgrad operand of unit u from the layer's fp32 kernel (HWIO [5,5,cin,cout], device pointer)
int tc_train_pack_weights(TcTrainPlan* h, int u, const float* w_dev, cudaStream_t s) {
  AAE_REQUIRE(u >= 0 && u < (int)h->units.size(), "tc trainer: unit %d out of range", u);
  TcUnit& U = h->units[u];
  if (U.enc) {
    pack_enc_dgrad_kernel<<<ew_grid(4LL * U.cin * 9 * U.cout / 8), 256, 0, s>>>(w_dev, U.cin, U.cout, W_SCALE, U.dg.w_hi, U.dg.w_lo);
    AAE_LAUNCH_OK();
    return AAE_OK;
  }
  AAE_TRY(launch_merge_subpixel_weights(w_dev, U.cin, U.cout, h->wm, s));
  return tc_train_pack_weights_merged(h, u, h->wm, s);
}

// decoder unit: dgrad operand from the already merged sub-pixel weights Wm [9][cin][4*cout] (device pointer)
int tc_train_pack_weights_merged(TcTrainPlan* h, int u, const float* wm_dev, cudaStream_t s) {
  AAE_REQUIRE(u >= 0 && u < h->n_dec, "tc trainer: unit %d is not a decoder unit", u);
  TcUnit& U = h->units[u];
  if (U.sep) pack_dec_dgrad_sep_kernel<<<ew_grid((long long)U.cin * 128), 256, 0, s>>>(wm_dev, U.cin, 4 * U.cout, W_SCALE, U.dg.w_hi, U.dg.w_lo);
  else pack_dec_dgrad_kernel<<<ew_grid((long long)U.cin * 9 * U.gN), 256, 0, s>>>(wm_dev, U.cin, U.n_real, U.gN, W_SCALE, U.dg.w_hi, U.dg.w_lo);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

// pre-sigmoid gradient of the reconstruction [B, H, W, C] -> G of unit 0 (the decoder output layer)
int tc_train_set_loss_grad(TcTrainPlan* h, const float* g_dev, int B, cudaStream_t s) {
  TcUnit& U = h->units[0];
  const int c = U.cout;
  const long long n = (long long)B * U.gh * U.gw * 4 * c;
  amax_scalar_kernel<<<ew_grid(n), 256, 0, s>>>(g_dev, n, h->amax + 0);
  AAE_LAUNCH_OK();
  if (U.sep) pack_loss_grad_sep_kernel<<<ew_grid((long long)B * U.gh * U.gw * 9), 256, 0, s>>>(g_dev, B, U.gh, U.gw, c, h->amax + 0, U.dg.in_hi, U.dg.in_lo);
  else pack_loss_grad_kernel<<<ew_grid(n), 256, 0, s>>>(g_dev, B, U.gh, U.gw, c, U.gN, h->amax + 0, U.dg.in_hi, U.dg.in_lo);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

// fp32 plain gradient [B, gh, gw, gN] (already masked) -> G of unit u
int tc_train_set_unit_grad(TcTrainPlan* h, int u, const float* g_dev, int B, cudaStream_t s) {
  TcUnit& U = h->units[u];
  const long long groups = (long long)B * U.gh * U.gw * U.gN / 8;
  amax_kernel<<<ew_grid(groups), 256, 0, s>>>(g_dev, nullptr, groups, h->amax + u);
  AAE_LAUNCH_OK();
  finish_kernel<<<ew_grid(groups), 256, 0, s>>>(const_cast<float*>(g_dev), nullptr, groups, REMAP_SAME, U.gh, U.gw, U.gN, h->amax + u, U.dg.in_hi,
                                                U.dg.in_lo, nullptr, 0, nullptr, 1);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

// dW of unit u: encoder units -> HWIO [25*cin][cout]; decoder units -> merged [9*cin][4*cout] (see launch_unmerge_subpixel_grads)
int tc_train_unit_wgrad(TcTrainPlan* h, int u, int B, float* dw_out, cudaStream_t s) {
  TcUnit& U = h->units[u];
  TcWgradParams w = U.wp;
  w.total_chunks = B * w.chunks_per_image;
  const int m_tiles = U.taps_w * w.cin_blocks, n_tiles = U.gN / U.wg_n_tile;
  const long long mn = (long long)w.ep.M * w.ep.N;
  int splits = (int)std::max<long long>(1, (444 + (long long)m_tiles * n_tiles / 2) / ((long long)m_tiles * n_tiles));
  splits = std::min(splits, std::max(1, w.total_chunks / 16));
  splits = (int)std::min<long long>(splits, (long long)(h->partial_floats / (size_t)mn));
  AAE_REQUIRE(splits >= 1, "tc trainer: wgrad partial scratch too small");
  w.chunks_per_split = (int)ceil_div(w.total_chunks, splits);
  splits = (int)ceil_div(w.total_chunks, w.chunks_per_split);
  w.ep.amax_bits = h->amax + u;
  w.ep.out_f32 = h->partials;
  dim3 grid((unsigned)m_tiles, (unsigned)n_tiles, (unsigned)splits);
  if (U.wg_n_tile == 256) AAE_TRY((launch_wgrad2<6>(U.tm_x_hi, U.tm_x_lo, U.tm_g_hi, U.tm_g_lo, w, grid, s)));
  else AAE_TRY((launch_wgrad<64, 6>(U.tm_x_hi, U.tm_x_lo, U.tm_g_hi, U.tm_g_lo, w, grid, s)));
  if (U.gN == U.n_real) return launch_splitk_reduce(h->partials, splits, mn, w.ep.N, nullptr, ACT_NONE, dw_out, s);
  AAE_REQUIRE((size_t)mn <= h->wm_floats, "tc trainer: merged-gradient scratch too small");
  AAE_TRY(launch_splitk_reduce(h->partials, splits, mn, w.ep.N, nullptr, ACT_NONE, h->wm, s));
  if (U.sep) {
    rearrange_sep_wgrad_kernel<<<ew_grid(9LL * U.cin * 4 * U.cout), 256, 0, s>>>(h->wm, U.cin, 4 * U.cout, dw_out);
    AAE_LAUNCH_OK();
    return AAE_OK;
  }
  compact_cols_kernel<<<ew_grid((long long)w.ep.M * U.n_real), 256, 0, s>>>(h->wm, w.ep.M, U.gN, U.n_real, dw_out);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

// dW of conv1 [75][cout] from the fp32 input image x [B, H, W, 3] and the unit's G (written by tc_train_finish(..., next = conv1 unit))
int tc_train_conv1_wgrad(TcTrainPlan* h, const float* x_dev, int B, float* dw_out, cudaStream_t s) {
  AAE_REQUIRE(h->c1 >= 0, "tc trainer: no tensor-core conv1 wgrad unit");
  TcUnit& U = h->units[h->c1];
  const aae_net_cfg& cfg = h->enc->cfg;
  const long long pixels = (long long)B * U.gh * U.gw;
  const int pad_t = std::max((U.gh - 1) * 2 + 5 - cfg.in_h, 0) / 2, pad_l = std::max((U.gw - 1) * 2 + 5 - cfg.in_w, 0) / 2;
  conv1_im2col_kernel<<<ew_grid(pixels * 16), 256, 0, s>>>(x_dev, pixels, cfg.in_h, cfg.in_w, U.gh, U.gw, pad_t, pad_l, ACT_SCALE, h->c1_x_hi, h->c1_x_lo);
  AAE_LAUNCH_OK();
  AAE_REQUIRE((size_t)128 * U.gN <= h->wm_floats, "tc trainer: scratch too small for the conv1 wgrad");
  AAE_TRY(tc_train_unit_wgrad(h, h->c1, B, h->wm, s));         // [128 im2col columns][cout]; rows 75.. are zero
  AAE_CUDA_OK(cudaMemcpyAsync(dw_out, h->wm, (size_t)75 * U.gN * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return AAE_OK;
}

// raw = dgrad of unit u: [B*gh*gw][nd] fp32 (decoder: gradient wrt the layer's plain input; encoder: wrt its space-to-depth input)
int tc_train_unit_dgrad(TcTrainPlan* h, int u, int B, cudaStream_t s) {
  TcUnit& U = h->units[u];
  TcLayer& T = U.dg;
  T.gp.M = B * U.gh * U.gw;
  T.gp.amax_bits = h->amax + u;
  const int m_tiles = (int)ceil_div(T.gp.M, 128), n_tiles = U.nd / T.n_tile;
  const int total_iters = T.gp.taps * T.gp.chunks_per_tap;
  // few output tiles and a long K (the 8x8 layers): split K so that the grid covers the SMs, fold the partials afterwards
  int splits = std::max(1, 148 / std::max(1, ((m_tiles + 1) & ~1) * n_tiles));
  splits = std::min(splits, std::max(1, total_iters / 64));
  const long long mn = (long long)T.gp.M * U.nd;
  if ((size_t)splits * (size_t)mn > h->partial_floats) splits = 1;
  T.gp.iters_per_split = (int)ceil_div(total_iters, splits);
  splits = (int)ceil_div(total_iters, T.gp.iters_per_split);
  T.gp.out_f32 = splits > 1 ? h->partials : h->raw;
  dim3 grid((unsigned)m_tiles, (unsigned)n_tiles, (unsigned)splits);
  AAE_TRY(tc_launch_layer(T, grid, s));
  if (splits > 1) AAE_TRY(launch_splitk_reduce(h->partials, splits, mn, U.nd, nullptr, ACT_NONE, h->raw, s));
  return AAE_OK;
}

// raw of unit u -> ReLU mask -> G of unit `next` (when next >= 0) and/or fp32 in the remapped layout (want_f32), the masked
// fp32 back in place (keep_masked) and its per-channel sums db_out (bias gradient of the layer that produced the masked
// activation).  Layout change: decoder plain -> space-to-depth (the producing layer's GEMM columns), encoder the reverse.
int tc_train_finish(TcTrainPlan* h, int u, int next, int B, bool want_f32, bool keep_masked, float* db_out, cudaStream_t s) {
  TcUnit& U = h->units[u];
  const long long groups = (long long)B * U.gh * U.gw * U.nd / 8;
  __half *hi = nullptr, *lo = nullptr;
  unsigned* slot = nullptr;
  if (next >= 0) {
    TcUnit& Nx = h->units[next];
    AAE_REQUIRE((long long)Nx.gh * Nx.gw * Nx.gN == (long long)U.gh * U.gw * U.nd, "tc trainer: unit %d does not feed unit %d", u, next);
    hi = Nx.dg.in_hi; lo = Nx.dg.in_lo; slot = h->amax + next;
    amax_kernel<<<ew_grid(groups), 256, 0, s>>>(h->raw, U.mask_hi, groups, slot);
    AAE_LAUNCH_OK();
  }
  const int mode = U.enc ? REMAP_S2D_TO_PLAIN : (next >= 0 ? REMAP_PLAIN_TO_S2D : REMAP_SAME);
  // source dims: decoder raw is plain [B, gh, gw, nd]; encoder raw is [B, gh, gw, (cls, cin)]
  const int C = U.enc ? U.cin : U.nd;
  const int gpr = U.nd / 8;                          // 8-column groups per raw row
  // with the fused column sums every block leaves one partial row: 4 blocks per SM keep the fold short
  const unsigned grid = db_out ? std::min(ew_grid(groups), 148u * 4u) : ew_grid(groups);
  float* colsum = nullptr;
  if (db_out) {
    AAE_REQUIRE(gpr <= 256 && 256 % gpr == 0, "tc trainer: %d columns unsupported by the fused bias gradient", U.nd);
    AAE_REQUIRE((size_t)grid * U.nd <= h->partial_floats, "tc trainer: column-sum scratch too small");
    colsum = h->partials;
  }
  finish_kernel<<<grid, 256, 0, s>>>(h->raw, U.mask_hi, groups, mode, U.gh, U.gw, C, slot, hi, lo, want_f32 ? h->f32_out : nullptr,
                                     keep_masked ? 1 : 0, colsum, std::max(gpr, 1));
  AAE_LAUNCH_OK();
  if (db_out) {
    colsum_final_kernel<<<(unsigned)ceil_div(C, 32), dim3(32, 32), 0, s>>>(colsum, (int)grid, U.nd / C, C, db_out);
    AAE_LAUNCH_OK();
  }
  return AAE_OK;
}

// fp32 copy of the encoder's last conv activation (the dense layer's input, plain [B, flat]) for the fp32 dense backward
int tc_train_unpack_flat(TcTrainPlan* h, int B, float* out, cudaStream_t s) {
  const TcLayer& D = h->enc->layers.back();
  const long long n = (long long)B * D.in_c;
  unpack_plain_kernel<<<ew_grid(n), 256, 0, s>>>(D.in_hi, D.in_lo, n, 1.f / ACT_SCALE, out);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

void tc_train_unit_info(const TcTrainPlan* h, int u, int* is_enc, int* cin, int* cout, int* gh, int* gw, int* nd) {
  const TcUnit& U = h->units[u];
  *is_enc = U.enc ? 1 : 0; *cin = U.cin; *cout = U.cout; *gh = U.gh; *gw = U.gw; *nd = U.nd;
}

}  // namespace aae
