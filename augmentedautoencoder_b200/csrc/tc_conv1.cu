// First encoder layer on tcgen05 (AAE_PREC_TC_SPLIT): conv 5x5 / stride 2 / TF-SAME(1,2), Cin = 3 -> Cout = 128, + bias +
// ReLU  (auto_pose/ae/encoder.py:43-50, first loop iteration), fused with the x/255. of auto_pose/ae/codebook.py:58-59.
//
// K = 25*3 = 75 is far too small and too ragged for TMA (patches overlap, 3-byte pixels), so the A operand is built in
// shared memory by 128 "builder" threads -- one output pixel (one im2col row) each -- straight from the uint8 crop:
// a 256-entry lookup table maps a byte to the fp16 (hi, lo) pair of 16 * (u8 / 255) (exact IEEE divide on the host of
// the kernel, so the fused path is bit-identical to the reference's float feed), and the row is written in the
// 128-byte-swizzle K-major canonical layout.  K is padded to 80 = 5 MMA K-steps.  The packed weights ([128][128] K-major,
// zero beyond k = 75) are TMA-loaded once per CTA and stay resident.  Persistent CTAs loop over 128-pixel tiles with a
// single-stage A buffer and a double-buffered TMEM accumulator: builders (warps 0-3), epilogue (warps 4-11, two per TMEM
// lane quadrant) and the MMA issuer (warp 12) all overlap.  The epilogue writes conv2's input directly: (hi, lo) fp16, space-to-depth layout.
#include <stdlib.h>

#include <algorithm>

#include "tc.cuh"
#include "tc_common.cuh"

namespace aae {

using namespace tc;

namespace {

constexpr int C1_ATOM = 128 * 128;                 // 128 rows x 128 B
constexpr int C1_STAGE = 4 * C1_ATOM;              // hi k[0,64), hi k[64,128), lo k[0,64), lo k[64,128)
constexpr int C1_STAGES = 1;                       // the build (~0.4k cycles) is short next to the MMAs + epilogue; smem goes to the output staging
constexpr int C1_OUT_LD = 1040;                    // staged output: 32 blocks of 1 KB (one space-to-depth position each), padded against bank conflicts
// consecutive 1 KB output blocks shipped by one bulk store: fewer, larger copies vs bank conflicts.  Measured 0.25 / 0.22 / 0.28 /
// 0.28 ms for groups of 1 / 2 / 4 / 8.
constexpr int C1_OUT_GROUP = 2;
constexpr int C1_KPAD = 80;
constexpr int C1_EPI_WARPS = 8;                    // two per TMEM lane quadrant (each takes every other 32-channel chunk)
constexpr int C1_MMA_WARP = 4 + C1_EPI_WARPS;
constexpr int C1_THREADS = 32 * (C1_MMA_WARP + 1);
constexpr int C1_PIX_ROWS = 7;                     // input rows feeding two output rows: 2*2 + 3
constexpr int C1_PIX_LD = 400;                     // (128 + 3 padding pixels) * 3 channels = 393 words, rounded up

struct Conv1Params {
  const void* x;           // crops NHWC, uint8 or float32
  int B, H, W, C;          // input dims (C <= 3)
  int OH, OW, N;           // output dims, N = Cout (<= 128)
  int pad_t, pad_l;
  int num_tiles;
  const float* bias;
  float unscale, out_scale, in_scale;
  __half* out_hi;
  __half* out_lo;
  unsigned* range_flag;    // run-time range guard (tc_plan.cuh): bit 0 = this layer's activation overflowed fp16 at out_scale
  long long* trace;        // AAE_C1_TRACE: clock64 stamps of CTA 0 (first 12 tiles): [i*8 + 0..2] builder start / stage free / tile built, +3,4 MMA issuer got accumulator / operands, +5,6 epilogue warp 4 start / end
};

template <int N>
struct Conv1Smem {
  static constexpr int W_BYTES = 4 * N * 128;
  static constexpr int PIX_BYTES = C1_PIX_ROWS * C1_PIX_LD * 4;       // staged input rows of one tile, (hi|lo) words
  static constexpr int OUT_BYTES = 2 * 32 * C1_OUT_LD;                // (hi, lo) output tile staged for bulk stores
  static constexpr int RAW_BYTES = ((C1_PIX_ROWS * 128 * 3 * (int)sizeof(float) + 127) / 128) * 128;   // fp32 worst case
  static constexpr int TOTAL = W_BYTES + C1_STAGES * C1_STAGE + PIX_BYTES + OUT_BYTES + RAW_BYTES + 1024 /*lut*/ + 1024 /*align*/ + 256;
};

template <bool U8>
__device__ __forceinline__ uint32_t conv1_fetch(const Conv1Params& p, const uint32_t* lut, long long idx, bool ok) {
  // returns (hi fp16 bits) | (lo fp16 bits << 16) of in_scale * pixel
  if (!ok) return 0u;
  if (U8) return lut[reinterpret_cast<const uint8_t*>(p.x)[idx]];
  const float v = __ldg(reinterpret_cast<const float*>(p.x) + idx) * p.in_scale;
  __half h, l;
  split_f16(v, h, l);
  return (uint32_t)__half_as_ushort(h) | ((uint32_t)__half_as_ushort(l) << 16);
}

template <int N, int CIN, bool U8>
__global__ void __launch_bounds__(C1_THREADS, 1)
tc_conv1_kernel(const __grid_constant__ CUtensorMap tm_w_hi, const __grid_constant__ CUtensorMap tm_w_lo, const Conv1Params p) {
  using S = Conv1Smem<N>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* w_smem = smem;                                   // hi k0, hi k1, lo k0, lo k1 (N rows x 128 B each)
  uint8_t* a_smem = smem + S::W_BYTES;
  uint32_t* pix = reinterpret_cast<uint32_t*>(a_smem + C1_STAGES * C1_STAGE);   // [C1_PIX_ROWS][C1_PIX_LD]
  uint8_t* out_smem = reinterpret_cast<uint8_t*>(pix + C1_PIX_ROWS * C1_PIX_LD);   // [2 (hi,lo)][32][C1_OUT_LD]
  uint32_t* lut = reinterpret_cast<uint32_t*>(out_smem + S::OUT_BYTES);
  uint8_t* raw_smem = reinterpret_cast<uint8_t*>(lut + 256);                    // raw input rows of the tile being staged
  uint64_t* w_full = reinterpret_cast<uint64_t*>(raw_smem + S::RAW_BYTES);
  uint64_t* a_full = w_full + 1;
  uint64_t* a_empty = a_full + C1_STAGES;
  uint64_t* acc_full = a_empty + C1_STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_empty + 2);
  __shared__ float bias_s[N];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int TMEM_COLS = 2 * N < 32 ? 32 : 2 * N;
  if (threadIdx.x < N) bias_s[threadIdx.x] = p.bias[threadIdx.x];

  if (threadIdx.x < 256) {
    // byte -> (hi, lo) of in_scale * (u8 / 255): the divide is the IEEE fp32 divide the reference's feed amounts to
    const float v = ((float)threadIdx.x / 255.0f) * p.in_scale;
    __half h, l;
    split_f16(v, h, l);
    lut[threadIdx.x] = (uint32_t)__half_as_ushort(h) | ((uint32_t)__half_as_ushort(l) << 16);
  }
  for (int i = threadIdx.x; i < C1_PIX_ROWS * C1_PIX_LD; i += blockDim.x) pix[i] = 0u;   // left/right padding pixels stay zero
  if (warp == C1_MMA_WARP && lane == 0) {
    prefetch_tmap(&tm_w_hi); prefetch_tmap(&tm_w_lo);
    mbar_init(w_full, 1);
    for (int s = 0; s < C1_STAGES; ++s) { mbar_init(&a_full[s], 128); mbar_init(&a_empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], C1_EPI_WARPS); }
    fence_barrier_init();
  }
  if (warp == C1_MMA_WARP) tmem_alloc<TMEM_COLS>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const int my_tiles = (p.num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int hw = p.OH * p.OW;

  if (warp < 4) {
    // ===================== A builders: thread r owns im2col row r of the tile =====================
    // Per tile (two output rows of one image) the 7 input rows it touches are first staged in shared memory with
    // coalesced 16-byte loads and converted ONCE to packed (hi | lo << 16) fp16 words; each builder thread then
    // assembles its 75-element patch from shared memory.  The raw rows of tile i+1 are fetched into registers before
    // tile i is built, so the global-load latency hides behind the build.
    const int r = threadIdx.x;
    constexpr int run = 5 * CIN;                             // words per kernel row (kw, c)
    constexpr int ROWW = 128 * CIN;                          // words per staged input row (image width 128)
    constexpr int NV = U8 ? (C1_PIX_ROWS * ROWW / 16 + 127) / 128 : (C1_PIX_ROWS * ROWW / 4 + 127) / 128;
    uint4 raw[NV];
    auto fetch = [&](int tile) {                             // global -> registers
      const int m_first = tile * 128;
      const int b = m_first / hw, oh0 = (m_first - b * hw) / p.OW;
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int u = r + v * 128;
        raw[v] = make_uint4(0u, 0u, 0u, 0u);
        if (U8) {
          const int row = u / (ROWW / 16), c16 = u - row * (ROWW / 16);
          const int ih = 2 * oh0 - p.pad_t + row;
          if (row < C1_PIX_ROWS && b < p.B && ih >= 0 && ih < p.H)
            raw[v] = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(p.x) + ((long long)(b * p.H + ih) * p.W) * CIN) + c16);
        } else {
          const int row = u / (ROWW / 4), c4 = u - row * (ROWW / 4);
          const int ih = 2 * oh0 - p.pad_t + row;
          if (row < C1_PIX_ROWS && b < p.B && ih >= 0 && ih < p.H)
            raw[v] = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(p.x) + ((long long)(b * p.H + ih) * p.W) * CIN) + c4);
        }
      }
    };
    uint8_t* rawbuf = raw_smem;
    auto stage = [&](uint32_t* dst) {                        // registers -> raw smem -> staged (hi|lo) words
      // step 1: park the raw 16-byte pieces (conflict-free STS.128); step 2: every thread converts CONSECUTIVE elements, so
      // the word stores to the staged rows are conflict-free too (converting 16 bytes per thread in place would put all 32
      // lanes on two banks).
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int u = r + v * 128;
        if (u < C1_PIX_ROWS * ROWW / (U8 ? 16 : 4)) reinterpret_cast<uint4*>(rawbuf)[u] = raw[v];
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      for (int e = r; e < C1_PIX_ROWS * ROWW; e += 128) {
        const int row = e / ROWW, col = e - row * ROWW;
        uint32_t w;
        if (U8) {
          w = lut[rawbuf[e]];
        } else {
          __half h, l;
          split_f16(reinterpret_cast<const float*>(rawbuf)[e] * p.in_scale, h, l);
          w = (uint32_t)__half_as_ushort(h) | ((uint32_t)__half_as_ushort(l) << 16);
        }
        dst[row * C1_PIX_LD + p.pad_l * CIN + col] = w;
      }
    };
    if (my_tiles > 0) {
      fetch((int)blockIdx.x);
      stage(pix);
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    const int ow = r % p.OW, dr = r / p.OW;
    for (int i = 0; i < my_tiles; ++i) {
      const int s = i % C1_STAGES;
      const bool more = i + 1 < my_tiles;
      if (more) fetch((int)blockIdx.x + (i + 1) * (int)gridDim.x);
      const uint32_t* src = pix + 2 * dr * C1_PIX_LD + 2 * ow * CIN;
      mbar_wait(&a_empty[s], ((uint32_t)(i / C1_STAGES) & 1u) ^ 1u);
      uint8_t* st = a_smem + s * C1_STAGE;
#pragma unroll
      for (int ci = 0; ci < C1_KPAD / 8; ++ci) {             // one 16-byte chunk = 8 K elements
        uint32_t e[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int k = ci * 8 + j;
          const int kh = k / run, jj = k - kh * run;
          e[j] = kh < 5 ? src[kh * C1_PIX_LD + jj] : 0u;
        }
        uint4 hv, lv;
        hv.x = __byte_perm(e[0], e[1], 0x5410); lv.x = __byte_perm(e[0], e[1], 0x7632);
        hv.y = __byte_perm(e[2], e[3], 0x5410); lv.y = __byte_perm(e[2], e[3], 0x7632);
        hv.z = __byte_perm(e[4], e[5], 0x5410); lv.z = __byte_perm(e[4], e[5], 0x7632);
        hv.w = __byte_perm(e[6], e[7], 0x5410); lv.w = __byte_perm(e[6], e[7], 0x7632);
        const int atom = ci >> 3, chunk = ci & 7;
        const uint32_t off = (uint32_t)(atom * C1_ATOM + r * 128 + ((chunk ^ (r & 7)) << 4));
        *reinterpret_cast<uint4*>(st + off) = hv;
        *reinterpret_cast<uint4*>(st + 2 * C1_ATOM + off) = lv;
      }
      fence_proxy_async_smem();
      mbar_arrive(&a_full[s]);
      if (more) stage(pix);                                   // (its internal barrier orders it after every thread's build of tile i)
      asm volatile("bar.sync 1, 128;" ::: "memory");       // staged rows of tile i+1 visible to all builders
    }
  } else if (warp < C1_MMA_WARP) {
    // ===================== epilogue =====================
    // The 128 pixels x 128 channels of a tile (two output rows of one image) are exactly ONE contiguous 32 KB slab of the
    // consumer's space-to-depth tensor (row oh/2, all 32 column pairs, all four parities) -- per (hi, lo).  Each thread
    // (= pixel) writes its 256 B into a padded shared-memory image of that slab; one thread then ships it with 1 KB bulk
    // stores, i.e. full-line HBM writes instead of 16-byte scattered ones.
    const int q = warp & 3, half = (warp - 4) >> 2, r = q * 32 + lane;
    const int ow = r % p.OW, dr = r / p.OW;
    // blocks are grouped G at a time (contiguous, one bulk store per group); 16 bytes of padding after every group
    constexpr int G = C1_OUT_GROUP, grp_ld = G * 8 * N + 16;
    uint8_t* my_hi = out_smem + ((ow >> 1) / G) * grp_ld + ((ow >> 1) % G) * (8 * N) + (((dr & 1) << 1) | (ow & 1)) * (2 * N);
    uint8_t* my_lo = my_hi + 32 * C1_OUT_LD;
    for (int i = 0; i < my_tiles; ++i) {
      const int as = i & 1;
      const int m_first = ((int)blockIdx.x + i * (int)gridDim.x) * 128;
      const int b = m_first / hw, oh0 = (m_first - b * hw) / p.OW;
      mbar_wait(&acc_full[as], (uint32_t)(i >> 1) & 1u);
      tc_fence_after();
      if (i > 0) {                                   // the previous tile's bulk stores must have finished reading the staging
        if (warp == 4) bulk_wait_read_all();
        asm volatile("bar.sync 2, %0;" ::"n"(32 * C1_EPI_WARPS) : "memory");
      }
#pragma unroll 1
      for (int c = half; c < N / 32; c += C1_EPI_WARPS / 4) {
        uint32_t v[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * N + c * 32), v);
        tmem_ld_wait();
        uint32_t hi[16], lo[16];
        float amax = 0.f;
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          const float a = fmaxf(__uint_as_float(v[j]) * p.unscale + bias_s[c * 32 + j], 0.f) * p.out_scale;
          const float bb = fmaxf(__uint_as_float(v[j + 1]) * p.unscale + bias_s[c * 32 + j + 1], 0.f) * p.out_scale;
          amax = fmaxf(amax, fmaxf(a, bb));
          split_f16x2(a, bb, hi[j >> 1], lo[j >> 1]);
        }
        if (p.range_flag != nullptr && !(amax < 65520.f)) atomicOr(p.range_flag, 1u);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          *reinterpret_cast<uint4*>(my_hi + c * 64 + j * 16) = make_uint4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
          *reinterpret_cast<uint4*>(my_lo + c * 64 + j * 16) = make_uint4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[as]);
      fence_proxy_async_smem();                      // generic-proxy writes -> visible to the bulk-copy engine
      asm volatile("bar.sync 2, %0;" ::"n"(32 * C1_EPI_WARPS) : "memory");
      if (warp == 4 && b < p.B) {                    // lane j ships group j (G KB) of the hi and of the lo slab
        const long long slab = ((long long)(b * (p.OH >> 1) + (oh0 >> 1)) * (p.OW >> 1)) * (4LL * N);   // elements
        if (lane < 32 / G) {
          bulk_store_1d(p.out_hi + slab + (long long)lane * G * 4 * N, out_smem + lane * grp_ld, (uint32_t)(G * 8 * N));
          bulk_store_1d(p.out_lo + slab + (long long)lane * G * 4 * N, out_smem + 32 * C1_OUT_LD + lane * grp_ld, (uint32_t)(G * 8 * N));
        }
        bulk_commit_group();
      }
    }
    if (warp == 4) bulk_wait_all();                    // all stores landed before the CTA exits
  } else {
    // ===================== weight TMA + MMA issuer (last warp) =====================
    if (lane == 0) {
      mbar_arrive_expect_tx(w_full, S::W_BYTES);
      tma_load_2d(w_smem, &tm_w_hi, w_full, 0, 0);
      tma_load_2d(w_smem + N * 128, &tm_w_hi, w_full, 64, 0);
      tma_load_2d(w_smem + 2 * N * 128, &tm_w_lo, w_full, 0, 0);
      tma_load_2d(w_smem + 3 * N * 128, &tm_w_lo, w_full, 64, 0);
      mbar_wait(w_full, 0);
      constexpr uint32_t idesc = make_idesc_f16(128, N, 0);
      const uint32_t wst = smem_u32(w_smem);
      for (int i = 0; i < my_tiles; ++i) {
        const int s = i % C1_STAGES, as = i & 1;
        mbar_wait(&acc_empty[as], ((uint32_t)(i >> 1) & 1u) ^ 1u);
        mbar_wait(&a_full[s], (uint32_t)(i / C1_STAGES) & 1u);
        tc_fence_after();
        const uint32_t ast = smem_u32(a_smem + s * C1_STAGE);
        const uint32_t d = tmem_base + (uint32_t)(as * N);
#pragma unroll
        for (int k = 0; k < C1_KPAD / 16; ++k) {
          const int atom = k >> 2, kk = k & 3;
          const uint64_t a_hi = desc_advance_k(make_sw128_kmajor_desc(ast + atom * C1_ATOM), kk);
          const uint64_t a_lo = desc_advance_k(make_sw128_kmajor_desc(ast + (2 + atom) * C1_ATOM), kk);
          const uint64_t w_hi = desc_advance_k(make_sw128_kmajor_desc(wst + atom * N * 128), kk);
          const uint64_t w_lo = desc_advance_k(make_sw128_kmajor_desc(wst + (2 + atom) * N * 128), kk);
          umma_f16(d, a_lo, w_hi, idesc, k > 0 ? 1u : 0u);
          umma_f16(d, a_hi, w_lo, idesc, 1u);
          umma_f16(d, a_hi, w_hi, idesc, 1u);
        }
        umma_commit(&a_empty[s]);
        umma_commit(&acc_full[as]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == C1_MMA_WARP) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}


// =====================================================================================================================
// uint8 feed, second generation (the path for uint8 crops; the kernel above takes those whose pointer is not 16-byte aligned).
// The first kernel ran at 0.35 of the HBM write roofline: 3.9 k shared-memory wavefronts per 128-pixel tile against an HBM
// budget of 2.8 k cycles per tile.  What changed:
//   * 1/255 is folded into the packed weights, so the A operand is the BYTE ITSELF as fp16 -- exact, no lo plane: two
//     products per K step (A*W_hi + A*W_lo) instead of three, half the A-tile bytes, and no lookup table;
//   * K is laid out as 5 kernel rows x 16 slots (slot 0 of every row meets a zero weight, slots 1..15 are the 15 (kw, c)
//     taps), so a kernel row of a pixel's patch is 32 contiguous, 4-byte-aligned bytes of the staged input row: 40 LDS.32 +
//     10 STS.128 per builder thread and tile (before: 80 + 20), bank-conflict free (lane -> pixel order below, 800-byte rows);
//   * the staged input rows are fp16 written straight from the 16-byte global loads (byte -> fp16 is two PRMT + two HSUB2
//     per four bytes), double buffered; the A tile is double buffered too, so builders run a tile ahead of the MMAs;
//   * TMEM lane r is output "slot" r of the tile's 32 KB slab of conv2's space-to-depth input (slot = (ow/2)*4 + (oh%2)*2 +
//     ow%2), so the staged output tile is the slab in order; it is written in the 128-byte-swizzle layout (conflict-free
//     STS.128) and leaves through eight 8 KB TMA tensor stores per tile, issued in two phases so that the staging double-buffers
//     itself (instead of 32 bulk copies behind a full stop).
constexpr int U8_A_STAGES = 2;
constexpr int U8_A_STAGE = 2 * C1_ATOM;           // K slots [0,64) and [64,80): two 128-row x 128-byte atoms
constexpr int U8_PIX_LD = 400;                    // fp16 elements per staged input row: 8 lead-in + 384 data + 8 tail
constexpr int U8_PIX_BUF = C1_PIX_ROWS * U8_PIX_LD * 2;   // bytes
constexpr int U8_W_BYTES = 4 * C1_ATOM;
constexpr int U8_OUT_BYTES = 4 * C1_ATOM;         // hi ch[0,64), hi ch[64,128), lo ch[0,64), lo ch[64,128): 128 slots x 128 B each
constexpr int U8_SMEM_TOTAL = U8_W_BYTES + U8_A_STAGES * U8_A_STAGE + U8_OUT_BYTES + 2 * U8_PIX_BUF + 1024 /*align*/ + 256 /*barriers*/;

// four bytes -> four fp16 (exact): 0x6400 | b is the fp16 1024 + b, minus 1024
__device__ __forceinline__ void bytes_to_half4(uint32_t x, uint32_t& lo2, uint32_t& hi2) {
  const __half2 k1024 = __floats2half2_rn(1024.f, 1024.f);
  const uint32_t a = __byte_perm(x, 0x64646464u, 0x4140), b = __byte_perm(x, 0x64646464u, 0x4342);
  const __half2 ha = __hsub2(*reinterpret_cast<const __half2*>(&a), k1024), hb = __hsub2(*reinterpret_cast<const __half2*>(&b), k1024);
  lo2 = *reinterpret_cast<const uint32_t*>(&ha);
  hi2 = *reinterpret_cast<const uint32_t*>(&hb);
}

// Epilogue warps of the uint8 kernel: 16, four per TMEM lane quadrant, one 32-channel chunk of the tile each.
// In-kernel trace (profiles/r02_conv1_trace.txt): the epilogue paces the kernel -- one chunk costs a warp ~1.7 k cycles of mostly
// latency (TMEM load, split, proxy fence, tensor-store issue), the builders and the MMAs are far ahead.
constexpr int U8_EPI_WARPS = 16;
constexpr int U8_THREADS = 32 * (4 + U8_EPI_WARPS + 1);

__global__ void __launch_bounds__(U8_THREADS, 1)
tc_conv1_u8_kernel(const __grid_constant__ CUtensorMap tm_w_hi, const __grid_constant__ CUtensorMap tm_w_lo,
                   const __grid_constant__ CUtensorMap tm_out_hi, const __grid_constant__ CUtensorMap tm_out_lo, const Conv1Params p) {
  constexpr int N = 128, CIN = 3;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* w_smem = smem;                                   // hi k0, hi k1, lo k0, lo k1 (128 rows x 128 B each)
  uint8_t* a_smem = w_smem + U8_W_BYTES;
  uint8_t* out_smem = a_smem + U8_A_STAGES * U8_A_STAGE;
  uint8_t* pix = out_smem + U8_OUT_BYTES;                   // [2][C1_PIX_ROWS][U8_PIX_LD] fp16
  uint64_t* w_full = reinterpret_cast<uint64_t*>(pix + 2 * U8_PIX_BUF);
  uint64_t* a_full = w_full + 1;
  uint64_t* a_empty = a_full + U8_A_STAGES;
  uint64_t* acc_full = a_empty + U8_A_STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_empty + 2);
  __shared__ float bias_s[N];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int n_epi = U8_EPI_WARPS, mma_warp = 4 + n_epi;                 // the epilogue warps, then the issuer warp
  constexpr int TMEM_COLS = 2 * N;
  if (threadIdx.x < N) bias_s[threadIdx.x] = p.bias[threadIdx.x] * p.out_scale;     // relu(x) * s == relu(x * s) for s > 0
  for (int i = threadIdx.x; i < 2 * U8_PIX_BUF / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(pix)[i] = 0u;   // lead-in / tail stay zero
  if (warp == mma_warp && lane == 0) {
    prefetch_tmap(&tm_w_hi); prefetch_tmap(&tm_w_lo); prefetch_tmap(&tm_out_hi); prefetch_tmap(&tm_out_lo);
    mbar_init(w_full, 1);
    for (int s = 0; s < U8_A_STAGES; ++s) { mbar_init(&a_full[s], 128); mbar_init(&a_empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], n_epi); }
    fence_barrier_init();
  }
  if (warp == mma_warp) tmem_alloc<TMEM_COLS>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const int my_tiles = (p.num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int hw = p.OH * p.OW;

  if (warp < 4) {
    // ===================== A builders: thread r owns output slot r of the tile =====================
    const int r = threadIdx.x;
    const int ow = ((r >> 2) << 1) | (r & 1), dr = (r >> 1) & 1;
    constexpr int ROW16 = 128 * CIN / 16;                    // 16-byte pieces per input row (24)
    constexpr int NPIECE = C1_PIX_ROWS * ROW16;              // 168 per tile: threads 0..127 take one, threads 0..39 a second
    uint4 raw[2];
    auto fetch = [&](int tile) {                             // global -> registers (rows outside the image: zeros)
      const int m_first = tile * 128;
      const int b = m_first / hw, oh0 = (m_first - b * hw) / p.OW;
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        const int u = r + v * 128;
        raw[v] = make_uint4(0u, 0u, 0u, 0u);
        const int row = u / ROW16, c16 = u - row * ROW16;
        const int ih = 2 * oh0 - p.pad_t + row;
        if (u < NPIECE && b < p.B && ih >= 0 && ih < p.H)
          raw[v] = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(p.x) + ((long long)(b * p.H + ih) * p.W) * CIN) + c16);
      }
    };
    auto stage = [&](uint8_t* buf) {                         // registers -> fp16 staged rows (data starts 8 elements into a row)
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        const int u = r + v * 128;
        if (u < NPIECE) {
          const int row = u / ROW16, c16 = u - row * ROW16;
          uint4 o0, o1;
          bytes_to_half4(raw[v].x, o0.x, o0.y);
          bytes_to_half4(raw[v].y, o0.z, o0.w);
          bytes_to_half4(raw[v].z, o1.x, o1.y);
          bytes_to_half4(raw[v].w, o1.z, o1.w);
          uint4* dst = reinterpret_cast<uint4*>(buf + row * (U8_PIX_LD * 2) + 16 + c16 * 32);
          dst[0] = o0;
          dst[1] = o1;
        }
      }
    };
    if (my_tiles > 0) {
      fetch((int)blockIdx.x);
      stage(pix);
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    for (int i = 0; i < my_tiles; ++i) {
      const int s = i % U8_A_STAGES;
      const bool more = i + 1 < my_tiles;
      const bool tr = p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0 && i < 12;
      if (tr) p.trace[i * 8 + 0] = clock64();
      if (more) fetch((int)blockIdx.x + (i + 1) * (int)gridDim.x);
      // kernel row kh of this pixel's patch = elements [4 + 6*ow, +16) of staged row 2*dr + kh: slot 0 is the element before the
      // patch (zero weight), slots 1..15 the 5 x 3 taps
      const uint8_t* src = pix + (i & 1) * U8_PIX_BUF + (2 * dr) * (U8_PIX_LD * 2) + (4 + 6 * ow) * 2;
      mbar_wait(&a_empty[s], ((uint32_t)(i / U8_A_STAGES) & 1u) ^ 1u);
      uint8_t* st = a_smem + s * U8_A_STAGE;
      if (tr) p.trace[i * 8 + 1] = clock64();
#pragma unroll
      for (int kh = 0; kh < 5; ++kh) {
        const uint32_t* q = reinterpret_cast<const uint32_t*>(src + kh * (U8_PIX_LD * 2));
        const uint4 c0 = make_uint4(q[0], q[1], q[2], q[3]), c1 = make_uint4(q[4], q[5], q[6], q[7]);
        const int atom = kh >> 2, ci = (kh & 3) * 2;
        uint8_t* row = st + atom * C1_ATOM + r * 128;
        *reinterpret_cast<uint4*>(row + (((ci) ^ (r & 7)) << 4)) = c0;
        *reinterpret_cast<uint4*>(row + (((ci + 1) ^ (r & 7)) << 4)) = c1;
      }
      fence_proxy_async_smem();
      mbar_arrive(&a_full[s]);
      if (tr) p.trace[i * 8 + 2] = clock64();
      if (more) stage(pix + ((i + 1) & 1) * U8_PIX_BUF);    // that buffer's last readers (tile i-1) passed the barrier below an iteration ago
      asm volatile("bar.sync 1, 128;" ::: "memory");
    }
  } else if (warp < mma_warp) {
    // ===================== epilogue: TMEM -> bias + ReLU + (hi, lo) split -> swizzled staging -> TMA tensor stores =====================
    // Warp (q, g) owns the tile's slots [32 q, 32 q + 32) and the 32-channel chunks g, g + groups, ... (groups = n_epi / 4: one
    // chunk per tile).  A chunk goes through 4 KB of the warp's own staging (hi 2 KB, lo 2 KB, 64-byte rows, 64-byte swizzle:
    // conflict-free STS.128 from a thread-per-slot warp) and is shipped by the warp's own lane 0, so the tile's tensor stores are
    // issued by n_epi lanes in parallel and no barrier couples the warps.  The buffer is reused a whole tile later.
    constexpr int groups = n_epi >> 2, per_warp = 4 / groups;
    const int q = warp & 3, g = (warp - 4) >> 2;
    const float us = p.unscale * p.out_scale;
    const int rsw = (lane >> 1) & 3;
    uint8_t* wbuf = out_smem + (warp - 4) * (U8_OUT_BYTES / n_epi);
    int ph = 0;
    for (int i = 0; i < my_tiles; ++i) {
      const int as = i & 1;
      const int tile = (int)blockIdx.x + i * (int)gridDim.x;
      mbar_wait(&acc_full[as], (uint32_t)(i >> 1) & 1u);
      tc_fence_after();
      const bool tr = p.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 128 && i < 12;
      if (tr) p.trace[i * 8 + 5] = clock64();
#pragma unroll 1
      for (int cc = 0; cc < per_warp; ++cc, ++ph) {
        const int c0 = (g + cc * groups) * 32;           // first channel of this chunk
        uint32_t v[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * N + c0), v);
        tmem_ld_wait();
        if (cc == per_warp - 1) {                        // this warp's TMEM columns have been read: the accumulator may be overwritten
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[as]);
        }
        uint32_t hi[16], lo[16];
        float amax = 0.f;
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          const float a = fmaxf(fmaf(__uint_as_float(v[j]), us, bias_s[c0 + j]), 0.f);
          const float bb = fmaxf(fmaf(__uint_as_float(v[j + 1]), us, bias_s[c0 + j + 1]), 0.f);
          amax = fmaxf(amax, fmaxf(a, bb));
          split_f16x2(a, bb, hi[j >> 1], lo[j >> 1]);
        }
        if (p.range_flag != nullptr && !(amax < 65520.f)) atomicOr(p.range_flag, 1u);
        if (ph >= per_warp) {                            // the buffer was shipped per_warp chunks ago: only newer groups may still be unread
          if (lane == 0) bulk_wait_read_all();
          __syncwarp();
        }
        uint8_t* sb = wbuf + cc * 4096;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int ch = (j ^ rsw) << 4;
          *reinterpret_cast<uint4*>(sb + lane * 64 + ch) = make_uint4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
          *reinterpret_cast<uint4*>(sb + 2048 + lane * 64 + ch) = make_uint4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
        }
        fence_proxy_async_smem();                        // generic-proxy writes -> visible to the TMA engine
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tm_out_hi, sb, c0, tile * 128 + q * 32);
          tma_store_2d(&tm_out_lo, sb + 2048, c0, tile * 128 + q * 32);
          bulk_commit_group();
        }
      }
      if (tr) p.trace[i * 8 + 6] = clock64();
    }
    if (lane == 0) bulk_wait_all();                      // all stores landed before the CTA exits
  } else {
    // ===================== weight TMA + MMA issuer (last warp) =====================
    if (lane == 0) {
      mbar_arrive_expect_tx(w_full, U8_W_BYTES);
      tma_load_2d(w_smem, &tm_w_hi, w_full, 0, 0);
      tma_load_2d(w_smem + C1_ATOM, &tm_w_hi, w_full, 64, 0);
      tma_load_2d(w_smem + 2 * C1_ATOM, &tm_w_lo, w_full, 0, 0);
      tma_load_2d(w_smem + 3 * C1_ATOM, &tm_w_lo, w_full, 64, 0);
      mbar_wait(w_full, 0);
      constexpr uint32_t idesc = make_idesc_f16(128, N, 0);
      const uint32_t wst = smem_u32(w_smem);
      for (int i = 0; i < my_tiles; ++i) {
        const int s = i % U8_A_STAGES, as = i & 1;
        mbar_wait(&acc_empty[as], ((uint32_t)(i >> 1) & 1u) ^ 1u);
        if (p.trace != nullptr && blockIdx.x == 0 && i < 12) p.trace[i * 8 + 3] = clock64();
        mbar_wait(&a_full[s], (uint32_t)(i / U8_A_STAGES) & 1u);
        if (p.trace != nullptr && blockIdx.x == 0 && i < 12) p.trace[i * 8 + 4] = clock64();
        tc_fence_after();
        const uint32_t ast = smem_u32(a_smem + s * U8_A_STAGE);
        const uint32_t d = tmem_base + (uint32_t)(as * N);
#pragma unroll
        for (int k = 0; k < C1_KPAD / 16; ++k) {
          const int atom = k >> 2, kk = k & 3;
          const uint64_t a = desc_advance_k(make_sw128_kmajor_desc(ast + atom * C1_ATOM), kk);
          const uint64_t w_hi = desc_advance_k(make_sw128_kmajor_desc(wst + atom * C1_ATOM), kk);
          const uint64_t w_lo = desc_advance_k(make_sw128_kmajor_desc(wst + (2 + atom) * C1_ATOM), kk);
          umma_f16(d, a, w_lo, idesc, k > 0 ? 1u : 0u);
          umma_f16(d, a, w_hi, idesc, 1u);
        }
        umma_commit(&a_empty[s]);
        umma_commit(&acc_full[as]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == mma_warp) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// W fp32 [75][N] (HWIO flattened) -> (hi, lo) fp16 [N][128] in the 5 x 16 slot order of the uint8 kernel: slot kh*16 + 1 + (kw*3 + c)
// holds scale * W[kh][kw][c][n] (scale = 2^16 / 255: the x/255 of codebook.py:58-59 lives here), every other slot is zero
__global__ void pack_conv1_u8_weights_kernel(const float* __restrict__ w, int N, float scale, __half* __restrict__ hi, __half* __restrict__ lo,
                                             unsigned* __restrict__ range_flag, unsigned range_bit) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * 128) return;
  const int n = i / 128, k = i - n * 128;
  const int kh = k >> 4, j = k & 15;
  const float v = (kh < 5 && j >= 1) ? w[(long long)(kh * 15 + j - 1) * N + n] * scale : 0.f;
  if (range_flag != nullptr && !(fabsf(v) < 65520.f)) atomicOr(range_flag, range_bit);
  __half h, l;
  split_f16(v, h, l);
  hi[i] = h;
  lo[i] = l;
}

// W fp32 [75][N] (HWIO flattened) -> (hi, lo) fp16 [N][128] K-major, scaled, zero for k >= K
__global__ void pack_conv1_weights_kernel(const float* __restrict__ w, int K, int N, float scale, __half* __restrict__ hi, __half* __restrict__ lo,
                                          unsigned* __restrict__ range_flag, unsigned range_bit) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * 128) return;
  const int n = i / 128, k = i - n * 128;
  const float v = k < K ? w[(long long)k * N + n] * scale : 0.f;
  if (range_flag != nullptr && !(fabsf(v) < 65520.f)) atomicOr(range_flag, range_bit);
  __half h, l;
  split_f16(v, h, l);
  hi[i] = h;
  lo[i] = l;
}

}  // namespace

struct TcConv1 {
  int N, sm_count;
  __half *w_hi = nullptr, *w_lo = nullptr;
  CUtensorMap tm_hi, tm_lo;
  // uint8 kernel: weights with 1/255 folded in, 5 x 16 slot order; output tensor maps over conv2's (hi, lo) input
  __half *w8_hi = nullptr, *w8_lo = nullptr;
  CUtensorMap tm8_hi, tm8_lo, tm_out32_hi, tm_out32_lo;   // output maps: one box = a warp's 32 slots x 32 channels
  const __half *bound_hi = nullptr, *bound_lo = nullptr;
  long long slots = 0;            // 256-byte output slots the tensor maps cover ((b, oh/2, ow/2, parity) positions)
  bool u8_ok = false;
};

bool tc_conv1_supported(const aae_net_cfg* cfg) {
  const int oh = (cfg->in_h + 1) / 2, ow = (cfg->in_w + 1) / 2;
  return cfg->kernel_size == 5 && cfg->strides[0] == 2 && cfg->in_c == 3 && cfg->filters[0] == 128 && (ow & (ow - 1)) == 0 &&
         ow == 64 && (oh % 2) == 0 && cfg->in_w == 128 && (cfg->in_h % 2 == 0);   // staging is laid out for 128-pixel-wide crops
}

int tc_conv1_create(int device, const aae_net_cfg* cfg, TcConv1** out) {
  *out = nullptr;
  TcConv1* h = new TcConv1();
  h->N = cfg->filters[0];
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  h->sm_count = prop.multiProcessorCount;
  cudaError_t e = cudaMalloc(&h->w_hi, (size_t)h->N * 128 * sizeof(__half));
  if (e == cudaSuccess) e = cudaMalloc(&h->w_lo, (size_t)h->N * 128 * sizeof(__half));
  if (e != cudaSuccess) { set_error("tc conv1 alloc failed: %s", cudaGetErrorString(e)); tc_conv1_destroy(h); return AAE_ERR_OOM; }
  const uint64_t dims[2] = {128, (uint64_t)h->N};
  const uint64_t strides[1] = {256};
  const uint32_t box[2] = {64, (uint32_t)h->N};
  int st = make_tmap_f16(&h->tm_hi, h->w_hi, 2, dims, strides, box);
  if (st == AAE_OK) st = make_tmap_f16(&h->tm_lo, h->w_lo, 2, dims, strides, box);
  if (st == AAE_OK && h->N == 128) {
    e = cudaMalloc(&h->w8_hi, (size_t)h->N * 128 * sizeof(__half));
    if (e == cudaSuccess) e = cudaMalloc(&h->w8_lo, (size_t)h->N * 128 * sizeof(__half));
    if (e != cudaSuccess) { set_error("tc conv1 alloc failed: %s", cudaGetErrorString(e)); tc_conv1_destroy(h); return AAE_ERR_OOM; }
    st = make_tmap_f16(&h->tm8_hi, h->w8_hi, 2, dims, strides, box);
    if (st == AAE_OK) st = make_tmap_f16(&h->tm8_lo, h->w8_lo, 2, dims, strides, box);
    if (st == AAE_OK) st = cudaFuncSetAttribute(tc_conv1_u8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, U8_SMEM_TOTAL) == cudaSuccess ? AAE_OK : AAE_ERR_CUDA;
    h->u8_ok = st == AAE_OK;
  }
  if (st != AAE_OK) { tc_conv1_destroy(h); return st; }
  *out = h;
  return AAE_OK;
}

void tc_conv1_destroy(TcConv1* h) {
  if (!h) return;
  cudaFree(h->w_hi); cudaFree(h->w_lo); cudaFree(h->w8_hi); cudaFree(h->w8_lo);
  delete h;
}

int tc_conv1_pack(TcConv1* h, const float* w_dev, int K, float w_scale, unsigned* range_flag, unsigned range_bit, cudaStream_t s) {
  pack_conv1_weights_kernel<<<(unsigned)ceil_div(h->N * 128, 256), 256, 0, s>>>(w_dev, K, h->N, w_scale, h->w_hi, h->w_lo, range_flag, range_bit);
  AAE_LAUNCH_OK();
  if (h->u8_ok) {
    AAE_REQUIRE(K == 75, "tc conv1 (uint8 kernel): K = %d, expected 75", K);
    pack_conv1_u8_weights_kernel<<<(unsigned)ceil_div(h->N * 128, 256), 256, 0, s>>>(w_dev, h->N, w_scale * 256.f / 255.f, h->w8_hi, h->w8_lo, range_flag,
                                                                                    range_bit);
    AAE_LAUNCH_OK();
  }
  return AAE_OK;
}

int tc_conv1_forward(TcConv1* h, const aae_net_cfg* cfg, const void* crops, int src_u8, int B, const float* bias, float act_scale,
                     float w_scale, __half* out_hi, __half* out_lo, unsigned* range_flag, cudaStream_t s) {
  Conv1Params p;
  p.trace = nullptr;
  p.range_flag = range_flag;
  p.x = crops; p.B = B; p.H = cfg->in_h; p.W = cfg->in_w; p.C = cfg->in_c;
  p.OH = cfg->in_h / 2; p.OW = cfg->in_w / 2; p.N = h->N;
  p.pad_t = std::max((p.OH - 1) * 2 + 5 - p.H, 0) / 2;
  p.pad_l = std::max((p.OW - 1) * 2 + 5 - p.W, 0) / 2;
  p.num_tiles = (int)ceil_div((int64_t)B * p.OH * p.OW, 128);
  p.bias = bias;
  p.in_scale = act_scale; p.out_scale = act_scale; p.unscale = 1.f / (act_scale * w_scale);
  p.out_hi = out_hi; p.out_lo = out_lo;
  const int grid = std::min(h->sm_count, p.num_tiles);
  using S = Conv1Smem<128>;
  if (src_u8 && h->u8_ok && (reinterpret_cast<uintptr_t>(crops) & 15u) == 0) {   // 16-byte row pieces are loaded as uint4
    // output tensor maps: [slot][128 channels] views of conv2's (hi, lo) input; the buffers hold max_batch crops, this call
    // may be shorter -- the maps cover exactly the slots this call writes
    const long long slots = (long long)p.num_tiles * 128;
    if (h->bound_hi != out_hi || h->bound_lo != out_lo || h->slots != slots) {
      const uint64_t dims[2] = {128, (uint64_t)slots};
      const uint64_t strides[1] = {256};
      const uint32_t box32[2] = {32, 32};                   // one warp's 32 slots x 32 channels, 64-byte swizzle
      AAE_TRY(make_tmap_f16(&h->tm_out32_hi, out_hi, 2, dims, strides, box32, 64));
      AAE_TRY(make_tmap_f16(&h->tm_out32_lo, out_lo, 2, dims, strides, box32, 64));
      h->bound_hi = out_hi; h->bound_lo = out_lo; h->slots = slots;
    }
    p.unscale = 1.f / (w_scale * 256.f);              // accumulators hold sum u8 * (w * w_scale * 256 / 255)
    static long long* trace_dev = nullptr;
    p.trace = nullptr;
    if (getenv("AAE_C1_TRACE")) {
      if (!trace_dev) cudaMalloc(&trace_dev, 96 * sizeof(long long));
      cudaMemsetAsync(trace_dev, 0, 96 * sizeof(long long), s);
      p.trace = trace_dev;
    }
    tc_conv1_u8_kernel<<<grid, U8_THREADS, U8_SMEM_TOTAL, s>>>(h->tm8_hi, h->tm8_lo, h->tm_out32_hi, h->tm_out32_lo, p);
    if (p.trace) {
      long long t[96];
      cudaStreamSynchronize(s);
      cudaMemcpy(t, p.trace, sizeof(t), cudaMemcpyDeviceToHost);
      fprintf(stderr, "[conv1 trace, CTA 0, clocks from the first builder stamp] tile: builder start | stage free | built || issuer: accumulator free | operands ready || epilogue warp 4: start | end\n");
      for (int i = 0; i < 12; ++i)
        fprintf(stderr, "  tile %2d: %6lld | %6lld | %6lld || %6lld | %6lld || %6lld | %6lld\n", i, t[i * 8] - t[0], t[i * 8 + 1] - t[0], t[i * 8 + 2] - t[0],
                t[i * 8 + 3] - t[0], t[i * 8 + 4] - t[0], t[i * 8 + 5] - t[0], t[i * 8 + 6] - t[0]);
    }
  } else if (src_u8) {
    AAE_CUDA_OK(cudaFuncSetAttribute(tc_conv1_kernel<128, 3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
    tc_conv1_kernel<128, 3, true><<<grid, C1_THREADS, S::TOTAL, s>>>(h->tm_hi, h->tm_lo, p);
  } else {
    AAE_CUDA_OK(cudaFuncSetAttribute(tc_conv1_kernel<128, 3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL));
    tc_conv1_kernel<128, 3, false><<<grid, C1_THREADS, S::TOTAL, s>>>(h->tm_hi, h->tm_lo, p);
  }
  AAE_LAUNCH_OK();
  return AAE_OK;
}

}  // namespace aae
