// Execution-plan structures of the tensor-core path, shared by tc_gemm.cu (inference plans, GEMM kernels) and
// tc_train.cu (backward plans).  Internal to the library.
#pragma once
#include <vector>

#include "tc.cuh"
#include "tc_common.cuh"

namespace aae {

enum TcOutMode : int {
  OUT_S2D_SPLIT = 0,      // (hi, lo) fp16, space-to-depth layout of the next stride-2 conv
  OUT_PLAIN_SPLIT = 1,    // (hi, lo) fp16, plain [M, N]
  OUT_F32 = 2,            // fp32 [splits, M, N] raw accumulators (split-K partials)
  OUT_D2S_SPLIT = 3,      // (hi, lo) fp16, depth-to-space: column (cls, co) of pixel (b,i,j) -> pixel (2i+py, 2j+px) of [B,2OH,2OW,N/4]
  OUT_D2S_F32 = 4         // fp32, depth-to-space with `cout_real` channels per parity (decoder output layer, N padded)
};

struct TcGemmParams {
  int M;                 // valid output rows (pixels, or batch rows for the dense layer)
  int N;                 // total output channels
  int OH, OW;            // output spatial dims (1,1 for dense)
  int BW, BH;            // pixel box of one 128-row tile: BW*BH*BB = 128
  int taps;              // 25 (conv) or 1 (dense)
  int chunks_per_tap;    // Cin / 64
  int iters_per_split;   // K iterations (tap, chunk) handled per blockIdx.z
  int8_t tap_di[32], tap_dj[32];
  int tap_ch[32];        // channel offset of the tap's parity plane in the space-to-depth tensor
  float unscale;         // 1 / (scale_A * scale_W)
  const unsigned* amax_bits;  // optional: the A operand was scaled by tc_dyn_scale(*amax_bits) (training gradients); folded into unscale
  float out_scale;       // scale applied before the hi/lo split of the output (next layer's scale_A)
  const float* bias;
  int relu;              // activation: 0 none, 1 ReLU, 2 sigmoid
  int cout_real;         // OUT_D2S_F32: real channels per parity class (columns >= 4*cout_real are padding)
  int out_mode;
  __half* out_hi;
  __half* out_lo;
  float* out_f32;        // OUT_F32: [splits, M, N]
  // run-time range guard of the static fp16 scaling: an output whose magnitude times out_scale would round to fp16 infinity
  // (|activation| >= 4094 at scale 16) sets `range_bit` in *range_flag instead of producing inf/garbage silently
  unsigned* range_flag;
  unsigned range_bit;
};

constexpr float TC_F16_OVERFLOW = 65520.f;   // smallest magnitude that rounds to infinity in fp16 (round to nearest even)



// Power-of-two scale that places a tensor whose largest magnitude is `amax` (given as fp32 bits) into [2^13, 2^14): the hi/lo
// fp16 split then keeps 22 significant bits for everything within ~2^-16 of the largest element and cannot overflow.
__host__ __device__ __forceinline__ int tc_dyn_exponent(unsigned amax_bits) {
  int e = (int)((amax_bits >> 23) & 0xffu) - 127;            // amax in [2^e, 2^(e+1))
  return e < -100 ? -100 : (e > 100 ? 100 : e);
}
__device__ __forceinline__ float tc_dyn_scale(unsigned amax_bits) { return __int_as_float((127 + 13 - tc_dyn_exponent(amax_bits)) << 23); }
__device__ __forceinline__ float tc_dyn_unscale(unsigned amax_bits) { return __int_as_float((127 - 13 + tc_dyn_exponent(amax_bits)) << 23); }

constexpr float ACT_SCALE = 16.f;     // activations (and the [0,1] input) are stored as 16 * x
constexpr float W_SCALE = 256.f;      // weights are stored as 256 * w
constexpr int TC_THREADS = 512;       // warp 0 TMA, 1 MMA, 2 TMEM allocator, 3 idle, 4-15 epilogue (three per TMEM lane quadrant)
// Twelve epilogue warps instead of eight took conv2 / conv3 / conv4 from 1.029 / 0.886 / 0.458 to 1.000 / 0.871 / 0.452 ms (the
// exposed epilogue shrinks); four warps: 1.170 / 0.941 / 0.468 (measured on a B200 in one process, +-0.1 %).
constexpr int TC_EPI_GROUPS = (TC_THREADS / 32 - 4) / 4;   // epilogue warps per TMEM lane quadrant: each takes every third 32-column chunk

struct TcLayer {
  int in_h, in_w, in_c, out_h, out_w, out_c;   // conv geometry (input is the space-to-depth tensor [B, in_h/2, in_w/2, 4*in_c])
  int taps, BW, BH, BB;
  __half *in_hi = nullptr, *in_lo = nullptr;    // activations entering this layer
  __half *w_hi = nullptr, *w_lo = nullptr;      // packed weights [out_c][taps*in_c]
  CUtensorMap tm_a_hi, tm_a_lo, tm_w_hi, tm_w_lo;
  CUtensorMap tm_w2_hi, tm_w2_lo;               // weight tile halves (128 rows) for the CTA-pair kernel
  CUtensorMap tm_o_hi, tm_o_lo;                 // output (= next layer's input) as a store target: box = 32 pixels x 32 channels
  bool tma_out = false;                         // the persistent pair kernel may ship its epilogue through tm_o_* (TMA tensor stores)
  const float* tma_f32_base = nullptr;          // OUT_F32: tm_o_hi describes THIS buffer (fp32 [rows, N] seen as fp16 [rows, 2N]); other targets use plain stores
  bool pair = false;
  TcGemmParams gp;
  int n_tile;
  int kch;    // K chunk per pipeline stage: 64 (128-byte swizzle) or 32 (64-byte swizzle, 4 stages)
};

// bits of the range flag word: bit l = the activation written by conv layer l (0-based; the decoder counts dense_1 as 0)
// overflowed; bit 16 + l = a weight of layer l overflowed when it was packed
struct TcEncoder {
  int device;
  aae_net_cfg cfg;
  unsigned* range_flag = nullptr;   // device word, see above
  std::vector<TcLayer> layers;   // conv layers 1..L-1 followed by the dense layer
  int flat;
  float* partials = nullptr;     // dense split-K partials [splits, max_batch, latent]
  float* fwd_partials = nullptr; // conv split-K partials of small-batch forwards [splits, M, N] (allocated on first use)
  size_t fwd_partial_floats = 0;
  int dense_splits = 1;
  TcConv1* conv1 = nullptr;      // tensor-core first layer (when the geometry allows), else the fp32 SIMT kernel
  float* dbg = nullptr;          // fp32 view of an activation (tests)
  size_t dbg_floats = 0;
  bool timer_on = false;
  std::vector<cudaEvent_t> ev;
  int ev_used = 0;
};


struct TcDecoder {
  int device;
  aae_net_cfg cfg;
  unsigned* range_flag = nullptr;
  std::vector<TcLayer> layers;     // [0] dense_1, [1..L-1] sub-pixel convs, [L] sub-pixel output layer
  std::vector<float*> bias_dev;    // per layer: bias in GEMM-column order (dense: the caller's; convs: tiled 4x, padded)
  float* wm_tmp = nullptr;         // fp32 merged-weight scratch
  // Output layer with 36 * Cout <= 128 (Cout = 3): "tap-separable" form.  P[pixel, (tap, cls, co)] = X[pixel, :] . Wm[tap, :, (cls, co)]
  // is ONE 1x1 GEMM (K = Cin, N = 128) that reads the activation once instead of once per tap; the 3x3 neighbourhood sum,
  // bias, sigmoid and depth-to-space scatter happen in a small gather kernel over P.
  bool sep_out = false;
  float* out_p = nullptr;          // [B*h*w (padded to 128 rows)][128] fp32
  const float* out_bias = nullptr; // the caller's bias [Cout] (device)
  size_t wm_floats = 0;
};


// ------------------------------------------------------------------------------------------------- shared epilogue
struct TcRow {
  bool valid;
  int b, i, j;            // pixel coordinates on the OH x OW grid
  long long row_off;      // element offset of column 0 for the row-contiguous output modes
};

__device__ __forceinline__ TcRow tc_decode_row(const TcGemmParams& p, int m) {
  TcRow r;
  r.valid = m < p.M;
  r.b = r.i = r.j = 0;
  r.row_off = 0;
  if (!r.valid) return r;
  const int hw = p.OH * p.OW;
  r.b = m / hw;
  const int rem = m - r.b * hw;
  r.i = rem / p.OW;
  r.j = rem - r.i * p.OW;
  if (p.out_mode == OUT_S2D_SPLIT)
    r.row_off = ((long long)(r.b * (p.OH >> 1) + (r.i >> 1)) * (p.OW >> 1) + (r.j >> 1)) * (4LL * p.N) + (((r.i & 1) << 1) | (r.j & 1)) * p.N;
  else
    r.row_off = (long long)m * p.N;
  return r;
}

// f[0..31]: accumulator values (already hh + cross, times unscale) of columns n .. n+31 of this thread's row
__device__ __forceinline__ void tc_store_chunk(const TcGemmParams& p, const TcRow& r, int n, float (&f)[32], int split_z) {
  if (p.out_mode == OUT_F32) {
    float* dst = p.out_f32 + (long long)split_z * p.M * p.N + r.row_off + n;
#pragma unroll
    for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
    return;
  }
  // bias + activation with the mode tests hoisted out of the element loops (per-element tests made this routine ~1000 issue
  // slots per chunk, and the epilogue of a one-CTA-per-SM GEMM is exposed)
  float b[32];
  if (p.bias != nullptr) {
#pragma unroll
    for (int j = 0; j < 32; ++j) b[j] = __ldg(p.bias + n + j);
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) b[j] = 0.f;
  }
  if (p.relu == 2) {
#pragma unroll
    for (int j = 0; j < 32; ++j) f[j] = 1.f / (1.f + expf(-(f[j] + b[j])));
  } else {
    const float floor_v = p.relu == 1 ? 0.f : -INFINITY;       // fmaxf(a, -inf) = a
#pragma unroll
    for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j] + b[j], floor_v);
  }
  if (p.out_mode == OUT_D2S_F32) {
    const int cr = p.cout_real;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const int nn = n + j;
      if (nn >= 4 * cr) continue;
      const int cls = nn / cr, co = nn - cls * cr;
      p.out_f32[((long long)(r.b * 2 * p.OH + 2 * r.i + (cls >> 1)) * (2 * p.OW) + 2 * r.j + (cls & 1)) * cr + co] = f[j];
    }
    return;
  }
  long long off = r.row_off + n;
  if (p.out_mode == OUT_D2S_SPLIT) {
    const int cq = p.N >> 2, cls = n / cq, co = n - cls * cq;     // a 32-column chunk never straddles a parity class (cq % 32 == 0)
    off = ((long long)(r.b * 2 * p.OH + 2 * r.i + (cls >> 1)) * (2 * p.OW) + 2 * r.j + (cls & 1)) * cq + co;
  }
  uint32_t hi[16], lo[16];
  float amax = 0.f;
#pragma unroll
  for (int j = 0; j < 32; j += 2) {
    amax = fmaxf(amax, fmaxf(fabsf(f[j]), fabsf(f[j + 1])));
    tc::split_f16x2(f[j] * p.out_scale, f[j + 1] * p.out_scale, hi[j >> 1], lo[j >> 1]);
  }
  if (p.range_flag != nullptr && !(amax * p.out_scale < TC_F16_OVERFLOW)) atomicOr(p.range_flag, p.range_bit);
  uint4* dh = reinterpret_cast<uint4*>(p.out_hi + off);
  uint4* dl = reinterpret_cast<uint4*>(p.out_lo + off);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    dh[j] = make_uint4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
    dl[j] = make_uint4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
  }
}


// The same arithmetic as tc_store_chunk's (hi, lo) branch without its per-element mode tests, for the persistent kernel whose
// epilogue is exposed (profiles/r02_conv_gemm_trace.txt): ReLU or identity, bias absent or 16-byte aligned, any of the three
// (hi, lo) layouts.  v / x are the raw hh and cross-term accumulators.
__device__ __forceinline__ bool tc_lean_epilogue_ok(const TcGemmParams& p) {
  return (p.out_mode == OUT_S2D_SPLIT || p.out_mode == OUT_PLAIN_SPLIT || p.out_mode == OUT_D2S_SPLIT) && p.relu != 2 &&
         (reinterpret_cast<uintptr_t>(p.bias) & 15) == 0;
}
// bias + activation + range guard + (hi, lo) split of one 32-column chunk: hi[k] / lo[k] = packed fp16 pair of columns 2k, 2k+1
template <bool BIAS>
__device__ __forceinline__ void tc_lean_chunk_t(const TcGemmParams& p, int n, const uint32_t (&v)[32], const uint32_t (&x)[32], float unscale,
                                                float floor_v, uint32_t (&hi)[16], uint32_t (&lo)[16]) {
  const float4* bp = reinterpret_cast<const float4*>(p.bias + n);
  const float os = p.out_scale;
  float amax = 0.f;
#pragma unroll
  for (int j = 0; j < 32; j += 4) {
    const float4 b = BIAS ? __ldg(bp + (j >> 2)) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float a0 = fmaxf(__fadd_rn(__fmul_rn(__fadd_rn(__uint_as_float(v[j]), __uint_as_float(x[j])), unscale), b.x), floor_v);
    const float a1 = fmaxf(__fadd_rn(__fmul_rn(__fadd_rn(__uint_as_float(v[j + 1]), __uint_as_float(x[j + 1])), unscale), b.y), floor_v);
    const float a2 = fmaxf(__fadd_rn(__fmul_rn(__fadd_rn(__uint_as_float(v[j + 2]), __uint_as_float(x[j + 2])), unscale), b.z), floor_v);
    const float a3 = fmaxf(__fadd_rn(__fmul_rn(__fadd_rn(__uint_as_float(v[j + 3]), __uint_as_float(x[j + 3])), unscale), b.w), floor_v);
    amax = fmaxf(fmaxf(amax, fmaxf(fabsf(a0), fabsf(a1))), fmaxf(fabsf(a2), fabsf(a3)));
    tc::split_f16x2(a0 * os, a1 * os, hi[j >> 1], lo[j >> 1]);
    tc::split_f16x2(a2 * os, a3 * os, hi[(j >> 1) + 1], lo[(j >> 1) + 1]);
  }
  if (p.range_flag != nullptr && !(amax * os < TC_F16_OVERFLOW)) atomicOr(p.range_flag, p.range_bit);
}
__device__ __forceinline__ void tc_lean_chunk(const TcGemmParams& p, int n, const uint32_t (&v)[32], const uint32_t (&x)[32], float unscale,
                                              float floor_v, uint32_t (&hi)[16], uint32_t (&lo)[16]) {
  if (p.bias != nullptr) tc_lean_chunk_t<true>(p, n, v, x, unscale, floor_v, hi, lo);
  else tc_lean_chunk_t<false>(p, n, v, x, unscale, floor_v, hi, lo);
}
__device__ __forceinline__ void tc_store_chunk_lean(const TcGemmParams& p, const TcRow& r, int n, const uint32_t (&v)[32], const uint32_t (&x)[32],
                                                    float unscale, float floor_v) {
  uint32_t hi[16], lo[16];
  tc_lean_chunk(p, n, v, x, unscale, floor_v, hi, lo);
  long long off = r.row_off + n;
  if (p.out_mode == OUT_D2S_SPLIT) {
    const int cq = p.N >> 2, cls = n / cq, co = n - cls * cq;     // a 32-column chunk never straddles a parity class (cq % 32 == 0)
    off = ((long long)(r.b * 2 * p.OH + 2 * r.i + (cls >> 1)) * (2 * p.OW) + 2 * r.j + (cls & 1)) * cq + co;
  }
  uint4* dh = reinterpret_cast<uint4*>(p.out_hi + off);
  uint4* dl = reinterpret_cast<uint4*>(p.out_lo + off);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    dh[j] = make_uint4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
    dl[j] = make_uint4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
  }
}

// launches the GEMM kernel instantiation that matches the layer's tile shape (CTA pair / single CTA, N tile, K chunk)
int tc_launch_layer(const TcLayer& T, dim3 grid, cudaStream_t s);
int tc_dev_alloc(void** p, size_t bytes);
// Tensor maps + packed-weight storage of a layer whose A operand is a PLAIN NHWC (hi, lo) tensor [B_pad, in_h, in_w, in_c]
// (taps = unit-stride boxes): fills tm_a_*, allocates w_hi/w_lo [ceil(N / n_tile) * n_tile][taps * in_c] and their maps.
// T.{in_h,in_w,in_c,taps,BW,BH,BB,n_tile,kch,gp.N} must be set; with alloc_input = false T.in_hi/in_lo are the caller's.
int tc_layer_setup_plain(TcLayer& T, int B, bool pair_ok, bool alloc_input);
// Store-side tensor maps for the persistent pair kernel's epilogue (T.tma_out): the (hi, lo) output of a layer whose gp.out_mode
// is OUT_S2D_SPLIT / OUT_PLAIN_SPLIT / OUT_D2S_SPLIT (out_rows_pad = images the destination buffers hold), or an fp32 [rows, N]
// buffer for OUT_F32 (out_rows_pad = rows it holds).  Leaves T.tma_out false when the geometry has no 32-pixel box.
int tc_layer_setup_out_maps(TcLayer& T, long long out_rows_pad);

}  // namespace aae
