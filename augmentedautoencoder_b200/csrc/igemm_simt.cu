// SIMT fp32 implicit-GEMM: the exact-order (IEEE FMA chain) path for every dense contraction of the
// AAE hot path -- conv forward (auto_pose/ae/encoder.py:43-50, decoder.py:56-62), dense layers
// (encoder.py:62-66, decoder.py:44-51) and their backward passes (TF autodiff behind
// auto_pose/ae/ae_factory.py:86-88).  It is the correctness anchor for the tcgen05 kernels and the
// arithmetic of AAE_PREC_FP32_SIMT.
//
// One kernel, three gather modes (common.cuh):  C[M,N] = sum_k A[m,k] * Bm[k,n]
//   tile 128x128x16, 256 threads, 8x8 register micro-tile, register-prefetch double buffering.
#include <stdlib.h>

#include "common.cuh"

namespace aae {

namespace {

constexpr int BM = 128, BN = 128, BK = 16, NT = 256;
constexpr int AS_LD = BM + 4;  // keeps float4 alignment of fragment reads, 2-way conflicts on the transposing stores

struct PixCoord {
  int n, ph, pw;      // batch index and position on the indexing pixel grid
  int out_row;        // row of C this m maps to (natural NHWC order), -1 if m >= M
};

__device__ __forceinline__ PixCoord decode_pixel(const IGemmParams& p, int m, int m_limit) {
  PixCoord c;
  if (m >= m_limit) { c.n = 0; c.ph = -100000; c.pw = -100000; c.out_row = -1; return c; }
  if (p.parity_major) {
    const int per_class = m_limit >> 2;
    const int cls = m / per_class, r = m - cls * per_class;
    const int h2 = p.PH >> 1, w2 = p.PW >> 1;
    c.n = r / (h2 * w2);
    const int q = r - c.n * (h2 * w2);
    c.ph = ((q / w2) << 1) + (cls >> 1);
    c.pw = ((q % w2) << 1) + (cls & 1);
  } else {
    const int hw = p.PH * p.PW;
    c.n = m / hw;
    const int q = m - c.n * hw;
    c.ph = q / p.PW;
    c.pw = q - c.ph * p.PW;
  }
  c.out_row = (c.n * p.PH + c.ph) * p.PW + c.pw;
  return c;
}

// Source coordinate of `tap` for the indexing pixel; returns element offset (in channels units) or -1.
template <int MODE>
__device__ __forceinline__ long long gather_base(const IGemmParams& p, const PixCoord& c, int kh, int kw) {
  int sh, sw;
  if (MODE == GATHER_DGRAD) {
    int th = c.ph + p.pad_t - kh, tw = c.pw + p.pad_l - kw;
    if (p.stride == 2) {
      if ((th | tw) & 1) return -1;
      th >>= 1; tw >>= 1;
    }
    sh = th; sw = tw;
    if (sh < 0 || sw < 0 || sh >= p.SH || sw >= p.SW) return -1;
  } else {
    sh = c.ph * p.stride + kh - p.pad_t;
    sw = c.pw * p.stride + kw - p.pad_l;
    if (sh < 0 || sw < 0 || sh >= (p.SH << p.ups) || sw >= (p.SW << p.ups)) return -1;
    sh >>= p.ups; sw >>= p.ups;
  }
  return ((long long)(c.n * p.SH + sh) * p.SW + sw) * p.SC;
}

template <bool U8>
__device__ __forceinline__ float load_src(const void* src, long long idx) {
  if (U8) return (float)reinterpret_cast<const uint8_t*>(src)[idx] / 255.0f;  // IEEE divide (codebook.py:58-59)
  return __ldg(reinterpret_cast<const float*>(src) + idx);
}

template <int MODE, bool VEC, bool U8>
__global__ void __launch_bounds__(NT) igemm_f32_kernel(const IGemmParams p) {
  __shared__ __align__(16) float As[2][BK][AS_LD];
  __shared__ __align__(16) float Bs[2][BK][BN];

  const int t = threadIdx.x;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int k_begin = blockIdx.z * p.k_per_split;
  const int k_end = min(p.K, k_begin + p.k_per_split);
  const int taps = p.KH * p.KW;

  // ---- loader roles ----
  // FWD/DGRAD: rows ra0 = t>>2 and ra0+64, k sub-vector (t&3)*4.   WGRAD: pixel (t>>4), m sub-vectors (t&15)*4 and +64.
  PixCoord pc0, pc1;
  if (MODE != GATHER_WGRAD) {
    pc0 = decode_pixel(p, m0 + (t >> 2), p.M);
    pc1 = decode_pixel(p, m0 + (t >> 2) + 64, p.M);
  }
  // parity class of this tile (DGRAD, stride 2, parity-major): taps of the wrong parity contribute nothing
  int cls_h = 0, cls_w = 0;
  const bool skip_taps = (MODE == GATHER_DGRAD) && p.parity_major;
  if (skip_taps) {
    const int cls = m0 / (p.M >> 2);
    cls_h = ((cls >> 1) + p.pad_t) & 1;
    cls_w = ((cls & 1) + p.pad_l) & 1;
  }

  float4 ra[2], rb[2];

  auto chunk_valid = [&](int kc) -> bool {
    if (!skip_taps) return true;
    // all 16 k of a chunk share one tap when SC % 16 == 0 (VEC); generic path never skips
    if (!VEC) return true;
    const int tap = (kc * BK) / p.SC;
    const int kh = tap / p.KW, kw = tap - kh * p.KW;
    return ((kh & 1) == cls_h) && ((kw & 1) == cls_w);
  };

  auto load_tiles = [&](int kc) {
    const int kbase = kc * BK;
    // ---------------- A ----------------
    if (MODE != GATHER_WGRAD) {
      const int kv = (t & 3) * 4;
      if (VEC) {
        const int kk = kbase + kv;
        const int tap = kk / p.SC, ci = kk - tap * p.SC;
        const int kh = tap / p.KW, kw = tap - kh * p.KW;
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const PixCoord& c = r ? pc1 : pc0;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (kk < k_end && c.out_row >= 0) {
            const long long base = gather_base<MODE>(p, c, kh, kw);
            if (base >= 0) v = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.src) + base + ci));
          }
          ra[r] = v;
        }
      } else {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const PixCoord& c = r ? pc1 : pc0;
          float v[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int kk = kbase + kv + i;
            v[i] = 0.f;
            if (kk < k_end && c.out_row >= 0) {
              const int tap = kk / p.SC, ci = kk - tap * p.SC;
              const int kh = tap / p.KW, kw = tap - kh * p.KW;
              const long long base = gather_base<MODE>(p, c, kh, kw);
              if (base >= 0) v[i] = load_src<U8>(p.src, base + ci);
            }
          }
          ra[r] = make_float4(v[0], v[1], v[2], v[3]);
        }
      }
    } else {
      // WGRAD: k indexes pixels; A[m=(tap,ci)][pix]
      const int pix = kbase + (t >> 4);
      PixCoord c = decode_pixel(p, pix, k_end);  // k_end <= K = number of pixels
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int mv = (t & 15) * 4 + r * 64;
        const int m = m0 + mv;
        if (VEC) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (m < p.M && c.out_row >= 0) {
            const int tap = m / p.SC, ci = m - tap * p.SC;
            const int kh = tap / p.KW, kw = tap - kh * p.KW;
            const long long base = gather_base<GATHER_FWD>(p, c, kh, kw);
            if (base >= 0) v = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.src) + base + ci));
          }
          ra[r] = v;
        } else {
          float v[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            v[i] = 0.f;
            const int mm = m + i;
            if (mm < p.M && c.out_row >= 0) {
              const int tap = mm / p.SC, ci = mm - tap * p.SC;
              const int kh = tap / p.KW, kw = tap - kh * p.KW;
              const long long base = gather_base<GATHER_FWD>(p, c, kh, kw);
              if (base >= 0) v[i] = load_src<U8>(p.src, base + ci);
            }
          }
          ra[r] = make_float4(v[0], v[1], v[2], v[3]);
        }
      }
    }
    // ---------------- B ----------------
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int kk = kbase + (t >> 5) + r * 8;
      const int n = n0 + (t & 31) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (kk < k_end && n < p.N) v = __ldg(reinterpret_cast<const float4*>(p.Bm + (long long)kk * p.N + n));
      rb[r] = v;
    }
  };

  auto store_tiles = [&](int buf) {
    if (MODE != GATHER_WGRAD) {
      const int kv = (t & 3) * 4, r0 = t >> 2;
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        As[buf][kv + 0][r0 + r * 64] = ra[r].x;
        As[buf][kv + 1][r0 + r * 64] = ra[r].y;
        As[buf][kv + 2][r0 + r * 64] = ra[r].z;
        As[buf][kv + 3][r0 + r * 64] = ra[r].w;
      }
    } else {
#pragma unroll
      for (int r = 0; r < 2; ++r)
        *reinterpret_cast<float4*>(&As[buf][t >> 4][(t & 15) * 4 + r * 64]) = ra[r];
    }
#pragma unroll
    for (int r = 0; r < 2; ++r)
      *reinterpret_cast<float4*>(&Bs[buf][(t >> 5) + r * 8][(t & 31) * 4]) = rb[r];
  };

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  const int tx = t & 15, ty = t >> 4;
  const int kc_begin = k_begin / BK, kc_end = (k_end + BK - 1) / BK;

  auto next_valid = [&](int kc) {
    while (kc < kc_end && !chunk_valid(kc)) ++kc;
    return kc;
  };

  int kc = next_valid(kc_begin);
  int buf = 0;
  if (kc < kc_end) {
    load_tiles(kc);
    store_tiles(0);
  }
  __syncthreads();
  while (kc < kc_end) {
    const int kn = next_valid(kc + 1);
    if (kn < kc_end) load_tiles(kn);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][k][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (kn < kc_end) store_tiles(buf ^ 1);
    __syncthreads();
    buf ^= 1;
    kc = kn;
  }

  // ---------------- epilogue ----------------
  const bool split = gridDim.z > 1;
  float* cbase = p.C + (split ? (long long)blockIdx.z * p.M * p.N : 0);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (m >= p.M) continue;
    long long row = m;
    if (MODE != GATHER_WGRAD) row = decode_pixel(p, m, p.M).out_row;
#pragma unroll
    for (int jh = 0; jh < 2; ++jh) {
      const int n = n0 + jh * 64 + tx * 4;
      if (n >= p.N) continue;
      float v[4] = {acc[i][jh * 4 + 0], acc[i][jh * 4 + 1], acc[i][jh * 4 + 2], acc[i][jh * 4 + 3]};
      if (!split) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (p.bias) v[j] += __ldg(p.bias + n + j);
          if (p.act == ACT_RELU) v[j] = fmaxf(v[j], 0.f);
          else if (p.act == ACT_SIGMOID) v[j] = 1.f / (1.f + expf(-v[j]));
        }
        if (p.relu_mask) {
          const float4 mk = __ldg(reinterpret_cast<const float4*>(p.relu_mask + row * p.N + n));
          v[0] = mk.x > 0.f ? v[0] : 0.f; v[1] = mk.y > 0.f ? v[1] : 0.f;
          v[2] = mk.z > 0.f ? v[2] : 0.f; v[3] = mk.w > 0.f ? v[3] : 0.f;
        }
      }
      if (MODE == GATHER_FWD && p.split_hi != nullptr) {
        long long o = row * p.N + n;
        if (p.split_s2d) {
          const PixCoord pc = decode_pixel(p, m, p.M);
          o = ((long long)(pc.n * (p.PH >> 1) + (pc.ph >> 1)) * (p.PW >> 1) + (pc.pw >> 1)) * (4LL * p.N) +
              (((pc.ph & 1) << 1) | (pc.pw & 1)) * p.N + n;
        }
        __half h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float x = v[j] * p.split_scale;
          h[j] = __float2half_rn(x);
          l[j] = __float2half_rn(x - __half2float(h[j]));
        }
        uint2 hv, lv;
        hv.x = (uint32_t)__half_as_ushort(h[0]) | ((uint32_t)__half_as_ushort(h[1]) << 16);
        hv.y = (uint32_t)__half_as_ushort(h[2]) | ((uint32_t)__half_as_ushort(h[3]) << 16);
        lv.x = (uint32_t)__half_as_ushort(l[0]) | ((uint32_t)__half_as_ushort(l[1]) << 16);
        lv.y = (uint32_t)__half_as_ushort(l[2]) | ((uint32_t)__half_as_ushort(l[3]) << 16);
        *reinterpret_cast<uint2*>(p.split_hi + o) = hv;
        *reinterpret_cast<uint2*>(p.split_lo + o) = lv;
      } else if (MODE == GATHER_FWD && p.d2s_out && !split) {
        const PixCoord pc = decode_pixel(p, m, p.M);
        const int co_n = p.N >> 2, cls = n / co_n, co = n - cls * co_n;
        const long long o = ((long long)(pc.n * 2 * p.PH + 2 * pc.ph + (cls >> 1)) * (2 * p.PW) + 2 * pc.pw + (cls & 1)) * co_n + co;
        *reinterpret_cast<float4*>(p.C + o) = make_float4(v[0], v[1], v[2], v[3]);
      } else {
        *reinterpret_cast<float4*>(cbase + row * p.N + n) = make_float4(v[0], v[1], v[2], v[3]);
      }
    }
  }
}

__global__ void splitk_reduce_kernel(const float* __restrict__ partials, int splits, long long MN, int N,
                                     const float* __restrict__ bias, int act, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= MN) return;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += partials[(long long)z * MN + i];  // fixed order: deterministic
  if (bias) s += bias[i % N];
  if (act == ACT_RELU) s = fmaxf(s, 0.f);
  else if (act == ACT_SIGMOID) s = 1.f / (1.f + expf(-s));
  out[i] = s;
}

// float4 variant for MN % 4 == 0, N % 4 == 0 (every large caller): 4x fewer threads, 16-byte accesses
__global__ void splitk_reduce4_kernel(const float4* __restrict__ partials, int splits, long long MN4, int N4, const float4* __restrict__ bias,
                                      int act, float4* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= MN4) return;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int z = 0; z < splits; ++z) {
    const float4 v = partials[(long long)z * MN4 + i];
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  if (bias) { const float4 b = bias[i % N4]; s.x += b.x; s.y += b.y; s.z += b.z; s.w += b.w; }
  if (act == ACT_RELU) { s.x = fmaxf(s.x, 0.f); s.y = fmaxf(s.y, 0.f); s.z = fmaxf(s.z, 0.f); s.w = fmaxf(s.w, 0.f); }
  else if (act == ACT_SIGMOID) { s.x = 1.f / (1.f + expf(-s.x)); s.y = 1.f / (1.f + expf(-s.y)); s.z = 1.f / (1.f + expf(-s.z)); s.w = 1.f / (1.f + expf(-s.w)); }
  out[i] = s;
}

template <int MODE>
int launch_mode(const IGemmParams& p, dim3 grid, cudaStream_t stream, bool vec) {
  if (p.src_u8) {
    if (MODE == GATHER_DGRAD) { set_error("igemm: u8 source unsupported for dgrad"); return AAE_ERR_UNSUPPORTED; }
    igemm_f32_kernel<MODE, false, true><<<grid, NT, 0, stream>>>(p);
  } else if (vec) {
    igemm_f32_kernel<MODE, true, false><<<grid, NT, 0, stream>>>(p);
  } else {
    igemm_f32_kernel<MODE, false, false><<<grid, NT, 0, stream>>>(p);
  }
  AAE_LAUNCH_OK();
  return AAE_OK;
}

}  // namespace

int launch_igemm(const IGemmParams& p, int mode, cudaStream_t stream) {
  AAE_REQUIRE(p.N % 4 == 0, "igemm: N=%d must be a multiple of 4", p.N);
  AAE_REQUIRE(p.k_per_split > 0 && p.k_per_split % BK == 0, "igemm: k_per_split=%d must be a positive multiple of %d", p.k_per_split, BK);
  AAE_REQUIRE(p.M > 0 && p.K > 0, "igemm: empty problem M=%d K=%d", p.M, p.K);
  const int splits = (int)ceil_div(p.K, p.k_per_split);
  dim3 grid((unsigned)ceil_div(p.M, BM), (unsigned)ceil_div(p.N, BN), (unsigned)splits);
  bool vec;
  if (mode == GATHER_WGRAD) vec = (p.SC % BM == 0) && !p.src_u8;
  else vec = (p.SC % BK == 0) && !p.src_u8;
  if (p.parity_major) {
    AAE_REQUIRE(mode == GATHER_DGRAD && p.stride == 2 && (p.PH % 2 == 0) && (p.PW % 2 == 0) && ((p.M / 4) % BM == 0) && vec,
                "igemm: parity-major ordering needs stride 2, even dims, (M/4)%%128==0 and SC%%16==0");
  }
  switch (mode) {
    case GATHER_FWD: return launch_mode<GATHER_FWD>(p, grid, stream, vec);
    case GATHER_DGRAD: return launch_mode<GATHER_DGRAD>(p, grid, stream, vec);
    case GATHER_WGRAD: return launch_mode<GATHER_WGRAD>(p, grid, stream, vec);
  }
  set_error("igemm: bad mode %d", mode);
  return AAE_ERR_INVALID_ARG;
}

int launch_splitk_reduce(const float* partials, int splits, int64_t MN, int N, const float* bias, int act, float* out,
                         cudaStream_t stream) {
  const int threads = 256;
  // This small kernel sits between kernels that use ~200 KB of shared memory per CTA (the dense GEMM before it, the fused match
  // after it).  Asking for the same carveout avoids an L1/shared-memory reconfiguration of every SM on both sides.
  static const bool hinted = [] {
    cudaFuncSetAttribute(splitk_reduce_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    cudaFuncSetAttribute(splitk_reduce4_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    return true;
  }();
  (void)hinted;
  const bool aligned = ((uintptr_t)partials % 16 == 0) && ((uintptr_t)out % 16 == 0) && (!bias || (uintptr_t)bias % 16 == 0);
  if (MN % 4 == 0 && N % 4 == 0 && aligned && MN >= (1 << 20))   // small outputs: keep one thread per element for parallelism
    splitk_reduce4_kernel<<<(unsigned)ceil_div(MN / 4, threads), threads, 0, stream>>>(reinterpret_cast<const float4*>(partials), splits, MN / 4, N / 4,
                                                                                     reinterpret_cast<const float4*>(bias), act,
                                                                                     reinterpret_cast<float4*>(out));
  else
    splitk_reduce_kernel<<<(unsigned)ceil_div(MN, threads), threads, 0, stream>>>(partials, splits, MN, N, bias, act, out);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

}  // namespace aae
