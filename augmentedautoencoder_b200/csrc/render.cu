// Batched rasteriser of the reference's phong renderer (auto_pose/meshrenderer/meshrenderer_phong.py with
// shader/depth_shader_phong.{vs,frag}, MODEL: reconst, ANTIALIASING: 1).  DESIGN.md "Renderer" states the contract and the
// operation order below, which the test suite's numpy restatement follows bit for bit.
//
// Per chunk of views:
//   1. vertex pass   view/projection transform of every vertex, 8-bit sub-pixel snap, window depth, w; per-view screen box of the
//                    vertices and the behind-the-camera flag (camera z <= near);
//   2. clear         the visibility buffer of each view, bounded by that screen box;
//   3. raster        one thread per (triangle, view), int64 edge functions, top-left fill rule, pixel centres; triangles whose
//                    box covers more than kLargeTri pixels are rasterised by their whole warp.  Every covered pixel does one
//                    64-bit atomicMin of (float bits of window depth << 32 | triangle index): GL_LESS with submission-order ties;
//   4. shade         per pixel (full frame) or per pixel the INTER_NEAREST crop samples (fused path): the winning triangle's three
//                    vertices are transformed again, their varyings interpolated perspective-correctly and the phong fragment
//                    evaluated.
// Every float step is an explicit IEEE-rounded fp32 operation (__fmul_rn, __fadd_rn, __fdiv_rn, __fsqrt_rn): no contraction.
#include <climits>
#include <vector>

#include "common.cuh"

namespace aae {
namespace {

constexpr int kSub = 256;                 // 8 sub-pixel bits
constexpr int kLargeTri = 64;             // bbox pixels above which the warp rasterises the triangle together
constexpr float kSnapLimit = 536870912.f; // |window coordinate| * 256 is clamped to 2^29 so that edge functions fit int64
constexpr unsigned long long kEmptyKey = (0x3f800000ull << 32) | 0xffffffffull;   // depth 1.0 (the clear value), no triangle

struct Mesh {
  int device;
  int64_t nv, nf;
  float* verts;   // [nv, 9]: position * vertex_scale, normal, colour / 255
  int* faces;     // [nf, 3]
};

__device__ __forceinline__ float fm(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fa(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fs(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fd(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float dot3(float ax, float ay, float az, float bx, float by, float bz) {
  return fa(fa(fm(ax, bx), fm(ay, by)), fm(az, bz));
}
// row r of a row-major 4x4 matrix times (x, y, z, w)
__device__ __forceinline__ float row4(const float* M, int r, float x, float y, float z, float w) {
  const float* m = M + 4 * r;
  return fa(fa(fa(fm(m[0], x), fm(m[1], y)), fm(m[2], z)), fm(m[3], w));
}

struct VertexOut { int X, Y; float zw, cw; };

// P = view . (pos, 1); clip = projection . P; window = ((ndc_x + 1) W/2, (1 - ndc_y) H/2) in image rows (top = 0), depth (ndc_z + 1)/2
__device__ __forceinline__ VertexOut project(const float* view, const float* proj, const float* pos, float halfW, float halfH,
                                             float* camera_z) {
  const float px = row4(view, 0, pos[0], pos[1], pos[2], 1.f), py = row4(view, 1, pos[0], pos[1], pos[2], 1.f);
  const float pz = row4(view, 2, pos[0], pos[1], pos[2], 1.f), pw = row4(view, 3, pos[0], pos[1], pos[2], 1.f);
  const float cx = row4(proj, 0, px, py, pz, pw), cy = row4(proj, 1, px, py, pz, pw);
  const float cz = row4(proj, 2, px, py, pz, pw), cw = row4(proj, 3, px, py, pz, pw);
  *camera_z = -pz;
  const float sx = fm(fa(fd(cx, cw), 1.f), halfW);
  const float sy = fm(fs(1.f, fd(cy, cw)), halfH);
  VertexOut o;
  o.X = __float2int_rn(fminf(fmaxf(fm(sx, (float)kSub), -kSnapLimit), kSnapLimit));
  o.Y = __float2int_rn(fminf(fmaxf(fm(sy, (float)kSub), -kSnapLimit), kSnapLimit));
  o.zw = fm(fa(fd(cz, cw), 1.f), 0.5f);
  o.cw = cw;
  return o;
}

// first / last pixel whose centre (p * 256 + 128) lies in [lo, hi] (fixed point)
__device__ __forceinline__ int first_px(int lo) { return -((128 - lo) >> 8); }
__device__ __forceinline__ int last_px(int hi) { return (hi - 128) >> 8; }

struct Box { int x0, y0, x1, y1; };   // inclusive pixel box, empty when x0 > x1 or y0 > y1

__device__ __forceinline__ Box view_box(const int4 b, int W, int H) {
  Box r;
  r.x0 = max(first_px(b.x), 0); r.y0 = max(first_px(b.y), 0);
  r.x1 = min(last_px(b.z), W - 1); r.y1 = min(last_px(b.w), H - 1);
  return r;
}

__device__ __forceinline__ long long orient(long long ax, long long ay, long long bx, long long by, long long cx, long long cy) {
  return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax);
}
// top-left rule in image coordinates (y down) for a triangle with positive orientation
__device__ __forceinline__ long long edge_bias(long long ax, long long ay, long long bx, long long by) {
  const long long dx = bx - ax, dy = by - ay;
  return (dy < 0 || (dy == 0 && dx > 0)) ? 0 : -1;
}

// A triangle in one view, vertices ordered so that its orientation A is positive (v1 and v2 swapped otherwise).
struct Tri {
  int idx[3];
  long long X[3], Y[3];
  float zw[3], cw[3];
  long long A;
};

__device__ __forceinline__ bool setup_tri(const int* faces, const int4* vb, int t, Tri& T) {
  const int f0 = faces[3 * t], f1 = faces[3 * t + 1], f2 = faces[3 * t + 2];
  int id[3] = {f0, f1, f2};
  int4 v[3] = {vb[f0], vb[f1], vb[f2]};
  long long A = orient(v[0].x, v[0].y, v[1].x, v[1].y, v[2].x, v[2].y);
  if (A == 0) return false;
  if (A < 0) {
    int4 tv = v[1]; v[1] = v[2]; v[2] = tv;
    int ti = id[1]; id[1] = id[2]; id[2] = ti;
    A = -A;
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    T.idx[k] = id[k]; T.X[k] = v[k].x; T.Y[k] = v[k].y;
    T.zw[k] = __int_as_float(v[k].z); T.cw[k] = __int_as_float(v[k].w);
  }
  T.A = A;
  return true;
}

// raw edge functions at the centre of pixel (px, py): w0 opposite v0 (edge v1 -> v2), w1 (v2 -> v0), w2 (v0 -> v1)
__device__ __forceinline__ void edges(const Tri& T, int px, int py, long long w[3]) {
  const long long cx = (long long)px * kSub + kSub / 2, cy = (long long)py * kSub + kSub / 2;
  w[0] = orient(T.X[1], T.Y[1], T.X[2], T.Y[2], cx, cy);
  w[1] = orient(T.X[2], T.Y[2], T.X[0], T.Y[0], cx, cy);
  w[2] = orient(T.X[0], T.Y[0], T.X[1], T.Y[1], cx, cy);
}

__device__ __forceinline__ void cover_pixel(const Tri& T, unsigned tri, const long long bias[3], int px, int py, const Box& vbox,
                                            unsigned long long* vis) {
  long long w[3];
  edges(T, px, py, w);
  if (w[0] + bias[0] < 0 || w[1] + bias[1] < 0 || w[2] + bias[2] < 0) return;
  const float fA = __ll2float_rn(T.A);
  const float l0 = fd(__ll2float_rn(w[0]), fA), l1 = fd(__ll2float_rn(w[1]), fA), l2 = fd(__ll2float_rn(w[2]), fA);
  const float z = fa(fa(fm(l0, T.zw[0]), fm(l1, T.zw[1])), fm(l2, T.zw[2]));
  if (!(z >= 0.f && z < 1.f)) return;   // outside [near, far], or not less than the cleared depth 1.0
  const unsigned long long key = ((unsigned long long)__float_as_uint(z) << 32) | tri;
  atomicMin(vis + (long long)(py - vbox.y0) * (vbox.x1 - vbox.x0 + 1) + (px - vbox.x0), key);
}

struct Params {
  const float* views;      // [n, AAE_RENDER_VIEW_FLOATS]
  int n, W, H;
  float near_;
  int64_t cap;             // visibility entries per view (W * H)
  unsigned long long* vis; // [n, cap]
  int4* vbuf;              // [n, nv]: X, Y, bits(zw), bits(cw)
  int4* vbox;              // [n]: min X, min Y, max X, max Y (fixed point)
  int4* cov;               // [n]: covered pixels min x, min y, max x, max y
  int* flags;              // [n]
};

__global__ void init_kernel(Params p) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= p.n) return;
  p.vbox[v] = make_int4(INT_MAX, INT_MAX, INT_MIN, INT_MIN);
  p.cov[v] = make_int4(INT_MAX, INT_MAX, INT_MIN, INT_MIN);
  p.flags[v] = 0;
}

__global__ void vertex_kernel(Params p, const float* __restrict__ verts, int nv) {
  const int v = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const float* vp = p.views + (long long)v * AAE_RENDER_VIEW_FLOATS;
  int4 mn = make_int4(INT_MAX, INT_MAX, INT_MIN, INT_MIN);
  bool behind = false;
  if (i < nv) {
    float camz;
    const VertexOut o = project(vp, vp + 16, verts + (long long)i * 9, 0.5f * (float)p.W, 0.5f * (float)p.H, &camz);
    behind = !(camz > p.near_);
    p.vbuf[(long long)v * nv + i] = make_int4(o.X, o.Y, __float_as_int(o.zw), __float_as_int(o.cw));
    mn = make_int4(o.X, o.Y, o.X, o.Y);
  }
  const unsigned all = 0xffffffffu;
  const int x0 = __reduce_min_sync(all, mn.x), y0 = __reduce_min_sync(all, mn.y);
  const int x1 = __reduce_max_sync(all, mn.z), y1 = __reduce_max_sync(all, mn.w);
  const bool any_behind = __any_sync(all, behind);
  if ((threadIdx.x & 31) == 0) {
    atomicMin(&p.vbox[v].x, x0); atomicMin(&p.vbox[v].y, y0);
    atomicMax(&p.vbox[v].z, x1); atomicMax(&p.vbox[v].w, y1);
    if (any_behind) atomicOr(&p.flags[v], AAE_RENDER_BEHIND_CAMERA);
  }
}

__global__ void clear_kernel(Params p) {
  const int v = blockIdx.y;
  const Box b = view_box(p.vbox[v], p.W, p.H);
  if (b.x0 > b.x1 || b.y0 > b.y1) return;
  const long long area = (long long)(b.x1 - b.x0 + 1) * (b.y1 - b.y0 + 1);
  unsigned long long* vis = p.vis + (long long)v * p.cap;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < area; k += (long long)gridDim.x * blockDim.x) vis[k] = kEmptyKey;
}

__global__ void raster_kernel(Params p, const int* __restrict__ faces, int nf, int nv) {
  const int v = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const Box vb = view_box(p.vbox[v], p.W, p.H);
  const bool view_ok = !(p.flags[v] & AAE_RENDER_BEHIND_CAMERA) && vb.x0 <= vb.x1 && vb.y0 <= vb.y1;
  unsigned long long* vis = p.vis + (long long)v * p.cap;
  Tri T;
  Box b = {0, 0, -1, -1};
  bool active = view_ok && t < nf && setup_tri(faces, p.vbuf + (long long)v * nv, t, T);
  long long bias[3] = {0, 0, 0};
  if (active) {
    b.x0 = max(first_px((int)min(min(T.X[0], T.X[1]), T.X[2])), vb.x0);
    b.y0 = max(first_px((int)min(min(T.Y[0], T.Y[1]), T.Y[2])), vb.y0);
    b.x1 = min(last_px((int)max(max(T.X[0], T.X[1]), T.X[2])), vb.x1);
    b.y1 = min(last_px((int)max(max(T.Y[0], T.Y[1]), T.Y[2])), vb.y1);
    active = b.x0 <= b.x1 && b.y0 <= b.y1;
    bias[0] = edge_bias(T.X[1], T.Y[1], T.X[2], T.Y[2]);
    bias[1] = edge_bias(T.X[2], T.Y[2], T.X[0], T.Y[0]);
    bias[2] = edge_bias(T.X[0], T.Y[0], T.X[1], T.Y[1]);
  }
  const long long area = active ? (long long)(b.x1 - b.x0 + 1) * (b.y1 - b.y0 + 1) : 0;
  if (active && area <= kLargeTri) {
    for (int py = b.y0; py <= b.y1; ++py)
      for (int px = b.x0; px <= b.x1; ++px) cover_pixel(T, (unsigned)t, bias, px, py, vb, vis);
  }
  // cooperative path: the warp walks each large triangle of its lanes together, one pixel per lane
  unsigned large = __ballot_sync(0xffffffffu, active && area > kLargeTri);
  const int lane = threadIdx.x & 31;
  while (large) {
    const int src = __ffs(large) - 1;
    large &= large - 1;
    Tri S;
    long long sb[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      S.idx[k] = __shfl_sync(0xffffffffu, T.idx[k], src);
      S.X[k] = __shfl_sync(0xffffffffu, T.X[k], src);
      S.Y[k] = __shfl_sync(0xffffffffu, T.Y[k], src);
      S.zw[k] = __shfl_sync(0xffffffffu, T.zw[k], src);
      S.cw[k] = __shfl_sync(0xffffffffu, T.cw[k], src);
      sb[k] = __shfl_sync(0xffffffffu, bias[k], src);
    }
    S.A = __shfl_sync(0xffffffffu, T.A, src);
    const int st = __shfl_sync(0xffffffffu, t, src);
    const int bx0 = __shfl_sync(0xffffffffu, b.x0, src), by0 = __shfl_sync(0xffffffffu, b.y0, src);
    const int bw = __shfl_sync(0xffffffffu, b.x1, src) - bx0 + 1;
    const long long sarea = __shfl_sync(0xffffffffu, area, src);
    for (long long k = lane; k < sarea; k += 32) {
      const int py = by0 + (int)(k / bw), px = bx0 + (int)(k % bw);
      cover_pixel(S, (unsigned)st, sb, px, py, vb, vis);
    }
  }
}

// light: (x, y, z, ambient, diffuse, specular)
struct Light { float lx, ly, lz, a, d, s; };

__device__ __forceinline__ Light light_of(const float* vp, int which) {
  const float* l = vp + 48 + 6 * which;
  Light L = {l[0], l[1], l[2], l[3], l[4], l[5]};
  return L;
}

__device__ __forceinline__ void normalize3(float& x, float& y, float& z) {
  const float n = __fsqrt_rn(dot3(x, y, z, x, y, z));
  x = fd(x, n); y = fd(y, n); z = fd(z, n);
}

// The fragment at pixel (px, py) of triangle t: bgr bytes and the camera-space depth.
__device__ void shade(const float* vp, const Light& Lt, const float* __restrict__ verts, const int* __restrict__ faces,
                      const int4* vb, unsigned t, int px, int py, uint8_t bgr[3], float* depth) {
  Tri T;
  setup_tri(faces, vb, (int)t, T);
  long long w[3];
  edges(T, px, py, w);
  const float fA = __ll2float_rn(T.A);
  float q[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) q[k] = fd(fd(__ll2float_rn(w[k]), fA), T.cw[k]);
  const float s = fa(fa(q[0], q[1]), q[2]);
  float r[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) r[k] = fd(q[k], s);
  // varyings of the vertex shader: v_view = -P.xyz, v_L = normalize(light - P.xyz), v_normal = normalize(nm . (n, 1)).xyz, v_color
  const float* view = vp;
  const float* nm = vp + 32;
  float acc[12];
#pragma unroll
  for (int j = 0; j < 12; ++j) acc[j] = 0.f;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float* a = verts + (long long)T.idx[k] * 9;
    const float px_ = row4(view, 0, a[0], a[1], a[2], 1.f), py_ = row4(view, 1, a[0], a[1], a[2], 1.f);
    const float pz_ = row4(view, 2, a[0], a[1], a[2], 1.f);
    float att[12];
    att[0] = -px_; att[1] = -py_; att[2] = -pz_;
    float lx = fs(Lt.lx, px_), ly = fs(Lt.ly, py_), lz = fs(Lt.lz, pz_);
    normalize3(lx, ly, lz);
    att[3] = lx; att[4] = ly; att[5] = lz;
    const float nx = row4(nm, 0, a[3], a[4], a[5], 1.f), ny = row4(nm, 1, a[3], a[4], a[5], 1.f);
    const float nz = row4(nm, 2, a[3], a[4], a[5], 1.f), nw = row4(nm, 3, a[3], a[4], a[5], 1.f);
    const float n4 = __fsqrt_rn(fa(dot3(nx, ny, nz, nx, ny, nz), fm(nw, nw)));
    att[6] = fd(nx, n4); att[7] = fd(ny, n4); att[8] = fd(nz, n4);
    att[9] = a[6]; att[10] = a[7]; att[11] = a[8];
#pragma unroll
    for (int j = 0; j < 12; ++j) acc[j] = k == 0 ? fm(r[0], att[j]) : fa(acc[j], fm(r[k], att[j]));
  }
  *depth = acc[2];
  float Vx = acc[0], Vy = acc[1], Vz = acc[2];
  float Lx = acc[3], Ly = acc[4], Lz = acc[5];
  float Nx = acc[6], Ny = acc[7], Nz = acc[8];
  normalize3(Nx, Ny, Nz);
  normalize3(Lx, Ly, Lz);
  normalize3(Vx, Vy, Vz);
  const float ndl = dot3(Nx, Ny, Nz, Lx, Ly, Lz);
  const float diff = fmaxf(ndl, 0.f);
  // reflect(-L, N) = -L - 2 dot(N, -L) N
  const float dni = dot3(Nx, Ny, Nz, -Lx, -Ly, -Lz);
  const float two_d = fm(2.f, dni);
  const float Rx = fs(-Lx, fm(two_d, Nx)), Ry = fs(-Ly, fm(two_d, Ny)), Rz = fs(-Lz, fm(two_d, Nz));
  const float spec = fmaxf(dot3(Rx, Ry, Rz, Vx, Vy, Vz), 0.f);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float col = acc[9 + c];
    float v = fa(fa(fm(Lt.a, col), fm(Lt.d, fm(diff, col))), fm(Lt.s, fm(spec, col)));
    v = fminf(v, 1.f);
    bgr[2 - c] = (uint8_t)__float2int_rn(fm(v, 255.f));
  }
}

__device__ __forceinline__ unsigned long long read_key(const Params& p, int v, const Box& vb, int px, int py) {
  if (px < vb.x0 || px > vb.x1 || py < vb.y0 || py > vb.y1) return kEmptyKey;
  return p.vis[(long long)v * p.cap + (long long)(py - vb.y0) * (vb.x1 - vb.x0 + 1) + (px - vb.x0)];
}

__device__ __forceinline__ void reduce_cov(int4* cov, bool hit, int px, int py) {
  const unsigned all = 0xffffffffu;
  const int x0 = __reduce_min_sync(all, hit ? px : INT_MAX), y0 = __reduce_min_sync(all, hit ? py : INT_MAX);
  const int x1 = __reduce_max_sync(all, hit ? px : INT_MIN), y1 = __reduce_max_sync(all, hit ? py : INT_MIN);
  if ((threadIdx.x & 31) == 0 && x1 != INT_MIN) {
    atomicMin(&cov->x, x0); atomicMin(&cov->y, y0);
    atomicMax(&cov->z, x1); atomicMax(&cov->w, y1);
  }
}

// full frames: bgr / depth for every pixel, and the covered-pixel box
__global__ void resolve_frame_kernel(Params p, const float* __restrict__ verts, const int* __restrict__ faces, int nv, uint8_t* bgr,
                                     float* depth) {
  const int v = blockIdx.y;
  const long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long npix = (long long)p.W * p.H;
  const int py = (int)(pix / p.W), px = (int)(pix - (long long)py * p.W);
  const Box vb = view_box(p.vbox[v], p.W, p.H);
  const float* vp = p.views + (long long)v * AAE_RENDER_VIEW_FLOATS;
  bool hit = false;
  if (pix < npix) {
    const unsigned long long key = (p.flags[v] & AAE_RENDER_BEHIND_CAMERA) ? kEmptyKey : read_key(p, v, vb, px, py);
    uint8_t c[3] = {0, 0, 0};
    float d = 0.f;
    const unsigned t = (unsigned)(key & 0xffffffffu);
    if (t != 0xffffffffu) {
      shade(vp, light_of(vp, 0), verts, faces, p.vbuf + (long long)v * nv, t, px, py, c, &d);
      hit = true;
    }
    uint8_t* o = bgr + ((long long)v * npix + pix) * 3;
    o[0] = c[0]; o[1] = c[1]; o[2] = c[2];
    depth[(long long)v * npix + pix] = d;
  }
  reduce_cov(p.cov + v, hit, px, py);
}

// covered-pixel box without materialising the frame (fused path)
__global__ void coverage_kernel(Params p) {
  const int v = blockIdx.y;
  const Box vb = view_box(p.vbox[v], p.W, p.H);
  if (vb.x0 > vb.x1 || vb.y0 > vb.y1 || (p.flags[v] & AAE_RENDER_BEHIND_CAMERA)) return;
  const int bw = vb.x1 - vb.x0 + 1;
  const long long area = (long long)bw * (vb.y1 - vb.y0 + 1);
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long start = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  // every lane of a warp runs the same number of iterations so that the warp reductions see all 32 lanes
  const long long iters = (area + stride - 1) / stride;
  for (long long it = 0; it < iters; ++it) {
    const long long k = start + it * stride;
    bool hit = false;
    int px = 0, py = 0;
    if (k < area) {
      py = vb.y0 + (int)(k / bw); px = vb.x0 + (int)(k % bw);
      hit = (unsigned)(p.vis[(long long)v * p.cap + k] & 0xffffffffu) != 0xffffffffu;
    }
    reduce_cov(p.cov + v, hit, px, py);
  }
}

// calc_2d_bbox of the covered pixels: +-1 pixel, clamped to (W - 1, H - 1)  (pysixd_stuff/view_sampler.py:10-15)
__device__ __forceinline__ bool obj_bb_of(const int4 c, int W, int H, int bb[4]) {
  if (c.z == INT_MIN) return false;
  const int x0 = max(c.x - 1, 0), y0 = max(c.y - 1, 0), x1 = min(c.z + 1, W - 1), y1 = min(c.w + 1, H - 1);
  bb[0] = x0; bb[1] = y0; bb[2] = x1 - x0; bb[3] = y1 - y0;
  return true;
}

__global__ void finalize_bb_kernel(Params p, int* obj_bb) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= p.n) return;
  int bb[4] = {0, 0, 0, 0};
  if (!obj_bb_of(p.cov[v], p.W, p.H, bb)) p.flags[v] |= AAE_RENDER_EMPTY;
  for (int k = 0; k < 4; ++k) obj_bb[4 * v + k] = bb[k];
}

struct Window { int left, top, cw, ch; bool ok; };

// Dataset.extract_square_patch (auto_pose/ae/dataset.py:354-373) in float64: the box is truncated to int32, the square side is
// int(max(h, w) * pad_factor), the window is clipped to the frame
__device__ __forceinline__ Window crop_window(double bx, double by, double bw, double bh, double pad, int W, int H) {
  const int x = (int)bx, y = (int)by, w = (int)bw, h = (int)bh;
  const int size = (int)__dmul_rn((double)max(h, w), pad);
  const double cx = __dadd_rn((double)x, (double)w / 2.0), cy = __dadd_rn((double)y, (double)h / 2.0), hs = (double)size / 2.0;
  const int left = (int)fmax(__dsub_rn(cx, hs), 0.0), right = (int)fmin(__dadd_rn(cx, hs), (double)W);
  const int top = (int)fmax(__dsub_rn(cy, hs), 0.0), bottom = (int)fmin(__dadd_rn(cy, hs), (double)H);
  Window r;
  r.left = left; r.top = top; r.cw = right - left; r.ch = bottom - top;
  r.ok = right >= 0 && bottom >= 0 && r.cw > 0 && r.ch > 0;
  return r;
}

// fused crops: x (light 0, box shifted by offset * (w, h)), optional mask of x, optional y (light 1, unshifted box)
__global__ void crop_kernel(Params p, const float* __restrict__ verts, const int* __restrict__ faces, int nv, const double* offsets,
                            double pad, int oh, int ow, const int* __restrict__ col_map, const int* __restrict__ row_map,
                            uint8_t* crop_x, uint8_t* mask_x, uint8_t* crop_y, int* obj_bb) {
  const int v = blockIdx.y;
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  int bb[4] = {0, 0, 0, 0};
  const bool visible = !(p.flags[v] & AAE_RENDER_BEHIND_CAMERA) && obj_bb_of(p.cov[v], p.W, p.H, bb);
  double ox = 0.0, oy = 0.0;
  if (offsets) {   // np.random.uniform(-m, m) * w, then obj_bb + [dx, dy, 0, 0]
    ox = __dmul_rn(offsets[2 * v], (double)bb[2]);
    oy = __dmul_rn(offsets[2 * v + 1], (double)bb[3]);
  }
  const Window wx = crop_window(__dadd_rn((double)bb[0], ox), __dadd_rn((double)bb[1], oy), (double)bb[2], (double)bb[3], pad, p.W, p.H);
  const Window wy = crop_window((double)bb[0], (double)bb[1], (double)bb[2], (double)bb[3], pad, p.W, p.H);
  if (pix == 0) {
    int f = 0;
    if (!visible) f |= AAE_RENDER_EMPTY;
    else if (!wx.ok || (crop_y && !wy.ok)) f |= AAE_RENDER_BAD_CROP;
    if (f) atomicOr(&p.flags[v], f);
    for (int k = 0; k < 4; ++k) obj_bb[4 * v + k] = bb[k];
  }
  if (pix >= oh * ow) return;
  const int dy = pix / ow, dx = pix - dy * ow;
  const long long o = (long long)v * oh * ow + pix;
  const Box vb = view_box(p.vbox[v], p.W, p.H);
  const float* vp = p.views + (long long)v * AAE_RENDER_VIEW_FLOATS;
  const int4* vbv = p.vbuf + (long long)v * nv;
  {
    uint8_t c[3] = {0, 0, 0};
    bool empty = true;
    if (visible && wx.ok) {
      const int sx = wx.left + col_map[(long long)wx.cw * ow + dx], sy = wx.top + row_map[(long long)wx.ch * oh + dy];
      const unsigned t = (unsigned)(read_key(p, v, vb, sx, sy) & 0xffffffffu);
      if (t != 0xffffffffu) {
        float d;
        shade(vp, light_of(vp, 0), verts, faces, vbv, t, sx, sy, c, &d);
        empty = false;
      }
    }
    crop_x[3 * o] = c[0]; crop_x[3 * o + 1] = c[1]; crop_x[3 * o + 2] = c[2];
    if (mask_x) mask_x[o] = empty ? 1 : 0;
  }
  if (crop_y) {
    uint8_t c[3] = {0, 0, 0};
    if (visible && wy.ok) {
      const int sx = wy.left + col_map[(long long)wy.cw * ow + dx], sy = wy.top + row_map[(long long)wy.ch * oh + dy];
      const unsigned t = (unsigned)(read_key(p, v, vb, sx, sy) & 0xffffffffu);
      if (t != 0xffffffffu) {
        float d;
        shade(vp, light_of(vp, 1), verts, faces, vbv, t, sx, sy, c, &d);
      }
    }
    crop_y[3 * o] = c[0]; crop_y[3 * o + 1] = c[1]; crop_y[3 * o + 2] = c[2];
  }
}

// Workspace sections, each starting on a 256-byte boundary (the int4 sections must not follow an odd count of 8-byte keys
// unaligned): visibility keys [n, W*H] u64, vertex buffer [n, nv] int4, vertex boxes [n] int4, covered boxes [n] int4.
constexpr int64_t kWsAlign = 256;
inline int64_t ws_round(int64_t b) { return (b + kWsAlign - 1) / kWsAlign * kWsAlign; }

int64_t workspace_bytes(const Mesh* m, int n, int W, int H) {
  return ws_round((int64_t)n * W * H * 8) + ws_round((int64_t)n * m->nv * 16) + 2 * ws_round((int64_t)n * 16);
}

int rasterise(const Mesh* m, Params& p, void* ws, int64_t ws_bytes, cudaStream_t s) {
  AAE_REQUIRE(ws && ws_bytes >= workspace_bytes(m, p.n, p.W, p.H), "render workspace too small (%lld bytes, need %lld)",
              (long long)ws_bytes, (long long)workspace_bytes(m, p.n, p.W, p.H));
  AAE_REQUIRE((uintptr_t)ws % kWsAlign == 0, "render workspace must be %d-byte aligned", (int)kWsAlign);
  p.cap = (int64_t)p.W * p.H;
  char* w = (char*)ws;
  p.vis = (unsigned long long*)w; w += ws_round((int64_t)p.n * p.cap * 8);
  p.vbuf = (int4*)w; w += ws_round((int64_t)p.n * m->nv * 16);
  p.vbox = (int4*)w; w += ws_round((int64_t)p.n * 16);
  p.cov = (int4*)w;
  init_kernel<<<(unsigned)ceil_div(p.n, 128), 128, 0, s>>>(p);
  AAE_LAUNCH_OK();
  vertex_kernel<<<dim3((unsigned)ceil_div(m->nv, 256), p.n), 256, 0, s>>>(p, m->verts, (int)m->nv);
  AAE_LAUNCH_OK();
  clear_kernel<<<dim3(64, p.n), 256, 0, s>>>(p);
  AAE_LAUNCH_OK();
  raster_kernel<<<dim3((unsigned)ceil_div(m->nf, 128), p.n), 128, 0, s>>>(p, m->faces, (int)m->nf, (int)m->nv);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

int check_call(const Mesh* m, const float* views, int n, int W, int H, float near_, float far_) {
  AAE_REQUIRE(m && views, "null argument");
  AAE_REQUIRE(n >= 1 && n <= 65535, "n_views must be in [1, 65535]");
  AAE_REQUIRE(W >= 1 && H >= 1 && W <= 2000 && H <= 2000, "frame size must be in [1, 2000]");
  AAE_REQUIRE(near_ > 0.f && far_ > near_, "need 0 < near < far");
  return AAE_OK;
}

}  // namespace
}  // namespace aae

using namespace aae;

extern "C" int aae_mesh_create(int device, const float* vertices, int64_t n_vertices, const int32_t* faces, int64_t n_faces,
                               aae_mesh** out) {
  AAE_REQUIRE(out && vertices && faces, "null argument");
  *out = nullptr;
  AAE_REQUIRE(n_vertices >= 1 && n_vertices < (1ll << 31) && n_faces >= 1 && n_faces < (1ll << 31) - 1, "bad mesh sizes");
  for (int64_t k = 0; k < 3 * n_faces; ++k)
    AAE_REQUIRE(faces[k] >= 0 && faces[k] < n_vertices, "face %lld refers to vertex %d of %lld", (long long)(k / 3), (int)faces[k],
                (long long)n_vertices);
  int count = 0;
  AAE_REQUIRE(cudaGetDeviceCount(&count) == cudaSuccess && device >= 0 && device < count, "no CUDA device %d", device);
  DeviceGuard g(device);
  AAE_REQUIRE(g.ok, "cannot select device %d", device);
  Mesh* m = new Mesh();
  m->device = device; m->nv = n_vertices; m->nf = n_faces;
  m->verts = nullptr; m->faces = nullptr;
  cudaError_t e = cudaMalloc(&m->verts, n_vertices * 9 * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&m->faces, n_faces * 3 * sizeof(int));
  if (e == cudaSuccess) e = cudaMemcpy(m->verts, vertices, n_vertices * 9 * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(m->faces, faces, n_faces * 3 * sizeof(int), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    cudaFree(m->verts); cudaFree(m->faces);
    delete m;
    set_error("mesh upload: %s", cudaGetErrorString(e));
    return AAE_ERR_CUDA;
  }
  *out = (aae_mesh*)m;
  return AAE_OK;
}

extern "C" int aae_mesh_destroy(aae_mesh* h) {
  if (!h) return AAE_OK;
  Mesh* m = (Mesh*)h;
  DeviceGuard g(m->device);
  cudaFree(m->verts);
  cudaFree(m->faces);
  delete m;
  return AAE_OK;
}

extern "C" int64_t aae_render_workspace_bytes(const aae_mesh* h, int n_views, int W, int H) {
  if (!h || n_views < 1 || W < 1 || H < 1) return -1;
  return workspace_bytes((const Mesh*)h, n_views, W, H);
}

extern "C" int aae_render_frames(const aae_mesh* h, const float* views_dev, int n_views, int W, int H, float near_, float far_,
                                 void* workspace_dev, int64_t workspace_bytes_, uint8_t* bgr_dev, float* depth_dev, int32_t* obj_bb_dev,
                                 int32_t* flags_dev, void* stream) {
  const Mesh* m = (const Mesh*)h;
  AAE_TRY(check_call(m, views_dev, n_views, W, H, near_, far_));
  AAE_REQUIRE(bgr_dev && depth_dev && obj_bb_dev && flags_dev, "null output");
  DeviceGuard g(m->device);
  cudaStream_t s = (cudaStream_t)stream;
  Params p;
  p.views = views_dev; p.n = n_views; p.W = W; p.H = H; p.near_ = near_; p.flags = flags_dev;
  AAE_TRY(rasterise(m, p, workspace_dev, workspace_bytes_, s));
  resolve_frame_kernel<<<dim3((unsigned)ceil_div((int64_t)W * H, 256), n_views), 256, 0, s>>>(p, m->verts, m->faces, (int)m->nv,
                                                                                              bgr_dev, depth_dev);
  AAE_LAUNCH_OK();
  finalize_bb_kernel<<<(unsigned)ceil_div(n_views, 128), 128, 0, s>>>(p, obj_bb_dev);
  AAE_LAUNCH_OK();
  return AAE_OK;
}

extern "C" int aae_render_crops(const aae_mesh* h, const float* views_dev, int n_views, int W, int H, float near_, float far_,
                                const double* offsets_dev, double pad_factor, int out_h, int out_w, const int32_t* col_map_dev,
                                const int32_t* row_map_dev, void* workspace_dev, int64_t workspace_bytes_, uint8_t* crop_x_dev,
                                uint8_t* mask_x_dev, uint8_t* crop_y_dev, int32_t* obj_bb_dev, int32_t* flags_dev, void* stream) {
  const Mesh* m = (const Mesh*)h;
  AAE_TRY(check_call(m, views_dev, n_views, W, H, near_, far_));
  AAE_REQUIRE(crop_x_dev && obj_bb_dev && flags_dev && col_map_dev && row_map_dev, "null argument");
  AAE_REQUIRE(out_h >= 1 && out_w >= 1 && out_h <= 1024 && out_w <= 1024, "crop size must be in [1, 1024]");
  AAE_REQUIRE(pad_factor > 0.0, "pad_factor must be positive");
  DeviceGuard g(m->device);
  cudaStream_t s = (cudaStream_t)stream;
  Params p;
  p.views = views_dev; p.n = n_views; p.W = W; p.H = H; p.near_ = near_; p.flags = flags_dev;
  AAE_TRY(rasterise(m, p, workspace_dev, workspace_bytes_, s));
  coverage_kernel<<<dim3(32, n_views), 256, 0, s>>>(p);
  AAE_LAUNCH_OK();
  crop_kernel<<<dim3((unsigned)ceil_div(out_h * out_w, 256), n_views), 256, 0, s>>>(
      p, m->verts, m->faces, (int)m->nv, offsets_dev, pad_factor, out_h, out_w, col_map_dev, row_map_dev, crop_x_dev, mask_x_dev, crop_y_dev,
      obj_bb_dev);
  AAE_LAUNCH_OK();
  return AAE_OK;
}
