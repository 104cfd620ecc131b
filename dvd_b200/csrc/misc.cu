#include "misc.cuh"
#include "tc_epilogue.cuh"
#include <algorithm>

namespace dvd {

// ------------------------------------------------------------------------------------------ layer norm
template <int NV>   // float4 per lane: C = 128 * NV
__global__ void __launch_bounds__(256) k_layernorm(const float* __restrict__ in, int ldin, float* __restrict__ out, int ldo,
                                                   __nv_bfloat16* __restrict__ out16, __nv_bfloat16* __restrict__ out16_lo, int ldo16,
                                                   int rows, float eps, const float* __restrict__ w, const float* __restrict__ b,
                                                   const float* __restrict__ msh, const float* __restrict__ msc) {
  pdl_trigger();
  pdl_wait();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  constexpr int C = 128 * NV;
  const float4* x4 = reinterpret_cast<const float4*>(in + (size_t)row * ldin);
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) { v[i] = __ldg(x4 + lane + 32 * i); s += (v[i].x + v[i].y) + (v[i].z + v[i].w); }
  const float mean = warp_sum(s) * (1.0f / C);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    float a = v[i].x - mean, bb = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    q += (a * a + bb * bb) + (c * c + d * d);
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / C) + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c0 = (lane + 32 * i) * 4;
    float y[4] = {(v[i].x - mean) * rstd, (v[i].y - mean) * rstd, (v[i].z - mean) * rstd, (v[i].w - mean) * rstd};
    if (w) {
      float4 ww = __ldg(reinterpret_cast<const float4*>(w + c0)), bb = __ldg(reinterpret_cast<const float4*>(b + c0));
      y[0] = y[0] * ww.x + bb.x; y[1] = y[1] * ww.y + bb.y; y[2] = y[2] * ww.z + bb.z; y[3] = y[3] * ww.w + bb.w;
    }
    if (msc) {
      float4 sc = __ldg(reinterpret_cast<const float4*>(msc + c0)), sh = __ldg(reinterpret_cast<const float4*>(msh + c0));
      y[0] = y[0] * (1.f + sc.x) + sh.x; y[1] = y[1] * (1.f + sc.y) + sh.y;
      y[2] = y[2] * (1.f + sc.z) + sh.z; y[3] = y[3] * (1.f + sc.w) + sh.w;
    }
    if (out) *reinterpret_cast<float4*>(out + (size_t)row * ldo + c0) = make_float4(y[0], y[1], y[2], y[3]);
    if (out16) {
      uint2 u, l;
      split_bf16x2(y[0], y[1], u.x, l.x);
      split_bf16x2(y[2], y[3], u.y, l.y);
      *reinterpret_cast<uint2*>(out16 + (size_t)row * ldo16 + c0) = u;
      if (out16_lo) *reinterpret_cast<uint2*>(out16_lo + (size_t)row * ldo16 + c0) = l;
    }
  }
}

int layernorm(const float* in, int ldin, float* out, int ldo, __nv_bfloat16* out16, __nv_bfloat16* out16_lo, int ldo16, int rows, int C,
              float eps, const float* w, const float* b, const float* msh, const float* msc, cudaStream_t st) {
  DVD_REQUIRE(in && (out || out16) && rows > 0, "layernorm: bad args");
  DVD_REQUIRE(C == 384 || C == 1536, "layernorm: C must be 384 or 1536 (got %d)", C);
  DVD_REQUIRE(ldin % 4 == 0 && ldo % 4 == 0 && ldo16 % 4 == 0, "layernorm: ld %% 4");
  dim3 grid(cdiv(rows, 8));
  if (C == 384) DVD_CUDA(launch_pdl(4, k_layernorm<3>, grid, dim3(256), (size_t)0, st, in, ldin, out, ldo, out16, out16_lo, ldo16, rows, eps, w, b, msh, msc));
  else          DVD_CUDA(launch_pdl(4, k_layernorm<12>, grid, dim3(256), (size_t)0, st, in, ldin, out, ldo, out16, out16_lo, ldo16, rows, eps, w, b, msh, msc));
  DVD_LAUNCH_CHECK("k_layernorm");
  return 0;
}

// ------------------------------------------------------------------------------------------ layout kernels
__global__ void k_pack_y4(const float* __restrict__ y, const float* __restrict__ m, float* __restrict__ out, int B) {
  const size_t plane = 512 * 512;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= plane * B) return;
  size_t b = i / plane, px = i % plane;
  const float* yb = y + b * 3 * plane;
  float4 v = make_float4(__ldg(yb + px), __ldg(yb + plane + px), __ldg(yb + 2 * plane + px), __ldg(m + b * plane + px));
  reinterpret_cast<float4*>(out)[i] = v;
}
int pack_y4(const float* y512, const float* mask, float* out, int B, cudaStream_t st) {
  DVD_REQUIRE(y512 && mask && out && B > 0, "pack_y4: bad args");
  k_pack_y4<<<cdiv((long long)B * 512 * 512, 256), 256, 0, st>>>(y512, mask, out, B);
  DVD_LAUNCH_CHECK("k_pack_y4");
  return 0;
}

__global__ void k_maxpool2(const float4* __restrict__ in, float4* __restrict__ out, int B, int H, int W, int C4) {
  const int Ho = H / 2, Wo = W / 2;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t total = (size_t)B * Ho * Wo * C4;
  if (i >= total) return;
  int c = i % C4; size_t r = i / C4;
  int xo = r % Wo; r /= Wo;
  int yo = r % Ho; int b = r / Ho;
  const float4* p = in + (((size_t)b * H + 2 * yo) * W + 2 * xo) * C4 + c;
  float4 a = __ldg(p), bb = __ldg(p + C4), cc = __ldg(p + (size_t)W * C4), d = __ldg(p + (size_t)W * C4 + C4);
  out[i] = make_float4(fmaxf(fmaxf(a.x, bb.x), fmaxf(cc.x, d.x)), fmaxf(fmaxf(a.y, bb.y), fmaxf(cc.y, d.y)),
                       fmaxf(fmaxf(a.z, bb.z), fmaxf(cc.z, d.z)), fmaxf(fmaxf(a.w, bb.w), fmaxf(cc.w, d.w)));
}
int maxpool2_nhwc(const float* in, float* out, int B, int H, int W, int C, cudaStream_t st) {
  DVD_REQUIRE(in && out && C % 4 == 0 && H % 2 == 0 && W % 2 == 0, "maxpool2: bad args");
  size_t total = (size_t)B * (H / 2) * (W / 2) * (C / 4);
  k_maxpool2<<<cdiv(total, 256), 256, 0, st>>>((const float4*)in, (float4*)out, B, H, W, C / 4);
  DVD_LAUNCH_CHECK("k_maxpool2");
  return 0;
}

// one thread = one (pixel, tap pair): 8 of the 16-byte chunks of a 128-byte output row; chunks 5..7 (k >= 40) are zero and
// chunk 4 holds tap 8 + zeros
__global__ void __launch_bounds__(256) k_im2col_c4(const float4* __restrict__ in, uint4* __restrict__ out, int H, int W, size_t total, int f16) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;          // total = B*H*W*8 chunks
  if (i >= total) return;
  const int chunk = i & 7; const size_t pix = i >> 3;
  const int x = pix % W; const int y = (pix / W) % H; const size_t b = pix / ((size_t)W * H);
  float4 v[2];
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int tap = chunk * 2 + t;
    v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tap < 9) {
      const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) v[t] = __ldg(in + (b * H + yy) * W + xx);
    }
  }
  if (f16)                                     // one IEEE fp16 value per element (two-pass mode of the pyramid)
    out[i] = make_uint4(pack_f16x2(v[0].x, v[0].y), pack_f16x2(v[0].z, v[0].w), pack_f16x2(v[1].x, v[1].y), pack_f16x2(v[1].z, v[1].w));
  else
    out[i] = make_uint4(pack_bf16x2(v[0].x, v[0].y), pack_bf16x2(v[0].z, v[0].w), pack_bf16x2(v[1].x, v[1].y), pack_bf16x2(v[1].z, v[1].w));
}
int im2col3x3_c4_bf16(const float* in, __nv_bfloat16* out, int B, int H, int W, cudaStream_t st, int out_f16) {
  DVD_REQUIRE(in && out && B > 0, "im2col: bad args");
  size_t total = (size_t)B * H * W * 8;
  k_im2col_c4<<<cdiv(total, 256), 256, 0, st>>>((const float4*)in, (uint4*)out, H, W, total, out_f16);
  DVD_LAUNCH_CHECK("k_im2col_c4");
  return 0;
}

// 2x2 max pool on 16-bit NHWC (8 channels = 16 bytes per thread): bf16, or IEEE fp16 when f16; the output is written in the input's
// 16-bit type and / or as fp32
__global__ void k_maxpool2_bf16(const uint4* __restrict__ in, uint4* __restrict__ out16, float* __restrict__ out32, int B, int H, int W,
                                int C8, int f16) {
  const int Ho = H / 2, Wo = W / 2;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t total = (size_t)B * Ho * Wo * C8;
  if (i >= total) return;
  int c = i % C8; size_t r = i / C8;
  int xo = r % Wo; r /= Wo;
  int yo = r % Ho; int b = r / Ho;
  const size_t base = (((size_t)b * H + 2 * yo) * W + 2 * xo) * C8 + c;
  const size_t offs[4] = {0, (size_t)C8, (size_t)W * C8, (size_t)W * C8 + C8};
  float m[8];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const uint4 q = __ldg(in + base + offs[t]);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
    float f[8] = {__low2float(h[0]), __high2float(h[0]), __low2float(h[1]), __high2float(h[1]),
                  __low2float(h[2]), __high2float(h[2]), __low2float(h[3]), __high2float(h[3])};
    if (f16) {                                 // input (and 16-bit output) are single IEEE fp16 values
      const __half2* g = reinterpret_cast<const __half2*>(&q);
#pragma unroll
      for (int k = 0; k < 4; ++k) { const float2 t2 = __half22float2(g[k]); f[2 * k] = t2.x; f[2 * k + 1] = t2.y; }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) m[k] = t == 0 ? f[k] : fmaxf(m[k], f[k]);
  }
  if (out16 && f16) {                          // (the maximum of 16-bit values is a 16-bit value: exact)
    out16[i] = make_uint4(pack_f16x2(m[0], m[1]), pack_f16x2(m[2], m[3]), pack_f16x2(m[4], m[5]), pack_f16x2(m[6], m[7]));
  } else if (out16) {
    out16[i] = make_uint4(pack_bf16x2(m[0], m[1]), pack_bf16x2(m[2], m[3]), pack_bf16x2(m[4], m[5]), pack_bf16x2(m[6], m[7]));
  }
  if (out32) {
    float4* o = reinterpret_cast<float4*>(out32 + i * 8);
    o[0] = make_float4(m[0], m[1], m[2], m[3]);
    o[1] = make_float4(m[4], m[5], m[6], m[7]);
  }
}
int maxpool2_nhwc_bf16(const __nv_bfloat16* in, __nv_bfloat16* out16, float* out32, int B, int H, int W, int C, cudaStream_t st, int f16) {
  DVD_REQUIRE(in && (out16 || out32) && C % 8 == 0 && H % 2 == 0 && W % 2 == 0, "maxpool2_bf16: bad args");
  size_t total = (size_t)B * (H / 2) * (W / 2) * (C / 8);
  k_maxpool2_bf16<<<cdiv(total, 256), 256, 0, st>>>((const uint4*)in, (uint4*)out16, out32, B, H, W, C / 8, f16);
  DVD_LAUNCH_CHECK("k_maxpool2_bf16");
  return 0;
}

__global__ void k_nhwc_to_nchw(const float* __restrict__ in, float* __restrict__ out, int HW, int C) {
  __shared__ float tile[32][33];
  int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += 8) {
    int p = p0 + r, c = c0 + threadIdx.x;
    tile[r][threadIdx.x] = (p < HW && c < C) ? in[((size_t)b * HW + p) * C + c] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {
    int c = c0 + r, p = p0 + threadIdx.x;
    if (p < HW && c < C) out[((size_t)b * C + c) * HW + p] = tile[threadIdx.x][r];
  }
}
int nhwc_to_nchw(const float* in, float* out, int B, int H, int W, int C, cudaStream_t st) {
  DVD_REQUIRE(in && out, "nhwc_to_nchw: null");
  k_nhwc_to_nchw<<<dim3(cdiv(H * W, 32), cdiv(C, 32), B), dim3(32, 8), 0, st>>>(in, out, H * W, C);
  DVD_LAUNCH_CHECK("k_nhwc_to_nchw");
  return 0;
}

// ------------------------------------------------------------------------------------------ patchify
struct Out16 { __nv_bfloat16* hi; __nv_bfloat16* lo; };      // bf16 destination: plain (lo == null) or split pair
__device__ __forceinline__ void store4(float* A, Out16 A16, size_t off, float a, float b, float c, float d) {
  if (A) *reinterpret_cast<float4*>(A + off) = make_float4(a, b, c, d);
  if (A16.hi) {
    uint2 u, l;
    split_bf16x2(a, b, u.x, l.x);
    split_bf16x2(c, d, u.y, l.y);
    *reinterpret_cast<uint2*>(A16.hi + off) = u;
    if (A16.lo) *reinterpret_cast<uint2*>(A16.lo + off) = l;
  }
}

// block = one (b, h) token row x 32 channels; smem tile gives coalesced reads AND writes
__global__ void __launch_bounds__(256) k_patchify_nchw(const float* __restrict__ in, float* __restrict__ A, Out16 A16, int lda, int C) {
  __shared__ float tile[32][2][65];
  const int h = blockIdx.x, c0 = blockIdx.y * 32, b = blockIdx.z;
  for (int i = threadIdx.x; i < 32 * 128; i += 256) {
    int cc = i / 128, r = (i % 128) / 64, x = i % 64;
    int c = c0 + cc;
    tile[cc][r][x] = (c < C) ? __ldg(in + (((size_t)b * C + c) * 64 + 2 * h + r) * 64 + x) : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 32 * 32; i += 256) {       // (w, cc)
    int w = i / 32, cc = i % 32, c = c0 + cc;
    if (c >= C) continue;
    size_t off = ((size_t)(b * 32 + h) * 32 + w) * lda + (size_t)c * 4;
    store4(A, A16, off, tile[cc][0][2 * w], tile[cc][0][2 * w + 1], tile[cc][1][2 * w], tile[cc][1][2 * w + 1]);
  }
}
int patchify_nchw(const float* in, float* A, __nv_bfloat16* A16, __nv_bfloat16* A16_lo, int lda, int B, int C, cudaStream_t st) {
  DVD_REQUIRE(in && (A || A16) && lda % 4 == 0 && lda >= 4 * C, "patchify_nchw: bad args");
  k_patchify_nchw<<<dim3(32, cdiv(C, 32), B), 256, 0, st>>>(in, A, Out16{A16, A16_lo}, lda, C);
  DVD_LAUNCH_CHECK("k_patchify_nchw");
  return 0;
}

__global__ void k_patchify_nhwc(const float* __restrict__ in, float* __restrict__ A, Out16 A16, int lda, int C, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int c = i % C; size_t row = i / C;          // row = (b*32 + h)*32 + w
  int w = row % 32, h = (row / 32) % 32; size_t b = row / 1024;
  const float* p = in + ((b * 64 + 2 * h) * 64 + 2 * w) * C + c;
  store4(A, A16, row * lda + (size_t)c * 4, __ldg(p), __ldg(p + C), __ldg(p + 64 * C), __ldg(p + 65 * C));
}
int patchify_nhwc(const float* in, float* A, __nv_bfloat16* A16, __nv_bfloat16* A16_lo, int lda, int B, int C, cudaStream_t st) {
  DVD_REQUIRE(in && (A || A16) && lda % 4 == 0 && lda >= 4 * C, "patchify_nhwc: bad args");
  size_t total = (size_t)B * 1024 * C;
  k_patchify_nhwc<<<cdiv(total, 256), 256, 0, st>>>(in, A, Out16{A16, A16_lo}, lda, C, total);
  DVD_LAUNCH_CHECK("k_patchify_nhwc");
  return 0;
}

// ------------------------------------------------------------------------------------------ r operand (+ feature warp)
__global__ void __launch_bounds__(256) k_build_r(const float* __restrict__ flow, const float* __restrict__ feat,
                                                 const float* __restrict__ init_feat, int init_feat_div, int mode,
                                                 float* __restrict__ A, Out16 A16, int lda, int n_hyp) {
  pdl_trigger();                                    // programmatic dependent launch: the successor may be scheduled now,
  pdl_wait();                                       // and this kernel was possibly scheduled before its predecessor finished
  const int row = blockIdx.x;                  // (n*32 + h)*32 + w
  const int w = row % 32, h = (row / 32) % 32, n = row / 1024;
  const int c = threadIdx.x;                   // feature channel 0..255
  const float* fl = flow + (size_t)n * 2 * 4096;
  const float* ft = feat + (size_t)(n / n_hyp) * 4096 * 256;
  float v[4];
#pragma unroll
  for (int pq = 0; pq < 4; ++pq) {
    const int y = 2 * h + (pq >> 1), x = 2 * w + (pq & 1);
    if (mode == FEAT_EXPLICIT_OR_ZERO) {
      v[pq] = init_feat ? __ldg(init_feat + (((size_t)(n / init_feat_div) * 256 + c) * 64 + y) * 64 + x) : 0.f;
    } else if (mode == FEAT_ASIS) {
      v[pq] = __ldg(ft + ((size_t)y * 64 + x) * 256 + c);
    } else {
      // GD:618-624: grid = (pred_flow + base64)*2 - 1 ; base64 = coords/63 ; WP:73 grid_sample
      float gx = (__ldg(fl + y * 64 + x) + (float)x / 63.0f) * 2.0f - 1.0f;
      float gy = (__ldg(fl + 4096 + y * 64 + x) + (float)y / 63.0f) * 2.0f - 1.0f;
      float ix = ((gx + 1.f) / 2.f) * 63.f, iy = ((gy + 1.f) / 2.f) * 63.f;
      float fx = fminf(fmaxf(floorf(ix), -2.f), 65.f), fy = fminf(fmaxf(floorf(iy), -2.f), 65.f);
      int x0 = (int)fx, y0 = (int)fy;
      float ax = ix - fx, ay = iy - fy, bx = (fx + 1.f) - ix, by = (fy + 1.f) - iy;
      bool vx0 = x0 >= 0 && x0 < 64, vx1 = x0 + 1 >= 0 && x0 + 1 < 64, vy0 = y0 >= 0 && y0 < 64, vy1 = y0 + 1 >= 0 && y0 + 1 < 64;
      const float* p = ft + ((long long)y0 * 64 + x0) * 256 + c;
      float acc = 0.f;
      if (vy0 && vx0) acc += __ldg(p) * (bx * by);
      if (vy0 && vx1) acc += __ldg(p + 256) * (ax * by);
      if (vy1 && vx0) acc += __ldg(p + 64 * 256) * (bx * ay);
      if (vy1 && vx1) acc += __ldg(p + 65 * 256) * (ax * ay);
      v[pq] = acc;
    }
  }
  store4(A, A16, (size_t)row * lda + 8 + (size_t)c * 4, v[0], v[1], v[2], v[3]);
  if (c < 2) {   // flow channels: k = c*4 + p*2 + q
    const float* p = fl + (size_t)c * 4096 + (2 * h) * 64 + 2 * w;
    store4(A, A16, (size_t)row * lda + (size_t)c * 4, __ldg(p), __ldg(p + 1), __ldg(p + 64), __ldg(p + 65));
  }
  // zero the K padding (lda may exceed 1032 for the tensor-core path)
  for (int k = 1032 + c; k < lda; k += 256) {
    if (A) A[(size_t)row * lda + k] = 0.f;
    if (A16.hi) A16.hi[(size_t)row * lda + k] = __float2bfloat16_rn(0.f);
    if (A16.lo) A16.lo[(size_t)row * lda + k] = __float2bfloat16_rn(0.f);
  }
}
int build_r_operand(const float* init_flow, const float* feat_nhwc, const float* init_feat_nchw, int init_feat_div, int mode,
                    float* A, __nv_bfloat16* A16, __nv_bfloat16* A16_lo, int lda, int N, int n_hyp, cudaStream_t st) {
  DVD_REQUIRE(init_flow && feat_nhwc && (A || A16) && lda >= 1032 && lda % 4 == 0 && n_hyp > 0 && init_feat_div > 0, "build_r: bad args");
  DVD_CUDA(launch_pdl(16, k_build_r, dim3(N * 1024), dim3(256), (size_t)0, st, init_flow, feat_nhwc, init_feat_nchw, init_feat_div, mode, A, Out16{A16, A16_lo}, lda, n_hyp));
  DVD_LAUNCH_CHECK("k_build_r");
  return 0;
}

__global__ void k_obs_embed(const float* __restrict__ x, const float* __restrict__ W, const float* __restrict__ bias,
                            const float* __restrict__ pos, float* __restrict__ out, size_t total) {
  pdl_trigger();                                    // programmatic dependent launch: the successor may be scheduled now,
  pdl_wait();                                       // and this kernel was possibly scheduled before its predecessor finished
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int j = i % kHid; size_t row = i / kHid;
  int w = row % 32, h = (row / 32) % 32; size_t n = row / 1024;
  const float* p = x + n * 2 * 4096 + (2 * h) * 64 + 2 * w;
  const float* wr = W + (size_t)j * 8;
  float acc = 0.f;
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    const float* q = p + c * 4096;
    acc += __ldg(wr + c * 4 + 0) * __ldg(q) + __ldg(wr + c * 4 + 1) * __ldg(q + 1) + __ldg(wr + c * 4 + 2) * __ldg(q + 64) +
           __ldg(wr + c * 4 + 3) * __ldg(q + 65);
  }
  out[i] = acc + __ldg(bias + j) + __ldg(pos + (row % 1024) * kHid + j);
}
int obs_embed(const float* x, const float* W, const float* bias, const float* pos, float* out, int N, cudaStream_t st) {
  DVD_REQUIRE(x && W && bias && pos && out, "obs_embed: null");
  size_t total = (size_t)N * 1024 * kHid;
  DVD_CUDA(launch_pdl(16, k_obs_embed, dim3(cdiv(total, 256)), dim3(256), (size_t)0, st, x, W, bias, pos, out, total));
  DVD_LAUNCH_CHECK("k_obs_embed");
  return 0;
}

// ------------------------------------------------------------------------------------------ softmax
template <int NV>   // float4 per lane, n = 128*NV
__global__ void __launch_bounds__(256) k_softmax(float* __restrict__ S, long long rows) {
  long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float4* p = reinterpret_cast<float4*>(S + row * (128 * NV));
  float4 v[NV];
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < NV; ++i) { v[i] = p[lane + 32 * i]; m = fmaxf(m, fmaxf(fmaxf(v[i].x, v[i].y), fmaxf(v[i].z, v[i].w))); }
  m = warp_max(m);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x = expf(v[i].x - m); v[i].y = expf(v[i].y - m); v[i].z = expf(v[i].z - m); v[i].w = expf(v[i].w - m);
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float inv = 1.0f / warp_sum(s);
#pragma unroll
  for (int i = 0; i < NV; ++i) p[lane + 32 * i] = make_float4(v[i].x * inv, v[i].y * inv, v[i].z * inv, v[i].w * inv);
}
int softmax_rows(float* S, long long rows, int n, cudaStream_t st) {
  DVD_REQUIRE(S && rows > 0 && n % 128 == 0 && n <= 1024, "softmax_rows: n must be a multiple of 128 <= 1024 (got %d)", n);
  dim3 grid(cdiv(rows, 8));
  switch (n / 128) {
    case 1: k_softmax<1><<<grid, 256, 0, st>>>(S, rows); break;
    case 2: k_softmax<2><<<grid, 256, 0, st>>>(S, rows); break;
    case 4: k_softmax<4><<<grid, 256, 0, st>>>(S, rows); break;
    case 8: k_softmax<8><<<grid, 256, 0, st>>>(S, rows); break;
    default: set_error("softmax_rows: unsupported n=%d", n); return DVD_E_BADARG;
  }
  DVD_LAUNCH_CHECK("k_softmax");
  return 0;
}

// ------------------------------------------------------------------------------------------ small dense layers
constexpr int GEMV_MAXR = 8;
// block = 8 warps = 8 output features.  Each warp first requests its whole weight row (<= 12 x 16 bytes per lane for K <= 1536): the
// weights do not depend on the previous kernel, so under programmatic dependent launch this HBM fetch (9.4 MB for the 1536x1536
// layers of the adaptive positional encoding) overlaps the predecessor's execution; only then does the block wait for its input
// rows, stage them (activated) in shared memory and reduce.
// blockIdx.y selects one of up to two independent problems of the same shape (the h- and w-branch of the adaptive positional
// encoding run side by side: two dependent launches per step instead of four).
struct GemvProb { const float* in[2]; const float* W[2]; const float* b[2]; float* out[2]; };
__global__ void __launch_bounds__(256) k_gemv(const GemvProb pr, int ldin, int ldo, int rows, int N, int K, int silu_in, int in_mod, int act) {
  extern __shared__ float xs[];                      // [rows][K]
  const float* __restrict__ in = pr.in[blockIdx.y];
  const float* __restrict__ W = pr.W[blockIdx.y];
  const float* __restrict__ b = pr.b[blockIdx.y];
  float* __restrict__ out = pr.out[blockIdx.y];
  pdl_trigger();
  const int j = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int K4 = K >> 2;
  float4 wv[12];
  {
    const float4* wr = reinterpret_cast<const float4*>(W + (size_t)min(j, N - 1) * K);
#pragma unroll
    for (int i = 0; i < 12; ++i) {
      const int k = lane + 32 * i;
      wv[i] = (k < K4) ? __ldg(wr + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  pdl_wait();                                        // the input rows are the previous kernel's output
  if (in_mod == 0 && (ldin & 3) == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0) {
    // the usual case: whole rows, 16-byte loads, all of a thread's loads in flight at once (the scalar loop below pays one L2 round
    // trip per iteration: 12 of them for two 1536-wide rows)
#pragma unroll 4
    for (int i = threadIdx.x; i < rows * K4; i += 256) {
      const int r = i / K4, k = i - r * K4;
      float4 x = __ldg(reinterpret_cast<const float4*>(in + (size_t)r * ldin) + k);
      if (silu_in) { x.x = silu(x.x); x.y = silu(x.y); x.z = silu(x.z); x.w = silu(x.w); }
      reinterpret_cast<float4*>(xs)[i] = x;
    }
  } else {
    for (int i = threadIdx.x; i < rows * K; i += 256) {
      const int r = i / K, k = i - r * K;
      float x = __ldg(in + (size_t)r * ldin + (in_mod > 0 ? (k % in_mod) : k));
      xs[i] = silu_in ? silu(x) : x;
    }
  }
  __syncthreads();
  if (j >= N) return;
  float acc[GEMV_MAXR];
#pragma unroll
  for (int r = 0; r < GEMV_MAXR; ++r) acc[r] = 0.f;
#pragma unroll
  for (int i = 0; i < 12; ++i) {
    const int k = lane + 32 * i;
    if (k < K4) {
#pragma unroll
      for (int r = 0; r < GEMV_MAXR; ++r) {
        if (r < rows) {
          const float4 x = *reinterpret_cast<const float4*>(xs + r * K + 4 * k);
          acc[r] += (wv[i].x * x.x + wv[i].y * x.y) + (wv[i].z * x.z + wv[i].w * x.w);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < GEMV_MAXR; ++r) {
    if (r < rows) {
      float v = warp_sum(acc[r]);
      if (lane == 0) {
        if (b) v += __ldg(b + j);
        if (act == 1) v = fmaxf(v, 0.f);
        else if (act == 3) v = sigmoidf_(v);
        else if (act == 4) v = silu(v);
        out[(size_t)r * ldo + j] = v;
      }
    }
  }
}
static int gemv_launch(const GemvProb& pr, int nprob, int ldin, int ldo, int rows, int N, int K, int silu_in, int in_mod, int act, cudaStream_t st) {
  for (int r0 = 0; r0 < rows; r0 += GEMV_MAXR) {
    int nr = rows - r0 < GEMV_MAXR ? rows - r0 : GEMV_MAXR;
    GemvProb q = pr;
    for (int i = 0; i < nprob; ++i) { q.in[i] = pr.in[i] + (size_t)r0 * ldin; q.out[i] = pr.out[i] + (size_t)r0 * ldo; }
    DVD_CUDA(launch_pdl(16, k_gemv, dim3(cdiv(N, 8), nprob), dim3(256), (size_t)nr * K * sizeof(float), st, q, ldin, ldo, nr, N, K, silu_in, in_mod,
                        act));
    DVD_LAUNCH_CHECK("k_gemv");
  }
  return 0;
}
int gemv(const float* in, int ldin, const float* W, const float* b, float* out, int ldo, int rows, int N, int K, int silu_in,
         int in_mod, int act, cudaStream_t st) {
  DVD_REQUIRE(in && W && out && N > 0 && K > 0 && K % 4 == 0 && K <= 1536, "gemv: bad args (K=%d)", K);
  DVD_REQUIRE((reinterpret_cast<uintptr_t>(W) & 15) == 0, "gemv: W must be 16-byte aligned");
  GemvProb pr{{in, in}, {W, W}, {b, b}, {out, out}};
  return gemv_launch(pr, 1, ldin, ldo, rows, N, K, silu_in, in_mod, act, st);
}
// two independent layers of the same shape in one launch: out0 = act(W0 in0 + b0), out1 = act(W1 in1 + b1)
int gemv_pair(const float* in0, const float* in1, int ldin, const float* W0, const float* W1, const float* b0, const float* b1, float* out0,
              float* out1, int ldo, int rows, int N, int K, int act, cudaStream_t st) {
  DVD_REQUIRE(in0 && in1 && W0 && W1 && out0 && out1 && N > 0 && K > 0 && K % 4 == 0 && K <= 1536, "gemv_pair: bad args (K=%d)", K);
  DVD_REQUIRE(((reinterpret_cast<uintptr_t>(W0) | reinterpret_cast<uintptr_t>(W1)) & 15) == 0, "gemv_pair: W must be 16-byte aligned");
  GemvProb pr{{in0, in1}, {W0, W1}, {b0, b1}, {out0, out1}};
  return gemv_launch(pr, 2, ldin, ldo, rows, N, K, 0, 0, act, st);
}

__global__ void k_timestep_embedding(const float* __restrict__ t, float* __restrict__ out, int rows) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * 128) return;
  int r = i / 128, k = i % 128;
  // CM:123-129: freqs = exp(-ln(10000) * k / 128) in fp32 ; args = t * freqs ; cat(cos, sin)
  float f = expf(-9.210340371976184f * (float)k / 128.0f);
  float a = t[r] * f;
  out[r * 256 + k] = cosf(a);
  out[r * 256 + 128 + k] = sinf(a);
}
int timestep_embedding(const float* t, float* out, int rows, cudaStream_t st) {
  k_timestep_embedding<<<cdiv(rows * 128, 128), 128, 0, st>>>(t, out, rows);
  DVD_LAUNCH_CHECK("k_timestep_embedding");
  return 0;
}

// ------------------------------------------------------------------------------------------ decoder positional encoding
// deterministic two-stage mean: 32 token chunks of 32, then a fixed-order finish
__global__ void __launch_bounds__(128) k_token_partial(const float* __restrict__ X, float* __restrict__ part, int C) {
  pdl_trigger();                                    // programmatic dependent launch: the successor may be scheduled now,
  pdl_wait();                                       // and this kernel was possibly scheduled before its predecessor finished
  const int c = blockIdx.x * 128 + threadIdx.x, chunk = blockIdx.y, n = blockIdx.z;
  if (c >= C) return;
  const float* p = X + ((size_t)n * 1024 + chunk * 32) * C + c;
  float s = 0.f;
#pragma unroll 8
  for (int t = 0; t < 32; ++t) s += __ldg(p + (size_t)t * C);
  part[((size_t)n * 32 + chunk) * C + c] = s;
}
__global__ void k_token_finish(const float* __restrict__ part, float* __restrict__ out, int C, int total) {
  pdl_trigger();                                    // programmatic dependent launch: the successor may be scheduled now,
  pdl_wait();                                       // and this kernel was possibly scheduled before its predecessor finished
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int n = i / C, c = i % C;
  float s = 0.f;
  for (int k = 0; k < 32; ++k) s += part[((size_t)n * 32 + k) * C + c];
  out[i] = s * (1.0f / 1024.0f);
}
int token_mean(const float* X, float* out, int N, int C, cudaStream_t st) {
  // `out` must have room for N*C results followed by N*32*C partials
  DVD_REQUIRE(X && out, "token_mean: null");
  float* part = out + (size_t)N * C;
  DVD_CUDA(launch_pdl(16, k_token_partial, dim3(cdiv(C, 128), 32, N), dim3(128), (size_t)0, st, X, part, C));
  DVD_LAUNCH_CHECK("k_token_partial");
  DVD_CUDA(launch_pdl(16, k_token_finish, dim3(cdiv(N * C, 256)), dim3(256), (size_t)0, st, (const float*)part, out, C, N * C));
  DVD_LAUNCH_CHECK("k_token_finish");
  return 0;
}

__global__ void k_posenc_add(float4* __restrict__ X, const float4* __restrict__ hs, const float4* __restrict__ ws,
                             const float4* __restrict__ hpe, const float4* __restrict__ wpe, int C4, size_t total) {
  pdl_trigger();                                    // programmatic dependent launch: the successor may be scheduled now,
  pdl_wait();                                       // and this kernel was possibly scheduled before its predecessor finished
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int c = i % C4; size_t row = i / C4;
  int tok = row % 1024; size_t n = row / 1024;
  float4 x = X[i], a = __ldg(hs + n * C4 + c), b = __ldg(ws + n * C4 + c);
  float4 hp = __ldg(hpe + (size_t)(tok / 32) * C4 + c), wp = __ldg(wpe + (size_t)(tok % 32) * C4 + c);
  // CA:153: out = x + h_pos_encoding + w_pos_encoding (left to right)
  x.x = (x.x + a.x * hp.x) + b.x * wp.x; x.y = (x.y + a.y * hp.y) + b.y * wp.y;
  x.z = (x.z + a.z * hp.z) + b.z * wp.z; x.w = (x.w + a.w * hp.w) + b.w * wp.w;
  X[i] = x;
}
int posenc_add(float* X, const float* hs, const float* ws, const float* hpe, const float* wpe, int N, int C, cudaStream_t st) {
  DVD_REQUIRE(X && hs && ws && hpe && wpe && C % 4 == 0, "posenc_add: bad args");
  size_t total = (size_t)N * 1024 * (C / 4);
  DVD_CUDA(launch_pdl(16, k_posenc_add, dim3(cdiv(total, 256)), dim3(256), (size_t)0, st, (float4*)X, (const float4*)hs, (const float4*)ws,
                      (const float4*)hpe, (const float4*)wpe, C / 4, total));
  DVD_LAUNCH_CHECK("k_posenc_add");
  return 0;
}

// posenc_add for the fused-LayerNorm path: one warp per token row; also writes the row as ONE fp16 value per element (the operand of
// the two-pass q|k|v GEMM) and its (sum, sum of squares) for the LayerNorm that GEMM's epilogue applies (slot 0 = whole row, the other
// chunk slots zero).
__global__ void __launch_bounds__(256) k_posenc_ln(float* __restrict__ X, const float4* __restrict__ hs, const float4* __restrict__ ws,
                                                   const float4* __restrict__ hpe, const float4* __restrict__ wpe, __nv_bfloat16* __restrict__ x16,
                                                   float* __restrict__ stats, int chunks, int rows) {
  pdl_trigger();                                    // programmatic dependent launch: the successor may be scheduled now,
  pdl_wait();                                       // and this kernel was possibly scheduled before its predecessor finished
  constexpr int C4 = 384;                       // 1536 / 4
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int tok = row & 1023, n = row >> 10;
  float4* xr = reinterpret_cast<float4*>(X) + (size_t)row * C4;
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < 12; ++i) {
    const int c = lane + 32 * i;
    float4 x = xr[c];
    const float4 a = __ldg(hs + (size_t)n * C4 + c), b = __ldg(ws + (size_t)n * C4 + c);
    const float4 hp = __ldg(hpe + (size_t)(tok >> 5) * C4 + c), wp = __ldg(wpe + (size_t)(tok & 31) * C4 + c);
    // CA:153: out = x + h_pos_encoding + w_pos_encoding (left to right)
    x.x = (x.x + a.x * hp.x) + b.x * wp.x; x.y = (x.y + a.y * hp.y) + b.y * wp.y;
    x.z = (x.z + a.z * hp.z) + b.z * wp.z; x.w = (x.w + a.w * hp.w) + b.w * wp.w;
    xr[c] = x;
    *reinterpret_cast<uint2*>(x16 + ((size_t)row * C4 + c) * 4) = make_uint2(pack_f16x2(x.x, x.y), pack_f16x2(x.z, x.w));
    s1 += (x.x + x.y) + (x.z + x.w);
    s2 += (x.x * x.x + x.y * x.y) + (x.z * x.z + x.w * x.w);
  }
  s1 = warp_sum(s1); s2 = warp_sum(s2);
  float2* sr = reinterpret_cast<float2*>(stats) + (size_t)row * chunks;
  for (int k = lane; k < chunks; k += 32) sr[k] = k == 0 ? make_float2(s1, s2) : make_float2(0.f, 0.f);
}
int posenc_add_ln(float* X, const float* hs, const float* ws, const float* hpe, const float* wpe, int N, int C, __nv_bfloat16* x16,
                  float* stats, int chunks, cudaStream_t st) {
  DVD_REQUIRE(X && hs && ws && hpe && wpe && x16 && stats && C == 1536 && chunks == C / 32, "posenc_add_ln: bad args");
  const int rows = N * 1024;
  DVD_CUDA(launch_pdl(16, k_posenc_ln, dim3(cdiv(rows, 8)), dim3(256), (size_t)0, st, X, (const float4*)hs, (const float4*)ws, (const float4*)hpe,
                      (const float4*)wpe, x16, stats, chunks, rows));
  DVD_LAUNCH_CHECK("k_posenc_ln");
  return 0;
}

// ------------------------------------------------------------------------------------------ depthwise 3x3
__global__ void __launch_bounds__(256) k_dwconv(const float4* __restrict__ in, const float4* __restrict__ w9, const float4* __restrict__ sc,
                                                const float4* __restrict__ sh, float* __restrict__ out, __nv_bfloat16* __restrict__ out16,
                                                int C4, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int c = i % C4; size_t row = i / C4;
  int tok = row % 1024; size_t n = row / 1024;
  int y = tok / 32, x = tok % 32;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    int yy = y + ky - 1;
    if (yy < 0 || yy >= 32) continue;
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      int xx = x + kx - 1;
      if (xx < 0 || xx >= 32) continue;
      float4 v = __ldg(in + (n * 1024 + yy * 32 + xx) * C4 + c), ww = __ldg(w9 + (size_t)(ky * 3 + kx) * C4 + c);
      acc.x = fmaf(v.x, ww.x, acc.x); acc.y = fmaf(v.y, ww.y, acc.y); acc.z = fmaf(v.z, ww.z, acc.z); acc.w = fmaf(v.w, ww.w, acc.w);
    }
  }
  float4 s = __ldg(sc + c), t = __ldg(sh + c);
  float r0 = fmaxf(acc.x * s.x + t.x, 0.f), r1 = fmaxf(acc.y * s.y + t.y, 0.f), r2 = fmaxf(acc.z * s.z + t.z, 0.f), r3 = fmaxf(acc.w * s.w + t.w, 0.f);
  store4(out, Out16{out16, nullptr}, i * 4, r0, r1, r2, r3);
}
// bf16 / bf16-pair variant for the tensor path.  CTA = one sample x one 64-channel slice x a band of kDwRows output rows across all
// 32 x positions.  The kDwRows + 2 input rows of the band are loaded once from global memory (all ten 16-byte loads per thread and
// array issued before any is used), converted to fp32 (hi + lo) and staged in shared memory; a thread then computes 8 channels of one
// x position for the whole band from there, walking the input column by column (kx outer) like the fp32 kernel: per output the taps
// are accumulated kx-major, ky-minor, and taps outside the image are skipped.  At batch 1 (N = 2) the 256 CTAs of 80 KB each run as
// one wave at 2 CTAs per SM; larger batches just add CTAs (one flat grid index).
constexpr int kDwRows = 8, kDwCh = 64, kDwThreads = 256;
constexpr int kDwSmem = (kDwRows + 2) * 32 * kDwCh * 4;
// float4 slot of channel quad q (0..15) inside a 64-channel row: the upper half is shifted by one slot so that the 8 threads of a
// quarter-warp (8 channel groups reading quads 2g, 2g + 1) hit 8 distinct 4-bank groups
__device__ __forceinline__ int dw_slot(int q) { return q ^ (q >> 3); }

__global__ void __launch_bounds__(kDwThreads, 2) k_dwconv_band(const uint4* __restrict__ in, const uint4* __restrict__ in_lo,
                                                               const float4* __restrict__ w9, const float4* __restrict__ sc,
                                                               const float4* __restrict__ sh, uint4* __restrict__ out,
                                                               uint4* __restrict__ out_lo, int C8) {
  extern __shared__ float4 s_in[];                        // [kDwRows + 2][32 x][16 slots]: fp32 hi + lo of input rows y0-1 .. y0+kDwRows
  __shared__ float4 s_w[9][16], s_sc[16], s_sh[16];
  pdl_trigger();
  constexpr int bands = 32 / kDwRows;
  const int slices = C8 / 8;                              // 64-channel slices
  const int slice = blockIdx.x % slices, band = (blockIdx.x / slices) % bands;
  const size_t n = blockIdx.x / slices / bands;
  const int y0 = band * kDwRows, C4 = C8 * 2;
  const int g = threadIdx.x & 7, x = threadIdx.x >> 3;    // this thread's 8 channels (quads 2g, 2g + 1) and x position
  // taps and BN of the slice do not depend on the previous kernel: staged before griddepcontrol.wait
  for (int e = threadIdx.x; e < 11 * 16; e += kDwThreads) {
    const int q = e & 15, c4 = slice * 16 + q;
    if (e < 9 * 16) s_w[e >> 4][dw_slot(q)] = __ldg(w9 + (size_t)(e >> 4) * C4 + c4);
    else if (e < 10 * 16) s_sc[dw_slot(q)] = __ldg(sc + c4);
    else s_sh[dw_slot(q)] = __ldg(sh + c4);
  }
  pdl_wait();
  const size_t base = n * 1024 * C8 + slice * 8 + g;     // 16-byte lane (sample n, token 0, this thread's channel group)
  uint4 vh[kDwRows + 2], vl[kDwRows + 2];
#pragma unroll
  for (int i = 0; i < kDwRows + 2; ++i) {                 // staged row i = input row y0 - 1 + i
    const int yy = y0 - 1 + i;
    if (yy < 0 || yy >= 32) continue;
    vh[i] = __ldg(in + base + (size_t)(yy * 32 + x) * C8);
    if (in_lo) vl[i] = __ldg(in_lo + base + (size_t)(yy * 32 + x) * C8);
  }
#pragma unroll
  for (int i = 0; i < kDwRows + 2; ++i) {
    const int yy = y0 - 1 + i;
    if (yy < 0 || yy >= 32) continue;
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&vh[i]);
    float f[8] = {__low2float(h[0]), __high2float(h[0]), __low2float(h[1]), __high2float(h[1]),
                  __low2float(h[2]), __high2float(h[2]), __low2float(h[3]), __high2float(h[3])};
    if (in_lo) {                                          // split pair: value = hi + lo
      const __nv_bfloat162* hl = reinterpret_cast<const __nv_bfloat162*>(&vl[i]);
#pragma unroll
      for (int k = 0; k < 4; ++k) { f[2 * k] += __low2float(hl[k]); f[2 * k + 1] += __high2float(hl[k]); }
    }
    float4* row = s_in + (i * 32 + x) * 16;
    row[dw_slot(2 * g)] = make_float4(f[0], f[1], f[2], f[3]);
    row[dw_slot(2 * g + 1)] = make_float4(f[4], f[5], f[6], f[7]);
  }
  __syncthreads();
  float acc[kDwRows][8];
#pragma unroll
  for (int o = 0; o < kDwRows; ++o)
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[o][k] = 0.f;
#pragma unroll 1                                             // (one copy of the column body: the kernel's code is fetched cold on every launch)
  for (int kx = 0; kx < 3; ++kx) {
    const int xx = x + kx - 1;
    if (xx < 0 || xx >= 32) continue;
    float w[3][8];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const float4 w0 = s_w[ky * 3 + kx][dw_slot(2 * g)], w1 = s_w[ky * 3 + kx][dw_slot(2 * g + 1)];
      w[ky][0] = w0.x; w[ky][1] = w0.y; w[ky][2] = w0.z; w[ky][3] = w0.w; w[ky][4] = w1.x; w[ky][5] = w1.y; w[ky][6] = w1.z; w[ky][7] = w1.w;
    }
#pragma unroll
    for (int r = -1; r <= kDwRows; ++r) {
      const int yy = y0 + r;
      if (yy < 0 || yy >= 32) continue;
      const float4* p = s_in + ((r + 1) * 32 + xx) * 16;
      const float4 a = p[dw_slot(2 * g)], b = p[dw_slot(2 * g + 1)];
      const float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const int o = r + 1 - ky;                          // output row (inside the band) that sees input row r through tap row ky
        if (o < 0 || o >= kDwRows) continue;
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[o][k] = fmaf(f[k], w[ky][k], acc[o][k]);
      }
    }
  }
  const float4 s0 = s_sc[dw_slot(2 * g)], s1 = s_sc[dw_slot(2 * g + 1)];
  const float4 t0 = s_sh[dw_slot(2 * g)], t1 = s_sh[dw_slot(2 * g + 1)];
#pragma unroll
  for (int o = 0; o < kDwRows; ++o) {
    const float r8[8] = {fmaxf(acc[o][0] * s0.x + t0.x, 0.f), fmaxf(acc[o][1] * s0.y + t0.y, 0.f), fmaxf(acc[o][2] * s0.z + t0.z, 0.f),
                         fmaxf(acc[o][3] * s0.w + t0.w, 0.f), fmaxf(acc[o][4] * s1.x + t1.x, 0.f), fmaxf(acc[o][5] * s1.y + t1.y, 0.f),
                         fmaxf(acc[o][6] * s1.z + t1.z, 0.f), fmaxf(acc[o][7] * s1.w + t1.w, 0.f)};
    uint4 ov, ol;
    split_bf16x2(r8[0], r8[1], ov.x, ol.x); split_bf16x2(r8[2], r8[3], ov.y, ol.y);
    split_bf16x2(r8[4], r8[5], ov.z, ol.z); split_bf16x2(r8[6], r8[7], ov.w, ol.w);
    const size_t at = base + (size_t)((y0 + o) * 32 + x) * C8;
    out[at] = ov;
    if (out_lo) out_lo[at] = ol;
  }
}
int dwconv3x3_bn_relu_bf16(const __nv_bfloat16* in, const __nv_bfloat16* in_lo, const float* w9c, const float* scale, const float* shift,
                           __nv_bfloat16* out, __nv_bfloat16* out_lo, int N, int C, cudaStream_t st) {
  DVD_REQUIRE(in && w9c && scale && shift && out, "dwconv_bf16: null pointer");
  DVD_REQUIRE(N > 0 && C > 0 && C % kDwCh == 0, "dwconv_bf16: N = %d, C = %d (C must be a positive multiple of %d)", N, C, kDwCh);
  DVD_REQUIRE((((uintptr_t)in | (uintptr_t)in_lo | (uintptr_t)w9c | (uintptr_t)scale | (uintptr_t)shift | (uintptr_t)out | (uintptr_t)out_lo) & 15) == 0,
              "dwconv_bf16: pointers must be 16-byte aligned");
  const long long ctas = (long long)N * (32 / kDwRows) * (C / kDwCh);
  DVD_REQUIRE(ctas <= 0x7fffffffLL, "dwconv_bf16: batch too large for the grid");
  DVD_SET_MAX_SMEM(k_dwconv_band, kDwSmem);
  DVD_CUDA(launch_pdl(8, k_dwconv_band, dim3((unsigned)ctas), dim3(kDwThreads), (size_t)kDwSmem, st, (const uint4*)in, (const uint4*)in_lo,
                      (const float4*)w9c, (const float4*)scale, (const float4*)shift, (uint4*)out, (uint4*)out_lo, C / 8));
  DVD_LAUNCH_CHECK("k_dwconv_band");
  return 0;
}

int dwconv3x3_bn_relu(const float* in, const float* w9c, const float* scale, const float* shift, float* out, __nv_bfloat16* out16,
                      int N, int C, cudaStream_t st) {
  DVD_REQUIRE(in && w9c && scale && shift && (out || out16) && C % 4 == 0, "dwconv: bad args");
  size_t total = (size_t)N * 1024 * (C / 4);
  k_dwconv<<<cdiv(total, 256), 256, 0, st>>>((const float4*)in, (const float4*)w9c, (const float4*)scale, (const float4*)shift, out, out16,
                                             C / 4, total);
  DVD_LAUNCH_CHECK("k_dwconv");
  return 0;
}

// ------------------------------------------------------------------------------------------ final layer + DDIM update
__global__ void __launch_bounds__(256) k_final(const float* __restrict__ X, const float* __restrict__ lw, const float* __restrict__ lb,
                                               const float* __restrict__ shift, const float* __restrict__ scale,
                                               const float* __restrict__ W8, const float* __restrict__ b8,
                                               const float* __restrict__ init_flow, const float* __restrict__ x_t, float a, float b,
                                               float* __restrict__ pred, float* __restrict__ x_prev, int rows) {
  pdl_trigger();                                    // programmatic dependent launch: the successor may be scheduled now,
  pdl_wait();                                       // and this kernel was possibly scheduled before its predecessor finished
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  constexpr int NV = 12, C = 1536;
  const float4* x4 = reinterpret_cast<const float4*>(X + (size_t)row * C);
  float v[NV][4];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    float4 t = __ldg(x4 + lane + 32 * i);
    v[i][0] = t.x; v[i][1] = t.y; v[i][2] = t.z; v[i][3] = t.w;
    s += (t.x + t.y) + (t.z + t.w);
  }
  float mean = warp_sum(s) * (1.0f / C), q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) { float d = v[i][j] - mean; q += d * d; }
  float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / C) + 1e-5f);            // decoder.layer_norm, CA:457
  s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c0 = (lane + 32 * i) * 4;
    float4 ww = __ldg(reinterpret_cast<const float4*>(lw + c0)), bb = __ldg(reinterpret_cast<const float4*>(lb + c0));
    v[i][0] = (v[i][0] - mean) * rstd * ww.x + bb.x; v[i][1] = (v[i][1] - mean) * rstd * ww.y + bb.y;
    v[i][2] = (v[i][2] - mean) * rstd * ww.z + bb.z; v[i][3] = (v[i][3] - mean) * rstd * ww.w + bb.w;
    s += (v[i][0] + v[i][1]) + (v[i][2] + v[i][3]);
  }
  mean = warp_sum(s) * (1.0f / C); q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) { float d = v[i][j] - mean; q += d * d; }
  rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / C) + 1e-6f);                  // norm_final, CM:321,334
  float acc[8];
#pragma unroll
  for (int o = 0; o < 8; ++o) acc[o] = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c0 = (lane + 32 * i) * 4;
    float4 sc = __ldg(reinterpret_cast<const float4*>(scale + c0)), sh = __ldg(reinterpret_cast<const float4*>(shift + c0));
    float y0 = (v[i][0] - mean) * rstd * (1.f + sc.x) + sh.x, y1 = (v[i][1] - mean) * rstd * (1.f + sc.y) + sh.y;
    float y2 = (v[i][2] - mean) * rstd * (1.f + sc.z) + sh.z, y3 = (v[i][3] - mean) * rstd * (1.f + sc.w) + sh.w;
#pragma unroll
    for (int o = 0; o < 8; ++o) {
      float4 w = __ldg(reinterpret_cast<const float4*>(W8 + (size_t)o * C + c0));
      acc[o] += (y0 * w.x + y1 * w.y) + (y2 * w.z + y3 * w.w);
    }
  }
#pragma unroll
  for (int o = 0; o < 8; ++o) acc[o] = warp_sum(acc[o]);
  if (lane < 8) {
    float val = 0.f;
#pragma unroll
    for (int o = 0; o < 8; ++o) if (lane == o) val = acc[o];
    const int o = lane;
    val += __ldg(b8 + o);
    // CM:563-565 unpatchify 'nhwpqc->nchpwq': o = p*4 + q*2 + c
    const int p = o >> 2, qq = (o >> 1) & 1, c = o & 1;
    const int tok = row % 1024, n = row / 1024, h = tok / 32, w = tok % 32;
    const size_t idx = ((size_t)(n * 2 + c) * 64 + 2 * h + p) * 64 + 2 * w + qq;
    const float pr = val + __ldg(init_flow + idx);                         // CM:645-646
    pred[idx] = pr;
    if (x_prev) x_prev[idx] = a * pr + b * __ldg(x_t + idx);              // GD:470-489 with eta = 0
  }
}
int final_layer(const float* X, const float* ln_w, const float* ln_b, const float* shift, const float* scale, const float* W8,
                const float* b8, const float* init_flow, const float* x_t, float a, float b, float* pred, float* x_prev, int N,
                cudaStream_t st) {
  DVD_REQUIRE(X && ln_w && ln_b && shift && scale && W8 && b8 && init_flow && pred && (x_t || !x_prev), "final_layer: null");
  DVD_CUDA(launch_pdl(16, k_final, dim3(cdiv(N * 1024, 8)), dim3(256), (size_t)0, st, X, ln_w, ln_b, shift, scale, W8, b8, init_flow, x_t, a, b, pred, x_prev, N * 1024));
  DVD_LAUNCH_CHECK("k_final");
  return 0;
}

__global__ void k_hyp_mean_clamp(const float* __restrict__ pred, float* __restrict__ out, int n_hyp, int total) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  int d = i / 8192, e = i % 8192;
  float s = 0.f;
  for (int h = 0; h < n_hyp; ++h) s += pred[((size_t)d * n_hyp + h) * 8192 + e];
  out[i] = fminf(fmaxf(s / (float)n_hyp, -1.f), 1.f);
}
int hyp_mean_clamp(const float* pred, float* out, int docs, int n_hyp, cudaStream_t st) {
  DVD_REQUIRE(pred && out && n_hyp > 0, "hyp_mean_clamp: bad args");
  if (docs == 0) return 0;
  k_hyp_mean_clamp<<<cdiv(docs * 8192, 256), 256, 0, st>>>(pred, out, n_hyp, docs * 8192);
  DVD_LAUNCH_CHECK("k_hyp_mean_clamp");
  return 0;
}

__global__ void k_f32_to_bf16(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __float2bfloat16_rn(in[i]);
}
int f32_to_bf16(const float* in, __nv_bfloat16* out, long long n, cudaStream_t st) {
  k_f32_to_bf16<<<cdiv(n, 256), 256, 0, st>>>(in, out, n);
  DVD_LAUNCH_CHECK("k_f32_to_bf16");
  return 0;
}

// fp32 -> split pair hi = bf16(v), lo = bf16(v - hi)   (test hooks; the product path splits in the producing epilogues)
__global__ void k_f32_split_bf16(const float* __restrict__ in, __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = in[i];
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  hi[i] = h;
  lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}
int f32_split_bf16(const float* in, __nv_bfloat16* hi, __nv_bfloat16* lo, long long n, cudaStream_t st) {
  k_f32_split_bf16<<<cdiv(n, 256), 256, 0, st>>>(in, hi, lo, n);
  DVD_LAUNCH_CHECK("k_f32_split_bf16");
  return 0;
}
__global__ void k_f32_to_f16(const float* __restrict__ in, __half* __restrict__ out, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __float2half_rn(in[i]);
}
int f32_to_f16(const float* in, void* out, long long n, cudaStream_t st) {
  k_f32_to_f16<<<cdiv(n, 256), 256, 0, st>>>(in, (__half*)out, n);
  DVD_LAUNCH_CHECK("k_f32_to_f16");
  return 0;
}
__global__ void k_f32_split_f16(const float* __restrict__ in, __half* __restrict__ hi, __half* __restrict__ lo, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = in[i];
  const __half h = __float2half_rn(v);
  hi[i] = h;
  lo[i] = __float2half_rn(v - __half2float(h));
}
int f32_split_f16(const float* in, void* hi, void* lo, long long n, cudaStream_t st) {
  k_f32_split_f16<<<cdiv(n, 256), 256, 0, st>>>(in, (__half*)hi, (__half*)lo, n);
  DVD_LAUNCH_CHECK("k_f32_split_f16");
  return 0;
}
// out = hi (+ lo)
__global__ void k_pair_to_f32(const __nv_bfloat16* __restrict__ hi, const __nv_bfloat16* __restrict__ lo, float* __restrict__ out, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __bfloat162float(hi[i]) + (lo ? __bfloat162float(lo[i]) : 0.f);
}
int pair_to_f32(const __nv_bfloat16* hi, const __nv_bfloat16* lo, float* out, long long n, cudaStream_t st) {
  k_pair_to_f32<<<cdiv(n, 256), 256, 0, st>>>(hi, lo, out, n);
  DVD_LAUNCH_CHECK("k_pair_to_f32");
  return 0;
}

}  // namespace dvd
namespace dvd {
__global__ void k_bf16_to_f32(const __nv_bfloat16* __restrict__ in, float* __restrict__ out, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __bfloat162float(in[i]);
}
int bf16_to_f32(const __nv_bfloat16* in, float* out, long long n, cudaStream_t st) {
  k_bf16_to_f32<<<cdiv(n, 256), 256, 0, st>>>(in, out, n);
  DVD_LAUNCH_CHECK("k_bf16_to_f32");
  return 0;
}
}  // namespace dvd
