// K11 — fused map-upsample + base ramp + affine + bilinear gather (HBM-bandwidth bound).
//
// Replaces, in ONE pass over the output, the reference chain
//   EV:301  F.interpolate(map64 -> HxW, bilinear, align_corners=True)
//   EV:304  F.interpolate(coords_grid(512,512)/511 -> HxW)          (the "base" identity ramp)
//   EV:306  ((s + base) * 2 - 1) * 0.987
//   visualization_utils.py:75 -> WP:73  F.grid_sample(photo, grid, bilinear, align_corners=True, zeros)
//   visualization_utils.py:76-77        .astype(uint8)               (u8 variants)
// Algorithmic HBM traffic: read photo once + write output once = 24 B/px (fp32 NCHW, C=3) or
// 6 B/px (uint8 HWC).  The reference moves ~88 B/px (two materialised fields, five elementwise
// passes, grid read, gather, store).
//
// Three kernels, one arithmetic:
//   k_unwarp_tma   fp32 photos (the roofline kernel): persistent CTAs, source windows staged in shared memory by TMA, output tiles
//                  leaving through TMA stores (see the comment above the kernel);
//   k_unwarp_fast  uint8 photos and shapes the TMA path does not take: a CTA covers a 128 x 8 pixel tile, per-tile coefficient tables
//                  and the vertically pre-blended coarse-map window in shared memory, gathers through L1;
//   k_unwarp       fully general fallback (tiny photos / huge maps).
// The 64x64 coarse map (32 KB) is read through the read-only path and stays L1/L2 resident.
// k_unwarp_u8_mixed and k_unwarp_u8_sized run the uint8 tile bodies over a host-planned table of documents.  The sized kernel writes an
// Ho x Wo page: EV:301,304 with size=(s*Ho, s*Wo) instead of the photo's (H, W), WP:73 at that grid, then the mean of each s x s block
// (box supersampling when shrinking; s = 1 is the reference chain at the output size) before the .astype(uint8) truncation.
#include "common.cuh"
#include "tc_common.cuh"
#include <stdlib.h>
#include <algorithm>

namespace dvd {

struct UnwarpGeom {
  int H, W, mh, mw;
  float sy, sx;      // (mh-1)/(H-1), (mw-1)/(W-1)   map upsample scales (align_corners=True)
  float by, bx;      // 511/(H-1), 511/(W-1)          base-ramp upsample scales
  float affine;      // 0.987
};

__host__ static UnwarpGeom make_geom(int H, int W, int mh, int mw, float affine) {
  UnwarpGeom g;
  g.H = H; g.W = W; g.mh = mh; g.mw = mw;
  // torch area_pixel_compute_scale(align_corners=True): (in-1)/(out-1) in fp32, 0 when out == 1
  g.sy = H > 1 ? (float)(mh - 1) / (float)(H - 1) : 0.f;
  g.sx = W > 1 ? (float)(mw - 1) / (float)(W - 1) : 0.f;
  g.by = H > 1 ? 511.0f / (float)(H - 1) : 0.f;
  g.bx = W > 1 ? 511.0f / (float)(W - 1) : 0.f;
  g.affine = affine;
  return g;
}

// bilinear weights of torch upsample_bilinear2d(align_corners=True) along one axis
__device__ __forceinline__ void up_coeff(float scale, int dst, int in_size, int& i0, int& ip, float& l0, float& l1) {
  float r = scale * (float)dst;
  i0 = (int)r;
  ip = (i0 < in_size - 1) ? 1 : 0;
  l1 = r - (float)i0;
  l0 = 1.0f - l1;
}

// value of the 512-ramp (k/511) upsampled to `dst` (EV:304 + EV:330-335 coords_grid_tensor)
__device__ __forceinline__ float base_ramp(float scale, int dst) {
  int k0, kp; float l0, l1;
  up_coeff(scale, dst, 512, k0, kp, l0, l1);
  float a = (float)k0 / 511.0f, b = (float)(k0 + kp) / 511.0f;
  return l0 * a + l1 * b;
}

// normalised sampling coordinates (gx, gy) in [-1,1]-ish for output pixel (i, j)
__device__ __forceinline__ void sample_coords(const UnwarpGeom& g, const float* __restrict__ map, int i, int j,
                                              float& gx, float& gy) {
  int y0, yp, x0, xp; float ly0, ly1, lx0, lx1;
  up_coeff(g.sy, i, g.mh, y0, yp, ly0, ly1);
  up_coeff(g.sx, j, g.mw, x0, xp, lx0, lx1);
  const float* m0 = map + (size_t)y0 * g.mw + x0;            // channel 0 = x displacement
  const float* m1 = m0 + (size_t)g.mh * g.mw;                // channel 1 = y displacement
  int dy = yp * g.mw;
  float sx = ly0 * (lx0 * __ldg(m0) + lx1 * __ldg(m0 + xp)) + ly1 * (lx0 * __ldg(m0 + dy) + lx1 * __ldg(m0 + dy + xp));
  float sy = ly0 * (lx0 * __ldg(m1) + lx1 * __ldg(m1 + xp)) + ly1 * (lx0 * __ldg(m1 + dy) + lx1 * __ldg(m1 + dy + xp));
  gx = ((sx + base_ramp(g.bx, j)) * 2.0f - 1.0f) * g.affine;
  gy = ((sy + base_ramp(g.by, i)) * 2.0f - 1.0f) * g.affine;
}

struct Taps {           // torch grid_sampler_2d bilinear, align_corners=True, padding zeros
  int x0, y0;
  float nw, ne, sw, se;
  bool vx0, vx1, vy0, vy1;
};

__device__ __forceinline__ Taps make_taps(float gx, float gy, int H, int W) {
  Taps t;
  float ix = ((gx + 1.f) / 2.f) * (float)(W - 1);
  float iy = ((gy + 1.f) / 2.f) * (float)(H - 1);
  float fx = floorf(ix), fy = floorf(iy);
  // clamp before the int conversion so that wild coordinates cannot overflow
  fx = fminf(fmaxf(fx, -2.f), (float)W + 1.f);
  fy = fminf(fmaxf(fy, -2.f), (float)H + 1.f);
  t.x0 = (int)fx; t.y0 = (int)fy;
  float ax = ix - fx, ay = iy - fy;       // == ix - ix_nw
  float bx = (fx + 1.f) - ix, by = (fy + 1.f) - iy;
  t.nw = bx * by; t.ne = ax * by; t.sw = bx * ay; t.se = ax * ay;
  t.vx0 = (t.x0 >= 0) & (t.x0 < W); t.vx1 = (t.x0 + 1 >= 0) & (t.x0 + 1 < W);
  t.vy0 = (t.y0 >= 0) & (t.y0 < H); t.vy1 = (t.y0 + 1 >= 0) & (t.y0 + 1 < H);
  return t;
}

template <typename T>
__device__ __forceinline__ float gather(const T* __restrict__ plane, const Taps& t, int W, int cstride) {
  // plane points at channel c of pixel (0,0); element (y,x) is plane[(y*W + x) * cstride]
  float v = 0.f;
  const T* p = plane + ((long long)t.y0 * W + t.x0) * cstride;
  if (t.vy0 & t.vx0) v += (float)__ldg(p) * t.nw;
  if (t.vy0 & t.vx1) v += (float)__ldg(p + cstride) * t.ne;
  if (t.vy1 & t.vx0) v += (float)__ldg(p + (long long)W * cstride) * t.sw;
  if (t.vy1 & t.vx1) v += (float)__ldg(p + (long long)(W + 1) * cstride) * t.se;
  return v;
}

__device__ __forceinline__ uint8_t to_u8_trunc(float v) {   // numpy .astype(uint8) on a non-negative value
  return (uint8_t)__float2uint_rz(fminf(fmaxf(v, 0.f), 255.f));
}

constexpr int TILE_W = 128, TILE_H = 8;   // 32 x 8 threads, 4 px per thread

// IN: 0 = fp32 NCHW, 1 = uint8 HWC.  OUT likewise.
//
// Per-CTA prologue: the column-only and row-only parts of the coordinate chain (upsample index / weight of the coarse
// map, upsampled base ramp with its two fp32 divisions) are computed ONCE per tile column / tile row into shared
// memory (128 + 8 entries), so the per-pixel path is: 8 coarse-map loads, 2 bilinear blends, affine, tap weights and
// 4*C gathers.  Tiles whose four taps are all inside the photo for every pixel of the warp (the common case) take an
// unpredicated path so that the 4*C*4 gathers of a thread are issued back to back.
//
// The per-tile bodies (unwarp_tile, unwarp_tile_fast) take photo / output / map bases, a geometry and the tile (x, y, image b):
// the fixed-size kernels pass the batch bases and blockIdx (so their address arithmetic is the one they always had), the
// persistent mixed-size and sized kernels one document's bases, their own tile walk and b = 0.  A body never returns early (the
// persistent loop has barriers): rows past the output skip the work and still reach every __syncthreads.
// The geometry g is the OUTPUT's (coordinate chain, tile walk, output rows); Hi x Wi is the photo the taps read.  Every caller but
// the sized kernel passes Hi = g.H, Wi = g.W.
template <int IN_U8, int OUT_U8, int C>
__device__ __forceinline__ void unwarp_tile(const void* __restrict__ photo_, const float* __restrict__ map, void* __restrict__ out_,
                                            const UnwarpGeom& g, unsigned tx, unsigned ty, unsigned b, int Hi, int Wi) {
  __shared__ float s_bx[TILE_W], s_lx[TILE_W], s_by[TILE_H], s_ly[TILE_H];
  __shared__ int s_x0[TILE_W], s_y0[TILE_H];
  const int tid = threadIdx.y * 32 + threadIdx.x;
  if (tid < TILE_W) {
    const int j = min(tx * TILE_W + tid, g.W - 1);
    int x0, xp; float l0, l1;
    up_coeff(g.sx, j, g.mw, x0, xp, l0, l1);
    s_x0[tid] = x0 | (xp << 16); s_lx[tid] = l1; s_bx[tid] = base_ramp(g.bx, j);
  } else if (tid < TILE_W + TILE_H) {
    const int r = tid - TILE_W;
    const int i = min(ty * TILE_H + r, g.H - 1);
    int y0, yp; float l0, l1;
    up_coeff(g.sy, i, g.mh, y0, yp, l0, l1);
    s_y0[r] = y0 | (yp << 16); s_ly[r] = l1; s_by[r] = base_ramp(g.by, i);
  }
  __syncthreads();
  const int i = ty * TILE_H + threadIdx.y;
  const int j0 = (tx * (TILE_W / 4) + threadIdx.x) * 4;
  // a warp is one tile row; its lanes left of the right edge are a prefix of the warp, and only they take part in the vote below
  if (i < g.H && j0 < g.W) {
  const int W = g.W, H = g.H;
  const int plane = H * W, pplane = Hi * Wi;                    // output / photo: < 2^31 elements per image (checked on the host)
  const float* __restrict__ mapb = map + (size_t)b * 2 * g.mh * g.mw;
  const int y0m = s_y0[threadIdx.y] & 0xffff, dy = (s_y0[threadIdx.y] >> 16) * g.mw;
  const float ly1 = s_ly[threadIdx.y], ly0 = 1.0f - ly1, byv = s_by[threadIdx.y];
  const float* __restrict__ mrow = mapb + y0m * g.mw;
  const int mplane = g.mh * g.mw;

  int off[4];                    // element offset of the NW tap: y0 * W + x0
  float wnw[4], wne[4], wsw[4], wse[4];
  bool inside = true;
  int vmask[4];
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    const int cj = threadIdx.x * 4 + p;                         // column inside the tile
    const int x0m = s_x0[cj] & 0xffff, xp = s_x0[cj] >> 16;
    const float lx1 = s_lx[cj], lx0 = 1.0f - lx1;
    const float* m0 = mrow + x0m;
    const float* m1 = m0 + mplane;
    const float sx = ly0 * (lx0 * __ldg(m0) + lx1 * __ldg(m0 + xp)) + ly1 * (lx0 * __ldg(m0 + dy) + lx1 * __ldg(m0 + dy + xp));
    const float sy = ly0 * (lx0 * __ldg(m1) + lx1 * __ldg(m1 + xp)) + ly1 * (lx0 * __ldg(m1 + dy) + lx1 * __ldg(m1 + dy + xp));
    const float gx = ((sx + s_bx[cj]) * 2.0f - 1.0f) * g.affine;
    const float gy = ((sy + byv) * 2.0f - 1.0f) * g.affine;
    const Taps t = make_taps(gx, gy, Hi, Wi);
    off[p] = t.y0 * Wi + t.x0;
    wnw[p] = t.nw; wne[p] = t.ne; wsw[p] = t.sw; wse[p] = t.se;
    vmask[p] = (int)t.vx0 | ((int)t.vx1 << 1) | ((int)t.vy0 << 2) | ((int)t.vy1 << 3);
    inside = inside && (vmask[p] == 15 || j0 + p >= W);
    if (j0 + p >= W) { vmask[p] = 0; off[p] = 0; }
  }
  float res[C][4];
  const int live = min(32, (W - (int)tx * TILE_W + 3) / 4);
  if (__all_sync(live == 32 ? 0xffffffffu : (1u << live) - 1u, inside) && j0 + 3 < W) {
    // ---- fast path: every tap of every pixel of this warp is inside the photo
    if (IN_U8) {
      const uint8_t* __restrict__ ph = (const uint8_t*)photo_ + (size_t)b * pplane * C;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const uint8_t* q = ph + (size_t)off[p] * C;
#pragma unroll
        for (int c = 0; c < C; ++c) {
          float v = (float)__ldg(q + c) * wnw[p];
          v += (float)__ldg(q + C + c) * wne[p];
          v += (float)__ldg(q + (size_t)Wi * C + c) * wsw[p];
          v += (float)__ldg(q + (size_t)(Wi + 1) * C + c) * wse[p];
          res[c][p] = v;
        }
      }
    } else {
      const float* __restrict__ ph = (const float*)photo_ + (size_t)b * C * pplane;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float* pc = ph + (size_t)c * pplane;
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          const float* q = pc + off[p];
          float v = __ldg(q) * wnw[p];
          v += __ldg(q + 1) * wne[p];
          v += __ldg(q + Wi) * wsw[p];
          v += __ldg(q + Wi + 1) * wse[p];
          res[c][p] = v;
        }
      }
    }
  } else {
    // ---- border path: per-tap validity (zeros padding), same accumulation order
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      Taps t;
      t.nw = wnw[p]; t.ne = wne[p]; t.sw = wsw[p]; t.se = wse[p];
      t.vx0 = vmask[p] & 1; t.vx1 = vmask[p] & 2; t.vy0 = vmask[p] & 4; t.vy1 = vmask[p] & 8;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        float v = 0.f;
        if (IN_U8) {
          const uint8_t* q = (const uint8_t*)photo_ + ((size_t)b * pplane + off[p]) * C + c;
          if (t.vy0 & t.vx0) v += (float)__ldg(q) * t.nw;
          if (t.vy0 & t.vx1) v += (float)__ldg(q + C) * t.ne;
          if (t.vy1 & t.vx0) v += (float)__ldg(q + (long long)Wi * C) * t.sw;
          if (t.vy1 & t.vx1) v += (float)__ldg(q + (long long)(Wi + 1) * C) * t.se;
        } else {
          const float* q = (const float*)photo_ + ((size_t)b * C + c) * pplane + off[p];
          if (t.vy0 & t.vx0) v += __ldg(q) * t.nw;
          if (t.vy0 & t.vx1) v += __ldg(q + 1) * t.ne;
          if (t.vy1 & t.vx0) v += __ldg(q + Wi) * t.sw;
          if (t.vy1 & t.vx1) v += __ldg(q + Wi + 1) * t.se;
        }
        res[c][p] = v;
      }
    }
  }
  const bool full = (j0 + 3 < W);
  if (OUT_U8) {
    uint8_t* o = (uint8_t*)out_ + ((size_t)b * plane + (size_t)i * W + j0) * C;
    uint8_t bytes[4 * C];
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int c = 0; c < C; ++c) bytes[p * C + c] = to_u8_trunc(res[c][p]);
    if (full && ((reinterpret_cast<uintptr_t>(o) & 3) == 0)) {
#pragma unroll
      for (int w = 0; w < C; ++w) {   // 4*C bytes = C 32-bit words
        uint32_t v = bytes[4 * w] | (bytes[4 * w + 1] << 8) | (bytes[4 * w + 2] << 16) | ((uint32_t)bytes[4 * w + 3] << 24);
        reinterpret_cast<uint32_t*>(o)[w] = v;
      }
    } else {
      int n = min(4, W - j0) * C;
      for (int q = 0; q < n; ++q) o[q] = bytes[q];
    }
  } else {
#pragma unroll
    for (int c = 0; c < C; ++c) {
      float* o = (float*)out_ + ((size_t)b * C + c) * plane + (size_t)i * W + j0;
      if (full && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
        __stcs(reinterpret_cast<float4*>(o), make_float4(res[c][0], res[c][1], res[c][2], res[c][3]));  // streaming store
      } else {
        for (int p = 0; p < 4 && j0 + p < W; ++p) o[p] = res[c][p];
      }
    }
  }
  }
}

template <int IN_U8, int OUT_U8, int C>
__global__ void __launch_bounds__(256) k_unwarp(const void* __restrict__ photo_, const float* __restrict__ map,
                                                void* __restrict__ out_, UnwarpGeom g) {
  unwarp_tile<IN_U8, OUT_U8, C>(photo_, map, out_, g, blockIdx.x, blockIdx.y, blockIdx.z, g.H, g.W);
}

// ---------------------------------------------------------------------------------------------------------------------
// Fast variant (the one the hot path uses).  Differences from k_unwarp above:
//   * the coarse map is blended VERTICALLY once per tile row in the CTA prologue (v[r][k] = ly0*m[y0][k] + ly1*m[y1][k] for the
//     few map columns the tile touches), so a pixel needs 2 shared-memory reads + 1 blend per channel instead of 4 global loads
//     + 3 blends (horizontal-then-vertical vs vertical-then-horizontal blending differ by <= 1 ulp of the map, ~1e-4 px);
//   * tap set-up without clamps: floor via cvt.rmi, one unsigned compare per axis decides "all four taps inside";
//   * taps of the four pixels of a thread are issued back to back on the (common) all-inside path.
// Falls back to k_unwarp when the tile would touch more than UW_WIN map columns (tiny photos / huge maps).
constexpr int UW_WIN = 16;

template <int IN_U8, int OUT_U8, int C>
__device__ __forceinline__ void unwarp_tile_fast(const void* __restrict__ photo_, const float* __restrict__ map,
                                                 void* __restrict__ out_, const UnwarpGeom& g, unsigned tx, unsigned ty, unsigned b,
                                                 int Hi, int Wi) {
  __shared__ float s_bx[TILE_W], s_lx[TILE_W], s_by[TILE_H], s_ly[TILE_H];
  __shared__ int s_kx[TILE_W], s_y0[TILE_H];
  __shared__ float s_v[2][TILE_H][UW_WIN];
  const int tid = threadIdx.y * 32 + threadIdx.x;
  const float* __restrict__ mapb = map + (size_t)b * 2 * g.mh * g.mw;
  const int jt0 = tx * TILE_W;
  // window of map columns touched by this tile: x0(first column) .. x0(last column) + 1
  int wx0;
  {
    int xp; float l0, l1;
    up_coeff(g.sx, min(jt0, g.W - 1), g.mw, wx0, xp, l0, l1);
  }
  if (tid < TILE_W) {
    const int j = min(jt0 + tid, g.W - 1);
    int x0, xp; float l0, l1;
    up_coeff(g.sx, j, g.mw, x0, xp, l0, l1);
    s_kx[tid] = (x0 - wx0) | (xp << 16); s_lx[tid] = l1; s_bx[tid] = base_ramp(g.bx, j);
  } else if (tid < TILE_W + TILE_H) {
    const int r = tid - TILE_W;
    const int i = min(ty * TILE_H + r, g.H - 1);
    int y0, yp; float l0, l1;
    up_coeff(g.sy, i, g.mh, y0, yp, l0, l1);
    s_y0[r] = y0 | (yp << 16); s_ly[r] = l1; s_by[r] = base_ramp(g.by, i);
  }
  __syncthreads();
  if (tid < 2 * TILE_H * UW_WIN) {             // vertical blend of the map window: [channel][tile row][window column]
    const int k = tid % UW_WIN, r = (tid / UW_WIN) % TILE_H, ch = tid / (UW_WIN * TILE_H);
    const int col = min(wx0 + k, g.mw - 1);
    const int y0 = s_y0[r] & 0xffff, yp = s_y0[r] >> 16;
    const float l1 = s_ly[r], l0 = 1.0f - l1;
    const float* m = mapb + (size_t)ch * g.mh * g.mw + (size_t)y0 * g.mw + col;
    s_v[ch][r][k] = l0 * __ldg(m) + l1 * __ldg(m + yp * g.mw);
  }
  __syncthreads();
  const int i = ty * TILE_H + threadIdx.y;
  const int j0 = jt0 + threadIdx.x;                       // pixel p of this thread is column j0 + 32*p: a warp-level
  if (i < g.H) {                                          // load/store then covers 32 CONSECUTIVE pixels (one 128-byte line);
                                                          // whole warps skip (a warp is one tile row): *_sync masks stay valid
  const int W = g.W, H = g.H;
  const int plane = H * W, pplane = Hi * Wi;                  // output / photo
  const float byv = s_by[threadIdx.y];
  const float fw = (float)(Wi - 1), fh = (float)(Hi - 1);
  int off[4];
  float wnw[4], wne[4], wsw[4], wse[4];
  int x0s[4], y0s[4];
  bool inside = true;
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    const int cj = threadIdx.x + 32 * p;
    const int k = s_kx[cj] & 0xffff, xp = s_kx[cj] >> 16;
    const float lx1 = s_lx[cj], lx0 = 1.0f - lx1;
    const float sx = lx0 * s_v[0][threadIdx.y][k] + lx1 * s_v[0][threadIdx.y][k + xp];
    const float sy = lx0 * s_v[1][threadIdx.y][k] + lx1 * s_v[1][threadIdx.y][k + xp];
    const float gx = ((sx + s_bx[cj]) * 2.0f - 1.0f) * g.affine;
    const float gy = ((sy + byv) * 2.0f - 1.0f) * g.affine;
    const float ix = ((gx + 1.f) / 2.f) * fw, iy = ((gy + 1.f) / 2.f) * fh;      // grid_sampler_unnormalize, align_corners=True
    const int x0 = __float2int_rd(ix), y0 = __float2int_rd(iy);
    const float fx = (float)x0, fy = (float)y0;
    const float ax = ix - fx, ay = iy - fy, bx = (fx + 1.f) - ix, byw = (fy + 1.f) - iy;
    wnw[p] = bx * byw; wne[p] = ax * byw; wsw[p] = bx * ay; wse[p] = ax * ay;
    x0s[p] = x0; y0s[p] = y0;
    off[p] = y0 * Wi + x0;
    inside = inside && (((unsigned)x0 < (unsigned)(Wi - 1)) & ((unsigned)y0 < (unsigned)(Hi - 1)));
  }
  float res[C][4];
  if (__all_sync(0xffffffffu, inside) && jt0 + TILE_W <= W) {
    // all-inside path.  Address arithmetic is kept to one 64-bit pointer per pixel plus one add per channel / row: the tap
    // loads then use immediate offsets (profiles/r1_ncu_unwarp.txt showed ~6 integer instructions per load before this).
    if (IN_U8) {
      const uint8_t* __restrict__ ph = (const uint8_t*)photo_ + (size_t)b * pplane * C;
      const size_t rowb = (size_t)Wi * C;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const uint8_t* q0 = ph + (size_t)off[p] * C;
        const uint8_t* q1 = q0 + rowb;
#pragma unroll
        for (int c = 0; c < C; ++c) {
          float v = (float)__ldg(q0 + c) * wnw[p];
          v += (float)__ldg(q0 + C + c) * wne[p];
          v += (float)__ldg(q1 + c) * wsw[p];
          v += (float)__ldg(q1 + C + c) * wse[p];
          res[c][p] = v;
        }
      }
    } else {
      const float* __restrict__ ph = (const float*)photo_ + (size_t)b * C * pplane;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const float* q0 = ph + off[p];
        const float* q1 = q0 + Wi;
#pragma unroll
        for (int c = 0; c < C; ++c) {
          const float* a = q0 + (size_t)c * pplane;
          const float* d = q1 + (size_t)c * pplane;
          float v = __ldg(a) * wnw[p];
          v += __ldg(a + 1) * wne[p];
          v += __ldg(d) * wsw[p];
          v += __ldg(d + 1) * wse[p];
          res[c][p] = v;
        }
      }
    }
  } else {
    // border path: per-tap validity (zeros padding); coordinates may be wild, so validity is tested before any address is formed
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const int x0 = x0s[p], y0 = y0s[p];
      const bool px_ok = (j0 + 32 * p < W);
      const bool vx0 = px_ok && x0 >= 0 && x0 < Wi, vx1 = px_ok && x0 >= -1 && x0 < Wi - 1;
      const bool vy0 = y0 >= 0 && y0 < Hi, vy1 = y0 >= -1 && y0 < Hi - 1;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        float v = 0.f;
        if (IN_U8) {
          const uint8_t* base = (const uint8_t*)photo_ + (size_t)b * pplane * C + c;
          if (vy0 && vx0) v += (float)__ldg(base + ((long long)y0 * Wi + x0) * C) * wnw[p];
          if (vy0 && vx1) v += (float)__ldg(base + ((long long)y0 * Wi + x0 + 1) * C) * wne[p];
          if (vy1 && vx0) v += (float)__ldg(base + ((long long)(y0 + 1) * Wi + x0) * C) * wsw[p];
          if (vy1 && vx1) v += (float)__ldg(base + ((long long)(y0 + 1) * Wi + x0 + 1) * C) * wse[p];
        } else {
          const float* base = (const float*)photo_ + ((size_t)b * C + c) * pplane;
          if (vy0 && vx0) v += __ldg(base + (long long)y0 * Wi + x0) * wnw[p];
          if (vy0 && vx1) v += __ldg(base + (long long)y0 * Wi + x0 + 1) * wne[p];
          if (vy1 && vx0) v += __ldg(base + (long long)(y0 + 1) * Wi + x0) * wsw[p];
          if (vy1 && vx1) v += __ldg(base + (long long)(y0 + 1) * Wi + x0 + 1) * wse[p];
        }
        res[c][p] = v;
      }
    }
  }
  if (OUT_U8) {
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      if (j0 + 32 * p < W) {
        uint8_t* o = (uint8_t*)out_ + ((size_t)b * plane + (size_t)i * W + j0 + 32 * p) * C;
#pragma unroll
        for (int c = 0; c < C; ++c) o[c] = to_u8_trunc(res[c][p]);
      }
    }
  } else {
#pragma unroll
    for (int c = 0; c < C; ++c) {
      float* o = (float*)out_ + ((size_t)b * C + c) * plane + (size_t)i * W + j0;
#pragma unroll
      for (int p = 0; p < 4; ++p)
        if (j0 + 32 * p < W) __stcs(o + 32 * p, res[c][p]);
    }
  }
  }
}

template <int IN_U8, int OUT_U8, int C>
__global__ void __launch_bounds__(256) k_unwarp_fast(const void* __restrict__ photo_, const float* __restrict__ map,
                                                     void* __restrict__ out_, UnwarpGeom g) {
  unwarp_tile_fast<IN_U8, OUT_U8, C>(photo_, map, out_, g, blockIdx.x, blockIdx.y, blockIdx.z, g.H, g.W);
}

// ---------------------------------------------------------------------------------------------------------------------
// TMA-staged, persistent, software-pipelined variant (the hot path).
//
// The gather kernels above are LATENCY bound (profiles/: ~45% of the warps active, "long scoreboard" stalls, 0.3 of the HBM
// roofline): a CTA computes coordinates, then waits for its gathers, then stores, and too few bytes are in flight per SM.
// Here the photo moves through shared memory with bulk-tensor copies that run AHEAD of the arithmetic:
//
//   * persistent CTAs (3-5 per SM) walk 32 x 32 output tiles (square tiles: a sheared / rotated source footprint grows with
//     (1 + shear)^2, the least for a square);  warp 8 is the (load) PRODUCER, warps 0..7 are CONSUMERS, joined by an NS-stage ring of
//     source windows with full/empty mbarriers;
//   * producer, per tile: the tap origins of an 8 x 8 sample grid of the tile (tile corners and edges included), straight from the
//     coarse map, give the predicted source window (+1 pixel margin); it then issues cp.async.bulk.tensor loads of that window:
//     8-row boxes per channel plane, first column aligned down to 16 bytes (a TMA requirement for unswizzled maps).  Elements
//     outside the photo arrive as zeros, which IS grid_sample's zeros padding.  The producer runs NS tiles ahead of the consumers,
//     so the HBM latency of a window is hidden behind the arithmetic of the previous tiles;
//   * consumers, per tile: the tile's column / row tables (coarse-map index + weight, upsampled base ramp) and the vertically
//     pre-blended coarse-map window (32 rows x 8 map columns x 2 channels) in shared memory; then thread (lane, warp) owns column
//     `lane` of rows warp, warp+8, warp+16, warp+24, so every warp access covers 32 consecutive pixels.  Per pixel: 2 x LDS.64 of the
//     blended map, the coordinate chain of the reference in the same order, then 4*C taps as shared-memory loads at compile-time
//     offsets from ONE address.  A pixel whose taps fall outside the predicted window (the prediction is a heuristic; strongly sheared
//     or wild maps) gathers from global memory with per-tap validity tests, so the result never depends on the prediction;
//   * the output tile is written to shared memory and handed (mbarrier) to the STORE warp (warp 9), which issues one
//     cp.async.bulk.tensor store per tile (asynchronous, full lines, clips ragged image edges) and frees the buffer again.
constexpr int T2 = 32;                  // output tile edge
constexpr int W8 = 8;                   // coarse-map window columns per tile
constexpr int SB_ROWS = 40;             // staged window: max rows (5 boxes of 8)
constexpr int SB_ROW_F32 = 56;          //   floats per staged row (NCHW fp32): >= 53 usable columns after alignment
constexpr int SB_ROW_U8 = 176;          //   bytes per staged row (HWC uint8, C <= 3): >= 53 pixels after alignment
constexpr int UW_THREADS = 320;         // 8 consumer warps + load (producer) warp + store warp

struct __align__(128) TileTab {         // per-tile tables, built by the consumer warps (double buffered)
  float2 sv[T2][W8];                    // vertically blended coarse map (x, y displacement) for tile row r, window column k
  float lx[T2], bx[T2], by[T2];         // horizontal blend weight, upsampled base ramp (x), base ramp (y)
  int k[T2];                            // window column of tile column j
};

__device__ __forceinline__ void tap_setup(const TileTab& tb, int k, float lx0, float lx1, float bxv, int rr, float affine, float fw, float fh,
                                          int& x0, int& y0, float& wnw, float& wne, float& wsw, float& wse) {
  const float2 va = tb.sv[rr][k], vb = tb.sv[rr][k + 1];
  const float sx = lx0 * va.x + lx1 * vb.x;
  const float sy = lx0 * va.y + lx1 * vb.y;
  const float gx = ((sx + bxv) * 2.0f - 1.0f) * affine;
  const float gy = ((sy + tb.by[rr]) * 2.0f - 1.0f) * affine;
  const float ix = ((gx + 1.f) / 2.f) * fw, iy = ((gy + 1.f) / 2.f) * fh;      // grid_sampler_unnormalize, align_corners=True
  x0 = __float2int_rd(ix); y0 = __float2int_rd(iy);                             // saturating: wild coordinates end up far outside
  const float fx = (float)x0, fy = (float)y0;
  const float ax = ix - fx, ay = iy - fy, bxw = (fx + 1.f) - ix, byw = (fy + 1.f) - iy;
  wnw = bxw * byw; wne = ax * byw; wsw = bxw * ay; wse = ax * ay;
}

// One pixel gathered from global memory (pixels whose taps fall outside the staged window).  Same accumulation order as the staged path.
template <int IN_U8, int C>
__device__ __forceinline__ void gather_px(const void* __restrict__ photo_, int b, int H, int W, int x0, int y0, float wnw, float wne,
                                          float wsw, float wse, float (&res)[C]) {
  const long long plane = (long long)H * W;
  if (((unsigned)x0 < (unsigned)(W - 1)) & ((unsigned)y0 < (unsigned)(H - 1))) {
    // all four taps inside the photo: one base address, no predicates
    if (IN_U8) {
      const uint8_t* q = (const uint8_t*)photo_ + ((size_t)b * plane + (size_t)y0 * W + x0) * C;
      const uint8_t* q1 = q + (size_t)W * C;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        float v = (float)__ldg(q + c) * wnw;
        v += (float)__ldg(q + C + c) * wne;
        v += (float)__ldg(q1 + c) * wsw;
        v += (float)__ldg(q1 + C + c) * wse;
        res[c] = v;
      }
    } else {
      const float* q = (const float*)photo_ + (size_t)b * C * plane + (size_t)y0 * W + x0;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float* a = q + (size_t)c * plane;
        float v = __ldg(a) * wnw;
        v += __ldg(a + 1) * wne;
        v += __ldg(a + W) * wsw;
        v += __ldg(a + W + 1) * wse;
        res[c] = v;
      }
    }
    return;
  }
  // per-tap validity (zeros padding) tested before any address is formed
  const bool vx0 = x0 >= 0 && x0 < W, vx1 = x0 >= -1 && x0 < W - 1;
  const bool vy0 = y0 >= 0 && y0 < H, vy1 = y0 >= -1 && y0 < H - 1;
  const bool any = (vx0 | vx1) && (vy0 | vy1);      // a pixel with no valid tap is exactly 0 even when its (wild) weights are inf / nan
#pragma unroll
  for (int c = 0; c < C; ++c) {
    float v = 0.f;
    if (IN_U8) {
      const uint8_t* base = (const uint8_t*)photo_ + (size_t)b * plane * C + c;
      v = (vy0 && vx0 ? (float)__ldg(base + ((long long)y0 * W + x0) * C) : 0.f) * wnw;
      v += (vy0 && vx1 ? (float)__ldg(base + ((long long)y0 * W + x0 + 1) * C) : 0.f) * wne;
      v += (vy1 && vx0 ? (float)__ldg(base + ((long long)(y0 + 1) * W + x0) * C) : 0.f) * wsw;
      v += (vy1 && vx1 ? (float)__ldg(base + ((long long)(y0 + 1) * W + x0 + 1) * C) : 0.f) * wse;
    } else {
      const float* base = (const float*)photo_ + ((size_t)b * C + c) * plane;
      v = (vy0 && vx0 ? __ldg(base + (long long)y0 * W + x0) : 0.f) * wnw;
      v += (vy0 && vx1 ? __ldg(base + (long long)y0 * W + x0 + 1) : 0.f) * wne;
      v += (vy1 && vx0 ? __ldg(base + (long long)(y0 + 1) * W + x0) : 0.f) * wsw;
      v += (vy1 && vx1 ? __ldg(base + (long long)(y0 + 1) * W + x0 + 1) : 0.f) * wse;
    }
    res[c] = any ? v : 0.f;
  }
}

// The four coarse-map values behind one entry (tile row rr8, window column kk) of a tile's blended map window + the vertical weight.
__device__ __forceinline__ void prefetch_map(const UnwarpGeom& g, const float* __restrict__ map, int b, int tyi, int txi, int kk, int rr8,
                                             float& m00, float& m10, float& m01, float& m11, float& l1) {
  const int wx0 = (int)(g.sx * (float)min(txi * T2, g.W - 1));       // first coarse-map column of the tile (= up_coeff's x0 of column jt0)
  int y0, yp; float l0;
  up_coeff(g.sy, min(tyi * T2 + rr8, g.H - 1), g.mh, y0, yp, l0, l1);
  // the column index is clamped to mw-1, which reproduces torch's "ip = 0" at the last map column (tap k+1 then equals tap k)
  const int mp = g.mh * g.mw, dy = yp * g.mw;
  const float* m = map + (size_t)b * 2 * mp + (size_t)y0 * g.mw + min(wx0 + kk, g.mw - 1);
  m00 = __ldg(m); m10 = __ldg(m + dy); m01 = __ldg(m + mp); m11 = __ldg(m + mp + dy);
}

template <int IN_U8, int OUT_U8, int C, int NS, int MINB>
__global__ void __launch_bounds__(UW_THREADS, MINB) k_unwarp_tma(const __grid_constant__ CUtensorMap tm_in, const __grid_constant__ CUtensorMap tm_out,
                                                           const void* __restrict__ photo_, const float* __restrict__ map,
                                                           void* __restrict__ out_, UnwarpGeom g, int tiles_x, int tiles_y, int n_tiles) {
  constexpr int ROW = IN_U8 ? SB_ROW_U8 : SB_ROW_F32;                                   // inner elements per staged row
  constexpr int ESZ = IN_U8 ? 1 : 4;
  constexpr int NPL = IN_U8 ? 1 : C;                                                    // planes per window
  constexpr int SRC_BYTES = NPL * SB_ROWS * ROW * ESZ;                                  // multiple of 128
  constexpr int STAGE_BYTES = SRC_BYTES;
  static_assert(SRC_BYTES % 128 == 0 && sizeof(TileTab) % 128 == 0, "smem carve-up must keep 128-byte alignment");
  extern __shared__ __align__(128) uint8_t s_dyn[];         // NS x source window | 2 x tables | output tile
  __shared__ __align__(8) uint64_t s_full[NS], s_empty[NS], s_out_full, s_out_empty;
  __shared__ int4 s_win[NS];                                // staged window of a stage: {first inner element, first row, rows, -}
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int W = g.W, H = g.H;
  if (threadIdx.x == 0) {
    for (int s = 0; s < NS; ++s) { tc::mbar_init(&s_full[s], 1); tc::mbar_init(&s_empty[s], 8); }
    tc::mbar_init(&s_out_full, 8); tc::mbar_init(&s_out_empty, 1);
    tc::fence_barrier_init();
  }
  __syncthreads();
  const float fw = (float)(W - 1), fh = (float)(H - 1);
  const int tiles_per_img = tiles_x * tiles_y;

  if (warp == 8) {
    // ================================================================ producer warp
    int n = 0;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++n) {
      const int s = n % NS, ph = (n / NS) & 1;
      const int b = t / tiles_per_img, rem = t - b * tiles_per_img;
      const int tyi = rem / tiles_x, txi = rem - tyi * tiles_x;
      const int jt0 = txi * T2, it0 = tyi * T2;
      const float* __restrict__ mapb = map + (size_t)b * 2 * g.mh * g.mw;
      // predicted window: tap origins on an 8 x 8 sample grid; pixels past a ragged edge repeat the edge pixel, as in the consumers
      int mnx = INT_MAX, mxx = INT_MIN, mny = INT_MAX, mxy = INT_MIN;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int cs = ((lane & 7) * 31 + 3) / 7, rs = (((lane >> 3) + 4 * h) * 31 + 3) / 7;     // {0,4,9,13,18,22,27,31}
        float gx, gy;
        sample_coords(g, mapb, min(it0 + rs, H - 1), min(jt0 + cs, W - 1), gx, gy);
        const int x0 = __float2int_rd(((gx + 1.f) / 2.f) * fw), y0 = __float2int_rd(((gy + 1.f) / 2.f) * fh);
        mnx = min(mnx, x0); mxx = max(mxx, x0); mny = min(mny, y0); mxy = max(mxy, y0);
      }
      mnx = __reduce_min_sync(0xffffffffu, mnx); mxx = __reduce_max_sync(0xffffffffu, mxx);
      mny = __reduce_min_sync(0xffffffffu, mny); mxy = __reduce_max_sync(0xffffffffu, mxy);
      // one pixel of margin; clamp (keeping the alignment) so that wild coordinates cannot produce absurd box coordinates
      const int inner_w = IN_U8 ? W * C : W;
      int xs = IN_U8 ? ((max(mnx, -(1 << 20)) - 1) * C) & ~15 : (max(mnx, -(1 << 20)) - 1) & ~3;
      xs = max(min(xs, inner_w & ~15), -ROW);
      const int wy0 = max(min(max(mny, -(1 << 20)) - 1, H), -SB_ROWS);
      const int need = min(mxy, 1 << 20) + 3 - wy0;                        // rows wy0 .. mxy + 2
      const int nq = max(1, min((need + 7) >> 3, SB_ROWS / 8));       // a window that is too small is still loaded: most of its pixels hit it
      tc::mbar_wait(&s_empty[s], ph ^ 1);
      if (lane == 0) {
        s_win[s] = make_int4(xs, wy0, 8 * nq, 0);
        tc::mbar_expect_tx(&s_full[s], (uint32_t)(nq * NPL * 8 * ROW * ESZ));     // release: s_win visible to the consumers
      }
      __syncwarp();
      if (lane < nq * NPL) {
        const int c = lane / nq, q = lane - c * nq;
        tc::tma_load_3d(s_dyn + (size_t)s * STAGE_BYTES + (size_t)((c * SB_ROWS + 8 * q) * ROW) * ESZ, &tm_in, &s_full[s], xs, wy0 + 8 * q,
                        IN_U8 ? b : b * C + c);
      }
    }
    return;
  }

  if (warp == 9) {
    // ================================================================ store warp: output tile -> global, one TMA store per tile
    if (lane == 0) {
      const uint8_t* const so = s_dyn + (size_t)NS * STAGE_BYTES + 2 * sizeof(TileTab);
      int n = 0;
      for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++n) {
        const int b = t / tiles_per_img, rem = t - b * tiles_per_img;
        const int tyi = rem / tiles_x, txi = rem - tyi * tiles_x;
        tc::mbar_wait(&s_out_full, n & 1);                    // all consumer warps have written (and proxy-fenced) the tile
        if (OUT_U8) tc::tma_store_3d(&tm_out, so, txi * T2 * C, tyi * T2, b);
        else        tc::tma_store_3d(&tm_out, so, txi * T2, tyi * T2, b * C);
        tc::tma_store_commit();
        tc::tma_store_wait_read_all();                        // the tile has been read: the consumers may overwrite it
        tc::mbar_arrive(&s_out_empty);
      }
      tc::tma_store_wait_all();
    }
    return;
  }

  // ================================================================== consumer warps
  TileTab* const tabs = reinterpret_cast<TileTab*>(s_dyn + (size_t)NS * STAGE_BYTES);        // double buffered
  uint8_t* const s_out = s_dyn + (size_t)NS * STAGE_BYTES + 2 * sizeof(TileTab);
  // tile walk without divisions inside the loop: tile t -> (b, tyi, txi); a step of gridDim.x tiles is (db, dty, dtx)
  int b = blockIdx.x / tiles_per_img, tyi = (blockIdx.x - b * tiles_per_img) / tiles_x, txi = blockIdx.x - b * tiles_per_img - tyi * tiles_x;
  const int db = gridDim.x / tiles_per_img, dty = (gridDim.x - db * tiles_per_img) / tiles_x,
            dtx = gridDim.x - db * tiles_per_img - dty * tiles_x;
  // software-pipelined coarse-map fetch: the four map values behind this thread's entry (tile row tid/8, window column tid%8) of the
  // NEXT tile's blended window are loaded one tile ahead, so their L2 latency is off the critical path
  const int kk = threadIdx.x & (W8 - 1), rr8 = threadIdx.x >> 3;
  float pm0 = 0.f, pm1 = 0.f, pm2 = 0.f, pm3 = 0.f, pl1 = 0.f;
  if ((int)blockIdx.x < n_tiles) prefetch_map(g, map, b, tyi, txi, kk, rr8, pm0, pm1, pm2, pm3, pl1);
  int n = 0;
  for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++n) {
    const int s = n % NS, ph = (n / NS) & 1;
    const uint8_t* const stage = s_dyn + (size_t)s * STAGE_BYTES;
    TileTab& tb = tabs[n & 1];
    const int jt0 = txi * T2, it0 = tyi * T2;
    // ---- tables of this tile.  Buffer n & 1 was last read for tile n-2, and every warp has passed the barrier of tile n-1 since.
    tb.sv[rr8][kk] = make_float2((1.0f - pl1) * pm0 + pl1 * pm1, (1.0f - pl1) * pm2 + pl1 * pm3);      // vertical blend
    if (warp == 0) {            // columns / rows past a ragged edge repeat the edge pixel (their results are clipped by the store)
      const int j = min(jt0 + lane, W - 1);
      int x0, xp; float l0, l1;
      up_coeff(g.sx, j, g.mw, x0, xp, l0, l1);
      tb.k[lane] = x0 - (int)(g.sx * (float)min(jt0, W - 1)); tb.lx[lane] = l1; tb.bx[lane] = base_ramp(g.bx, j);
    } else if (warp == 1) {
      tb.by[lane] = base_ramp(g.by, min(it0 + lane, H - 1));
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    // next tile of this CTA
    const int cb = b;
    txi += dtx; if (txi >= tiles_x) { txi -= tiles_x; ++tyi; }
    tyi += dty; if (tyi >= tiles_y) { tyi -= tiles_y; ++b; }
    b += db;
    if (t + (int)gridDim.x < n_tiles) prefetch_map(g, map, b, tyi, txi, kk, rr8, pm0, pm1, pm2, pm3, pl1);
    const int k = tb.k[lane];
    const float lx1 = tb.lx[lane], lx0 = 1.0f - lx1, bxv = tb.bx[lane];
    tc::mbar_wait(&s_full[s], ph);                            // the window of this tile has landed
    const int4 win = s_win[s];
    const int xs = win.x, wy0 = win.y, nrows = win.z;
    tc::mbar_wait(&s_out_empty, (n & 1) ^ 1);                 // the store of the previous tile has read the output buffer
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      int x0, y0; float wnw, wne, wsw, wse;
      tap_setup(tb, k, lx0, lx1, bxv, warp + 8 * p, g.affine, fw, fh, x0, y0, wnw, wne, wsw, wse);
      // all four taps inside the staged window?  (inner elements [xs, xs+ROW), rows [wy0, wy0+nrows))
      const unsigned ux = (IN_U8 ? (unsigned)x0 * (unsigned)C : (unsigned)x0) - (unsigned)xs, uy = (unsigned)y0 - (unsigned)wy0;
      const bool in = (ux <= (unsigned)(ROW - (IN_U8 ? 2 * C : 2))) & (uy < (unsigned)max(nrows - 1, 0)) &
                      (!IN_U8 || (x0 > -(1 << 20) && x0 < (1 << 20)));               // x0 * C must not have wrapped
      float res[C];
      if (__all_sync(0xffffffffu, in) || in) {
        if (IN_U8) {
          const uint8_t* q = stage + (uy * ROW + ux);
#pragma unroll
          for (int c = 0; c < C; ++c) {
            float v = (float)q[c] * wnw;
            v += (float)q[C + c] * wne;
            v += (float)q[ROW + c] * wsw;
            v += (float)q[ROW + C + c] * wse;
            res[c] = v;
          }
        } else {
          const float* q = reinterpret_cast<const float*>(stage) + (uy * ROW + ux);
#pragma unroll
          for (int c = 0; c < C; ++c) {
            float v = q[c * SB_ROWS * ROW] * wnw;
            v += q[c * SB_ROWS * ROW + 1] * wne;
            v += q[c * SB_ROWS * ROW + ROW] * wsw;
            v += q[c * SB_ROWS * ROW + ROW + 1] * wse;
            res[c] = v;
          }
        }
      } else {
        gather_px<IN_U8, C>(photo_, cb, H, W, x0, y0, wnw, wne, wsw, wse, res);
      }
      if (OUT_U8) {
        uint8_t* o = s_out + ((warp + 8 * p) * T2 + lane) * C;
#pragma unroll
        for (int c = 0; c < C; ++c) o[c] = to_u8_trunc(res[c]);
      } else {
        float* o = reinterpret_cast<float*>(s_out) + (warp + 8 * p) * T2 + lane;
#pragma unroll
        for (int c = 0; c < C; ++c) o[c * T2 * T2] = res[c];
      }
    }
    tc::fence_proxy_async();                                  // generic-proxy writes of the tile -> visible to the TMA store
    __syncwarp();
    if (lane == 0) {
      tc::mbar_arrive(&s_empty[s]);                           // this warp is done with the window
      tc::mbar_arrive(&s_out_full);                           // ... and has written its rows of the output tile
    }
  }
}


__global__ void k_fullres_grid(const float* __restrict__ map, float* __restrict__ grid, UnwarpGeom g) {
  int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y, b = blockIdx.z;
  if (j >= g.W) return;
  float gx, gy;
  sample_coords(g, map + (size_t)b * 2 * g.mh * g.mw, i, j, gx, gy);
  size_t plane = (size_t)g.H * g.W;
  grid[((size_t)b * 2 + 0) * plane + (size_t)i * g.W + j] = gx;
  grid[((size_t)b * 2 + 1) * plane + (size_t)i * g.W + j] = gy;
}

// generic grid_sample (WP:73): img [B,C,H,W], grid [B,2,Ho,Wo]
__global__ void k_grid_sample(const float* __restrict__ img, const float* __restrict__ grid, float* __restrict__ out,
                              int C, int H, int W, int Ho, int Wo) {
  int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y, b = blockIdx.z;
  if (j >= Wo) return;
  size_t po = (size_t)Ho * Wo, pi = (size_t)H * W;
  float gx = __ldg(grid + ((size_t)b * 2 + 0) * po + (size_t)i * Wo + j);
  float gy = __ldg(grid + ((size_t)b * 2 + 1) * po + (size_t)i * Wo + j);
  Taps t = make_taps(gx, gy, H, W);
  for (int c = 0; c < C; ++c)
    out[((size_t)b * C + c) * po + (size_t)i * Wo + j] = gather(img + ((size_t)b * C + c) * pi, t, W, 1);
}

template <int IN_U8, int OUT_U8>
static int launch_unwarp(const void* photo, const float* map, void* out, int B, int C, int H, int W, int mh, int mw,
                         float affine, cudaStream_t st) {
  DVD_REQUIRE(B >= 0 && H >= 0 && W >= 0 && mh >= 1 && mw >= 1 && C >= 1 && C <= 4, "unwarp: bad shape B=%d C=%d H=%d W=%d", B, C, H, W);
  if (B == 0 || H == 0 || W == 0) return 0;          // empty batch / empty photo: nothing to do
  DVD_REQUIRE(photo && map && out, "unwarp: null pointer");
  DVD_REQUIRE(B <= 65535 && cdiv(H, TILE_H) <= 65535, "unwarp: grid too large");
  DVD_REQUIRE((long long)H * W * C < (1ll << 31) && mh < 65536 && mw < 65536, "unwarp: image too large for 32-bit tap offsets");
  UnwarpGeom g = make_geom(H, W, mh, mw, affine);
  dim3 grid(cdiv(W, TILE_W), cdiv(H, TILE_H), B), block(32, 8);
  // map columns a 128-pixel tile can touch: floor(127 * sx) + 2 (+1 for the clamped last column)
  const bool fast = (int)(127.0f * g.sx) + 3 <= UW_WIN && W > 1 && H > 1;
  // TMA-staged kernel: 16-byte aligned rows and bases on both sides (W*4 or W*C bytes), <= 8 coarse-map columns per 32-pixel tile
  // uint8 HWC photos stay on the gather kernel by default: their taps are byte loads + conversions, the kernel is instruction bound
  // either way, and the gather kernel measured faster (23.5 vs 26.5 us at 1500x2000); DVD_UNWARP_TMA_U8=1 opts in.
  static const int no_tma = getenv("DVD_UNWARP_NO_TMA") ? atoi(getenv("DVD_UNWARP_NO_TMA")) : 0;
  static const int tma_u8 = getenv("DVD_UNWARP_TMA_U8") ? atoi(getenv("DVD_UNWARP_TMA_U8")) : 0;
  const size_t in_row = IN_U8 ? (size_t)W * C : (size_t)W * 4, out_row = OUT_U8 ? (size_t)W * C : (size_t)W * 4;
  const bool tma = !no_tma && (!IN_U8 || tma_u8) && C <= 3 && W >= 64 && H >= 8 && (int)(31.0f * g.sx) + 3 <= W8 && in_row % 16 == 0 && out_row % 16 == 0 &&
                   (reinterpret_cast<uintptr_t>(photo) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
                   (long long)B * cdiv(H, T2) * cdiv(W, T2) < (1ll << 31);
  if (tma) {
    CUtensorMap tm_in, tm_out;
    int rc = IN_U8 ? make_tmap_image3d(&tm_in, photo, 1, (uint64_t)W * C, H, B, SB_ROW_U8, 8, 1)
                   : make_tmap_image3d(&tm_in, photo, 4, W, H, (uint64_t)B * C, SB_ROW_F32, 8, 1);
    if (rc) return rc;
    rc = OUT_U8 ? make_tmap_image3d(&tm_out, out, 1, (uint64_t)W * C, H, B, T2 * C, T2, 1)
                : make_tmap_image3d(&tm_out, out, 4, W, H, (uint64_t)B * C, T2, T2, C);
    if (rc) return rc;
    const int tiles_x = cdiv(W, T2), tiles_y = cdiv(H, T2), n_tiles = B * tiles_x * tiles_y;
    constexpr int NS = IN_U8 ? 4 : 2;
    const size_t smem = (size_t)NS * (IN_U8 ? (size_t)SB_ROWS * SB_ROW_U8 : (size_t)C * SB_ROWS * SB_ROW_F32 * 4) + 2 * sizeof(TileTab) +
                        (size_t)T2 * T2 * C * (OUT_U8 ? 1 : 4);
    static int n_sm = 0;
    if (!n_sm) { int dev = 0; DVD_CUDA(cudaGetDevice(&dev)); DVD_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev)); }
    static const int minb = getenv("DVD_UNWARP_MINB") ? atoi(getenv("DVD_UNWARP_MINB")) : 3;
#define DVD_UNWARP_TMA(CC, MB)                                                                                                     \
  do {                                                                                                                             \
    auto kfn = k_unwarp_tma<IN_U8, OUT_U8, CC, NS, MB>;                                                                            \
    static int per_sm = 0;                                                                                                         \
    if (!per_sm) {                                                                                                                 \
      DVD_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                                 \
      DVD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kfn, UW_THREADS, smem));                                     \
      DVD_REQUIRE(per_sm >= 1, "unwarp: kernel does not fit an SM (smem %zu)", smem);                                              \
    }                                                                                                                              \
    const int ctas = std::min(n_tiles, n_sm * per_sm);                                                                             \
    kfn<<<ctas, UW_THREADS, smem, st>>>(tm_in, tm_out, photo, map, out, g, tiles_x, tiles_y, n_tiles);                             \
  } while (0)
    if (C == 1) DVD_UNWARP_TMA(1, 4);
    else if (C == 2) DVD_UNWARP_TMA(2, 4);
    else if (minb == 3) DVD_UNWARP_TMA(3, 3);
    else if (minb == 5) DVD_UNWARP_TMA(3, 5);
    else DVD_UNWARP_TMA(3, 4);
#undef DVD_UNWARP_TMA
  } else if (fast) {
    switch (C) {
      case 1: k_unwarp_fast<IN_U8, OUT_U8, 1><<<grid, block, 0, st>>>(photo, map, out, g); break;
      case 2: k_unwarp_fast<IN_U8, OUT_U8, 2><<<grid, block, 0, st>>>(photo, map, out, g); break;
      case 3: k_unwarp_fast<IN_U8, OUT_U8, 3><<<grid, block, 0, st>>>(photo, map, out, g); break;
      default: k_unwarp_fast<IN_U8, OUT_U8, 4><<<grid, block, 0, st>>>(photo, map, out, g); break;
    }
  } else {
    switch (C) {
      case 1: k_unwarp<IN_U8, OUT_U8, 1><<<grid, block, 0, st>>>(photo, map, out, g); break;
      case 2: k_unwarp<IN_U8, OUT_U8, 2><<<grid, block, 0, st>>>(photo, map, out, g); break;
      case 3: k_unwarp<IN_U8, OUT_U8, 3><<<grid, block, 0, st>>>(photo, map, out, g); break;
      default: k_unwarp<IN_U8, OUT_U8, 4><<<grid, block, 0, st>>>(photo, map, out, g); break;
    }
  }
  DVD_LAUNCH_CHECK("k_unwarp");
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// Mixed-size batch (uint8 HWC): one persistent launch walks the 128 x 8 tiles of documents of different sizes.  The caller plans a
// table on the host (dvd_unwarp_u8_plan) and uploads it; the grid depends only on the device, so a CUDA graph captured once
// serves every batch composition planned into the same device table.
struct MixedTableHeader {
  int32_t n_docs, total_tiles, C, pad;
};
struct MixedDoc {                         // 64 bytes
  const uint8_t* photo;
  uint8_t* out;
  UnwarpGeom g;                           // make_geom(): the same coefficients as the fixed-size launch
  int32_t tiles_x, tile_begin, fast;      // tile_begin: prefix sum of cdiv(W, 128) * cdiv(H, 8)
};
static_assert(sizeof(MixedTableHeader) == 16 && sizeof(MixedDoc) == 64, "mixed unwarp table layout");
constexpr int MIXED_MAX_TILES = 1 << 30;  // tile indices and t + gridDim.x stay inside int32

template <int C>
__global__ void __launch_bounds__(256) k_unwarp_u8_mixed(const MixedTableHeader* __restrict__ hdr, const MixedDoc* __restrict__ docs,
                                                         const float* __restrict__ map) {
  const int n_docs = __ldg(&hdr->n_docs), total = __ldg(&hdr->total_tiles);
  if (__ldg(&hdr->C) != C) return;        // planned for another channel count: write nothing (uniform over the grid)
  for (int t = blockIdx.x; t < total; t += gridDim.x) {
    // the document of tile t: the last one whose tile_begin <= t (empty documents own no tile and are never selected)
    int lo = 0, hi = n_docs - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (__ldg(&docs[mid].tile_begin) <= t) lo = mid; else hi = mid - 1;
    }
    const MixedDoc& d = docs[lo];
    const UnwarpGeom g = d.g;
    const int r = t - d.tile_begin, ty = r / d.tiles_x, tx = r - ty * d.tiles_x;
    const float* mapb = map + (size_t)lo * 2 * g.mh * g.mw;          // document d reads map row d
    __syncthreads();                      // the previous tile's threads are done reading the shared tables the prologue rewrites
    if (d.fast) unwarp_tile_fast<1, 1, C>(d.photo, mapb, d.out, g, tx, ty, 0, g.H, g.W);
    else        unwarp_tile<1, 1, C>(d.photo, mapb, d.out, g, tx, ty, 0, g.H, g.W);
  }
}

static size_t mixed_table_bytes(int max_docs) {
  return max_docs < 0 ? 0 : sizeof(MixedTableHeader) + (size_t)max_docs * sizeof(MixedDoc);
}

static int plan_mixed(const dvd_unwarp_doc_t* docs_host, int n_docs, int C, int mh, int mw, float affine, void* table_host,
                      size_t table_bytes, long long* total_tiles) {
  DVD_REQUIRE(n_docs >= 0 && (n_docs == 0 || docs_host) && table_host, "unwarp_u8_plan: n_docs=%d, docs %p, table %p", n_docs,
              (const void*)docs_host, table_host);
  DVD_REQUIRE(table_bytes >= mixed_table_bytes(n_docs), "unwarp_u8_plan: table of %zu bytes is too small for %d documents (%zu needed)",
              table_bytes, n_docs, mixed_table_bytes(n_docs));
  DVD_REQUIRE(C >= 1 && C <= 4, "unwarp_u8_plan: C=%d outside 1..4", C);
  DVD_REQUIRE(mh >= 1 && mw >= 1 && mh < 65536 && mw < 65536, "unwarp_u8_plan: bad map size %dx%d", mh, mw);
  MixedTableHeader* hdr = static_cast<MixedTableHeader*>(table_host);
  MixedDoc* recs = reinterpret_cast<MixedDoc*>(hdr + 1);
  long long tiles = 0;
  for (int d = 0; d < n_docs; ++d) {
    const dvd_unwarp_doc_t& in = docs_host[d];
    DVD_REQUIRE(in.H >= 0 && in.W >= 0, "unwarp_u8_plan: document %d has a negative size %dx%d", d, in.H, in.W);
    DVD_REQUIRE((long long)in.H * in.W * C < (1ll << 31), "unwarp_u8_plan: document %d (%dx%dx%d) is too large for 32-bit offsets", d,
                in.H, in.W, C);
    const bool empty = in.H == 0 || in.W == 0;
    DVD_REQUIRE(empty || (in.photo && in.out), "unwarp_u8_plan: document %d has a null photo or output pointer", d);
    MixedDoc r;
    r.photo = in.photo; r.out = in.out;
    r.g = make_geom(in.H, in.W, mh, mw, affine);
    r.tiles_x = empty ? 0 : cdiv(in.W, TILE_W);
    r.tile_begin = (int32_t)tiles;
    r.fast = (int)(127.0f * r.g.sx) + 3 <= UW_WIN && in.W > 1 && in.H > 1;     // the condition launch_unwarp uses
    tiles += empty ? 0 : (long long)r.tiles_x * cdiv(in.H, TILE_H);
    DVD_REQUIRE(tiles < MIXED_MAX_TILES, "unwarp_u8_plan: more than %d tiles in one batch", MIXED_MAX_TILES);
    recs[d] = r;
  }
  *hdr = MixedTableHeader{n_docs, (int32_t)tiles, C, 0};
  if (total_tiles) *total_tiles = tiles;
  return 0;
}

static int launch_unwarp_u8_mixed(const void* table, int C, const float* map, cudaStream_t st) {
  DVD_REQUIRE(table && map, "unwarp_u8_mixed: null pointer");
  DVD_REQUIRE(C >= 1 && C <= 4, "unwarp_u8_mixed: C=%d outside 1..4", C);
  const MixedTableHeader* hdr = static_cast<const MixedTableHeader*>(table);
  const MixedDoc* docs = reinterpret_cast<const MixedDoc*>(hdr + 1);
  int dev = 0, n_sm = 0;
  DVD_CUDA(cudaGetDevice(&dev));
  DVD_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  DVD_REQUIRE(dev < 64, "unwarp_u8_mixed: device %d", dev);
#define DVD_UNWARP_MIXED(CC)                                                                                                       \
  do {                                                                                                                             \
    static int per_sm[64] = {};                   /* per device: occupancy of this instantiation */                                \
    if (!per_sm[dev]) {                                                                                                            \
      DVD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[dev], k_unwarp_u8_mixed<CC>, 256, 0));                        \
      DVD_REQUIRE(per_sm[dev] >= 1, "unwarp_u8_mixed: kernel does not fit an SM");                                                 \
    }                                                                                                                              \
    k_unwarp_u8_mixed<CC><<<n_sm * per_sm[dev], dim3(32, 8), 0, st>>>(hdr, docs, map);                                             \
  } while (0)
  switch (C) {
    case 1: DVD_UNWARP_MIXED(1); break;
    case 2: DVD_UNWARP_MIXED(2); break;
    case 3: DVD_UNWARP_MIXED(3); break;
    default: DVD_UNWARP_MIXED(4); break;
  }
#undef DVD_UNWARP_MIXED
  DVD_LAUNCH_CHECK("k_unwarp_u8_mixed");
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// Sized batch (uint8 HWC): document d dewarps its Hi x Wi photo into an Ho x Wo output.  With supersampling factor s, output pixel
// (i, j) is the mean of the s x s block (s*i + a, s*j + b) of the reference chain evaluated on the VIRTUAL s*Ho x s*Wo grid:
//   out = trunc(avg_pool2d(grid_sample(photo, fullres_grid(map[d], s*Ho, s*Wo)), s))
// s = 1 documents run the fixed-size bodies on their output geometry (fast body under the same window rule as plan_mixed), so a
// same-size s = 1 document is dvd_unwarp_u8 byte for byte.  s > 1 documents run unwarp_tile_ss.  The table design (host plan,
// device table, grid independent of the table) is the mixed-size batch's; a separate kernel keeps k_unwarp_u8_mixed's registers.
struct SizedDoc {                         // 88 bytes
  const uint8_t* photo;
  uint8_t* out;
  UnwarpGeom g;                           // s = 1: make_geom(Ho, Wo); s > 1: make_geom(s*Ho, s*Wo), the virtual grid
  int32_t Hi, Wi, Ho, Wo;                 // photo, output
  int32_t s, win;                         // supersampling factor; win: fast body (s = 1) / pre-blended map window (s > 1)
  int32_t tiles_x, tile_begin;            // tile_begin: prefix sum of the tiles of the documents before
};
static_assert(sizeof(SizedDoc) == 88, "sized unwarp table layout");
constexpr int SS_TW = 32, SS_TH = 8, SS_MAX = 8;   // output tile of the supersampling body (one pixel per thread); largest factor

// One 32 x 8 output tile of an s > 1 document: thread (x, y) owns output pixel (ty*8 + y, tx*32 + x) and accumulates its s*s
// subsamples a-major, b-minor, in fp32; the mean is truncated like .astype(uint8).  Each subsample runs the coordinate chain of an
// s = 1 pixel of the virtual grid from per-tile column / row tables (8*s rows, 32*s columns); the coarse map is blended
// vertically once per virtual row when the tile touches at most UW_WIN map columns (fast body's order), else it is read per
// subsample in the general body's order.
// One thread per output pixel rather than one lane per subsample column + a shuffle reduction over groups of s lanes: the
// reduction would idle 32 mod s lanes for s in {3,5,6,7} and sum in a tree order, while here every lane is busy for every s, the
// order is a plain sequential sum, and the s-pixel stride between neighbouring lanes' taps costs more L1 wavefronts per load, not
// more bytes: the b loop re-reads the same lines from L1 a few instructions later.
template <int C>
__device__ __forceinline__ void unwarp_tile_ss(const uint8_t* __restrict__ photo, const float* __restrict__ map, uint8_t* __restrict__ out,
                                               const UnwarpGeom& g, int s, bool win, int Ho, int Wo, int Hi, int Wi, unsigned tx,
                                               unsigned ty) {
  __shared__ float s_bx[SS_TW * SS_MAX], s_lx[SS_TW * SS_MAX], s_by[SS_TH * SS_MAX], s_ly[SS_TH * SS_MAX];
  __shared__ int s_kx[SS_TW * SS_MAX], s_y0[SS_TH * SS_MAX];
  __shared__ float s_v[2][SS_TH * SS_MAX][UW_WIN];
  const int tid = threadIdx.y * 32 + threadIdx.x;
  const int vw = SS_TW * s, vh = SS_TH * s;               // virtual columns / rows of the tile
  const int jt0 = tx * vw, it0 = ty * vh;
  int wx0 = 0;                                            // first map column of the window (0: absolute column indices)
  if (win) {
    int xp; float l0, l1;
    up_coeff(g.sx, min(jt0, g.W - 1), g.mw, wx0, xp, l0, l1);
  }
  for (int e = tid; e < vw + vh; e += SS_TW * SS_TH) {    // virtual columns / rows past the edge repeat the last one
    if (e < vw) {
      const int j = min(jt0 + e, g.W - 1);
      int x0, xp; float l0, l1;
      up_coeff(g.sx, j, g.mw, x0, xp, l0, l1);
      s_kx[e] = (x0 - wx0) | (xp << 16); s_lx[e] = l1; s_bx[e] = base_ramp(g.bx, j);
    } else {
      const int r = e - vw, i = min(it0 + r, g.H - 1);
      int y0, yp; float l0, l1;
      up_coeff(g.sy, i, g.mh, y0, yp, l0, l1);
      s_y0[r] = y0 | (yp << 16); s_ly[r] = l1; s_by[r] = base_ramp(g.by, i);
    }
  }
  __syncthreads();
  if (win) {                                              // vertical blend of the map window: [channel][virtual row][window column]
    for (int e = tid; e < 2 * vh * UW_WIN; e += SS_TW * SS_TH) {
      const int k = e % UW_WIN, r = (e / UW_WIN) % vh, ch = e / (UW_WIN * vh);
      const int col = min(wx0 + k, g.mw - 1);
      const int y0 = s_y0[r] & 0xffff, yp = s_y0[r] >> 16;
      const float l1 = s_ly[r], l0 = 1.0f - l1;
      const float* m = map + (size_t)ch * g.mh * g.mw + (size_t)y0 * g.mw + col;
      s_v[ch][r][k] = l0 * __ldg(m) + l1 * __ldg(m + yp * g.mw);
    }
  }
  __syncthreads();
  const int io = ty * SS_TH + threadIdx.y, jo = tx * SS_TW + threadIdx.x;
  if (io < Ho && jo < Wo) {
    const float fw = (float)(Wi - 1), fh = (float)(Hi - 1);
    const int mplane = g.mh * g.mw;
    float acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = 0.f;
#pragma unroll 1
    for (int a = 0; a < s; ++a) {
      const int rr = threadIdx.y * s + a;
      const int dy = (s_y0[rr] >> 16) * g.mw;
      const float ly1 = s_ly[rr], ly0 = 1.0f - ly1, byv = s_by[rr];
      const float* __restrict__ mrow = map + (s_y0[rr] & 0xffff) * g.mw;
#pragma unroll 1
      for (int b = 0; b < s; ++b) {
        const int cj = threadIdx.x * s + b;
        const int k = s_kx[cj] & 0xffff, xp = s_kx[cj] >> 16;
        const float lx1 = s_lx[cj], lx0 = 1.0f - lx1;
        float sx, sy;
        if (win) {
          sx = lx0 * s_v[0][rr][k] + lx1 * s_v[0][rr][k + xp];
          sy = lx0 * s_v[1][rr][k] + lx1 * s_v[1][rr][k + xp];
        } else {
          const float* m0 = mrow + k;
          const float* m1 = m0 + mplane;
          sx = ly0 * (lx0 * __ldg(m0) + lx1 * __ldg(m0 + xp)) + ly1 * (lx0 * __ldg(m0 + dy) + lx1 * __ldg(m0 + dy + xp));
          sy = ly0 * (lx0 * __ldg(m1) + lx1 * __ldg(m1 + xp)) + ly1 * (lx0 * __ldg(m1 + dy) + lx1 * __ldg(m1 + dy + xp));
        }
        const float gx = ((sx + s_bx[cj]) * 2.0f - 1.0f) * g.affine;
        const float gy = ((sy + byv) * 2.0f - 1.0f) * g.affine;
        const float ix = ((gx + 1.f) / 2.f) * fw, iy = ((gy + 1.f) / 2.f) * fh;      // grid_sampler_unnormalize, align_corners=True
        const int x0 = __float2int_rd(ix), y0 = __float2int_rd(iy);
        const float fx = (float)x0, fy = (float)y0;
        const float ax = ix - fx, ay = iy - fy, bxw = (fx + 1.f) - ix, byw = (fy + 1.f) - iy;
        const float wnw = bxw * byw, wne = ax * byw, wsw = bxw * ay, wse = ax * ay;
        if (((unsigned)x0 < (unsigned)(Wi - 1)) & ((unsigned)y0 < (unsigned)(Hi - 1))) {
          const uint8_t* q0 = photo + ((size_t)y0 * Wi + x0) * C;
          const uint8_t* q1 = q0 + (size_t)Wi * C;
#pragma unroll
          for (int c = 0; c < C; ++c) {
            float v = (float)__ldg(q0 + c) * wnw;
            v += (float)__ldg(q0 + C + c) * wne;
            v += (float)__ldg(q1 + c) * wsw;
            v += (float)__ldg(q1 + C + c) * wse;
            acc[c] += v;
          }
        } else {
          // per-tap validity (zeros padding); coordinates may be wild, so validity is tested before any address is formed
          const bool vx0 = x0 >= 0 && x0 < Wi, vx1 = x0 >= -1 && x0 < Wi - 1;
          const bool vy0 = y0 >= 0 && y0 < Hi, vy1 = y0 >= -1 && y0 < Hi - 1;
#pragma unroll
          for (int c = 0; c < C; ++c) {
            float v = 0.f;
            if (vy0 && vx0) v += (float)__ldg(photo + ((long long)y0 * Wi + x0) * C + c) * wnw;
            if (vy0 && vx1) v += (float)__ldg(photo + ((long long)y0 * Wi + x0 + 1) * C + c) * wne;
            if (vy1 && vx0) v += (float)__ldg(photo + ((long long)(y0 + 1) * Wi + x0) * C + c) * wsw;
            if (vy1 && vx1) v += (float)__ldg(photo + ((long long)(y0 + 1) * Wi + x0 + 1) * C + c) * wse;
            acc[c] += v;
          }
        }
      }
    }
    const float n = (float)(s * s);
    uint8_t* o = out + ((size_t)io * Wo + jo) * C;
#pragma unroll
    for (int c = 0; c < C; ++c) o[c] = to_u8_trunc(acc[c] / n);
  }
}

// At least 3 CTAs per SM (80 registers) for C <= 3 and 2 for C = 4: the most that compile without spills (ptxas's own choice,
// 64 registers for C <= 3, spills a few bytes; 3 CTAs at C = 4 spill 8 bytes)
template <int C>
__global__ void __launch_bounds__(256, C < 4 ? 3 : 2) k_unwarp_u8_sized(const MixedTableHeader* __restrict__ hdr, const SizedDoc* __restrict__ docs,
                                                         const float* __restrict__ map) {
  const int n_docs = __ldg(&hdr->n_docs), total = __ldg(&hdr->total_tiles);
  if (__ldg(&hdr->C) != C) return;        // planned for another channel count: write nothing (uniform over the grid)
  for (int t = blockIdx.x; t < total; t += gridDim.x) {
    int lo = 0, hi = n_docs - 1;          // the document of tile t (see k_unwarp_u8_mixed)
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (__ldg(&docs[mid].tile_begin) <= t) lo = mid; else hi = mid - 1;
    }
    const SizedDoc& d = docs[lo];
    const UnwarpGeom g = d.g;
    const int r = t - d.tile_begin, ty = r / d.tiles_x, tx = r - ty * d.tiles_x;
    const float* mapb = map + (size_t)lo * 2 * g.mh * g.mw;
    __syncthreads();                      // the previous tile's threads are done reading the shared tables the prologue rewrites
    if (d.s > 1)    unwarp_tile_ss<C>(d.photo, mapb, d.out, g, d.s, d.win, d.Ho, d.Wo, d.Hi, d.Wi, tx, ty);
    else if (d.win) unwarp_tile_fast<1, 1, C>(d.photo, mapb, d.out, g, tx, ty, 0, d.Hi, d.Wi);
    else            unwarp_tile<1, 1, C>(d.photo, mapb, d.out, g, tx, ty, 0, d.Hi, d.Wi);
  }
}

static size_t sized_table_bytes(int max_docs) {
  return max_docs < 0 ? 0 : sizeof(MixedTableHeader) + (size_t)max_docs * sizeof(SizedDoc);
}

static int plan_sized(const dvd_unwarp_sized_doc_t* docs_host, int n_docs, int C, int mh, int mw, float affine, void* table_host,
                      size_t table_bytes, long long* total_tiles, int32_t* s_out) {
  DVD_REQUIRE(n_docs >= 0 && (n_docs == 0 || docs_host) && table_host, "unwarp_u8_sized_plan: n_docs=%d, docs %p, table %p", n_docs,
              (const void*)docs_host, table_host);
  DVD_REQUIRE(table_bytes >= sized_table_bytes(n_docs),
              "unwarp_u8_sized_plan: table of %zu bytes is too small for %d documents (%zu needed)", table_bytes, n_docs,
              sized_table_bytes(n_docs));
  DVD_REQUIRE(C >= 1 && C <= 4, "unwarp_u8_sized_plan: C=%d outside 1..4", C);
  DVD_REQUIRE(mh >= 1 && mw >= 1 && mh < 65536 && mw < 65536, "unwarp_u8_sized_plan: bad map size %dx%d", mh, mw);
  MixedTableHeader* hdr = static_cast<MixedTableHeader*>(table_host);
  SizedDoc* recs = reinterpret_cast<SizedDoc*>(hdr + 1);
  long long tiles = 0;
  for (int d = 0; d < n_docs; ++d) {
    const dvd_unwarp_sized_doc_t& in = docs_host[d];
    DVD_REQUIRE(in.H >= 0 && in.W >= 0 && in.Ho >= 0 && in.Wo >= 0,
                "unwarp_u8_sized_plan: document %d has a negative size (photo %dx%d, output %dx%d)", d, in.H, in.W, in.Ho, in.Wo);
    DVD_REQUIRE(in.supersample >= 0 && in.supersample <= 8, "unwarp_u8_sized_plan: document %d has supersample=%d outside 0..8", d,
                in.supersample);
    DVD_REQUIRE((long long)in.H * in.W * C < (1ll << 31), "unwarp_u8_sized_plan: document %d photo (%dx%dx%d) is too large for 32-bit offsets",
                d, in.H, in.W, C);
    DVD_REQUIRE((long long)in.Ho * in.Wo * C < (1ll << 31),
                "unwarp_u8_sized_plan: document %d output (%dx%dx%d) is too large for 32-bit offsets", d, in.Ho, in.Wo, C);
    const bool empty = in.H == 0 || in.W == 0 || in.Ho == 0 || in.Wo == 0;
    DVD_REQUIRE(empty || (in.photo && in.out), "unwarp_u8_sized_plan: document %d has a null photo or output pointer", d);
    int s = in.supersample;
    if (s == 0) s = empty ? 1 : std::min(8, std::max({1, cdiv(in.H, in.Ho), cdiv(in.W, in.Wo)}));
    DVD_REQUIRE((long long)s * in.Ho < (1ll << 31) && (long long)s * in.Wo < (1ll << 31),
                "unwarp_u8_sized_plan: document %d output %dx%d at supersample %d is too large for 32-bit coordinates", d, in.Ho, in.Wo, s);
    SizedDoc r;
    r.photo = in.photo; r.out = in.out;
    r.g = make_geom(s * in.Ho, s * in.Wo, mh, mw, affine);
    r.Hi = in.H; r.Wi = in.W; r.Ho = in.Ho; r.Wo = in.Wo; r.s = s;
    if (s == 1) {                         // the rule of launch_unwarp / plan_mixed, on the output geometry
      r.win = (int)(127.0f * r.g.sx) + 3 <= UW_WIN && in.Wo > 1 && in.Ho > 1;
      r.tiles_x = empty ? 0 : cdiv(in.Wo, TILE_W);
    } else {                              // map columns a 32*s-column virtual tile can touch
      r.win = (int)((float)(SS_TW * s - 1) * r.g.sx) + 3 <= UW_WIN;
      r.tiles_x = empty ? 0 : cdiv(in.Wo, SS_TW);
    }
    r.tile_begin = (int32_t)tiles;
    tiles += empty ? 0 : (long long)r.tiles_x * cdiv(in.Ho, s == 1 ? TILE_H : SS_TH);
    DVD_REQUIRE(tiles < MIXED_MAX_TILES, "unwarp_u8_sized_plan: more than %d tiles in one batch", MIXED_MAX_TILES);
    recs[d] = r;
    if (s_out) s_out[d] = s;
  }
  *hdr = MixedTableHeader{n_docs, (int32_t)tiles, C, 0};
  if (total_tiles) *total_tiles = tiles;
  return 0;
}

static int launch_unwarp_u8_sized(const void* table, int C, const float* map, cudaStream_t st) {
  DVD_REQUIRE(table && map, "unwarp_u8_sized: null pointer");
  DVD_REQUIRE(C >= 1 && C <= 4, "unwarp_u8_sized: C=%d outside 1..4", C);
  const MixedTableHeader* hdr = static_cast<const MixedTableHeader*>(table);
  const SizedDoc* docs = reinterpret_cast<const SizedDoc*>(hdr + 1);
  int dev = 0, n_sm = 0;
  DVD_CUDA(cudaGetDevice(&dev));
  DVD_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
  DVD_REQUIRE(dev < 64, "unwarp_u8_sized: device %d", dev);
#define DVD_UNWARP_SIZED(CC)                                                                                                       \
  do {                                                                                                                             \
    static int per_sm[64] = {};                   /* per device: occupancy of this instantiation */                                \
    if (!per_sm[dev]) {                                                                                                            \
      DVD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[dev], k_unwarp_u8_sized<CC>, 256, 0));                        \
      DVD_REQUIRE(per_sm[dev] >= 1, "unwarp_u8_sized: kernel does not fit an SM");                                                 \
    }                                                                                                                              \
    k_unwarp_u8_sized<CC><<<n_sm * per_sm[dev], dim3(32, 8), 0, st>>>(hdr, docs, map);                                             \
  } while (0)
  switch (C) {
    case 1: DVD_UNWARP_SIZED(1); break;
    case 2: DVD_UNWARP_SIZED(2); break;
    case 3: DVD_UNWARP_SIZED(3); break;
    default: DVD_UNWARP_SIZED(4); break;
  }
#undef DVD_UNWARP_SIZED
  DVD_LAUNCH_CHECK("k_unwarp_u8_sized");
  return 0;
}

}  // namespace dvd

using namespace dvd;

extern "C" int dvd_unwarp_f32(const float* photo, const float* map, float* out, int B, int C, int H, int W, int mh, int mw,
                              float affine, void* stream) {
  return launch_unwarp<0, 0>(photo, map, out, B, C, H, W, mh, mw, affine, (cudaStream_t)stream);
}
extern "C" int dvd_unwarp_u8(const uint8_t* photo, const float* map, uint8_t* out, int B, int C, int H, int W, int mh, int mw,
                             float affine, void* stream) {
  return launch_unwarp<1, 1>(photo, map, out, B, C, H, W, mh, mw, affine, (cudaStream_t)stream);
}
extern "C" int dvd_unwarp_f32_u8(const float* photo, const float* map, uint8_t* out, int B, int C, int H, int W, int mh, int mw,
                                 float affine, void* stream) {
  return launch_unwarp<0, 1>(photo, map, out, B, C, H, W, mh, mw, affine, (cudaStream_t)stream);
}
extern "C" size_t dvd_unwarp_table_bytes(int max_docs) { return mixed_table_bytes(max_docs); }
extern "C" int dvd_unwarp_u8_plan(const dvd_unwarp_doc_t* docs_host, int n_docs, int C, int mh, int mw, float affine, void* table_host,
                                  size_t table_bytes, long long* total_tiles) {
  return plan_mixed(docs_host, n_docs, C, mh, mw, affine, table_host, table_bytes, total_tiles);
}
extern "C" int dvd_unwarp_u8_mixed(const void* table, int C, const float* map, void* stream) {
  return launch_unwarp_u8_mixed(table, C, map, (cudaStream_t)stream);
}
extern "C" size_t dvd_unwarp_sized_table_bytes(int max_docs) { return sized_table_bytes(max_docs); }
extern "C" int dvd_unwarp_u8_sized_plan(const dvd_unwarp_sized_doc_t* docs_host, int n_docs, int C, int mh, int mw, float affine,
                                        void* table_host, size_t table_bytes, long long* total_tiles, int32_t* supersample_out) {
  return plan_sized(docs_host, n_docs, C, mh, mw, affine, table_host, table_bytes, total_tiles, supersample_out);
}
extern "C" int dvd_unwarp_u8_sized(const void* table, int C, const float* map, void* stream) {
  return launch_unwarp_u8_sized(table, C, map, (cudaStream_t)stream);
}
extern "C" int dvd_fullres_grid_f32(const float* map, float* grid, int B, int H, int W, int mh, int mw, float affine,
                                    void* stream) {
  DVD_REQUIRE(map && grid, "fullres_grid: null pointer");
  if (B == 0 || H == 0 || W == 0) return 0;
  UnwarpGeom g = make_geom(H, W, mh, mw, affine);
  k_fullres_grid<<<dim3(cdiv(W, 256), H, B), 256, 0, (cudaStream_t)stream>>>(map, grid, g);
  DVD_LAUNCH_CHECK("k_fullres_grid");
  return 0;
}
extern "C" int dvd_grid_sample_f32(const float* img, const float* grid, float* out, int B, int C, int H, int W, int Ho, int Wo,
                                   void* stream) {
  DVD_REQUIRE(img && grid && out, "grid_sample: null pointer");
  if (B == 0 || C == 0 || Ho == 0 || Wo == 0) return 0;
  k_grid_sample<<<dim3(cdiv(Wo, 256), Ho, B), 256, 0, (cudaStream_t)stream>>>(img, grid, out, C, H, W, Ho, Wo);
  DVD_LAUNCH_CHECK("k_grid_sample");
  return 0;
}
