// Fused attention on tcgen05: O = softmax(scale * Q K^T) V for one (sample, head, 128-query tile) per CTA.
//
//   S = Q K^T  : UMMA M=128 (queries) x N=64 (keys) x K=d, accumulator in TMEM (two S buffers for d = 256, one for d = 64)
//   softmax    : 8 warps; TMEM lane == query row, and each row is shared by TWO threads (one per 32-key half, the two warps that
//                may access the same TMEM lane quarter): tcgen05.ld S, row max exchanged through smem + a 64-thread named barrier,
//                exp2 / partial sums in fp32, P (bf16) written to shared memory in the 128-byte-swizzled K-major layout
//   O += P V   : UMMA M=128 x N=d x K=64, accumulator resident in TMEM for the whole KV sweep; rescaled in place
//                (tcgen05.ld / tcgen05.st, each half-warp pair owns half of the d columns) only when a row maximum grows by more
//                than 2^8 (lazy rescale; exact after the final division by the row sum)
//   epilogue   : O / rowsum -> bf16 -> global
// All three operands are K-major: Q [T, d], K [T, d] and V^T [d, T] (the QKV GEMM epilogue writes V transposed), so the
// same SWIZZLE_128B TMA boxes + UMMA descriptors as the GEMM are used.  K and V^T have separate mbarrier rings (a K stage is
// released right after QK^T(t)).  Warp roles: 0 = TMA producer, 1 = MMA issuer, 2..9 = softmax / correction / epilogue.
// d in {64, 256}; T a multiple of 128.
#include "gemm_tc.cuh"
#include "tc_common.cuh"
#include "tc_epilogue.cuh"
#include <string.h>

namespace dvd {
using namespace tc;

constexpr int AQ = 128;      // queries per CTA
constexpr int AKV = 64;      // keys per pipeline step
constexpr int ATHREADS = 320;

template <int D>
struct AttnCfg {
  // d = 64 (DiT block): ONE S buffer, 128 TMEM columns and a 2-stage ring, so that three CTAs share an SM and the 384-CTA launches of
  // the DiT block fit one wave (444 slots) instead of 1.3 waves of two CTAs per SM; the co-resident CTAs overlap each other's softmax.
  // d = 256 (decoder): O alone needs 256 columns -> one CTA per SM, two S buffers so that QK^T(t+1) overlaps softmax(t).
  static constexpr int NSB = (D == 64) ? 1 : 2;
  static constexpr int STAGES = 2;
  static constexpr int Q_BYTES = AQ * D * 2;
  static constexpr int K_BYTES = AKV * D * 2, V_BYTES = D * AKV * 2;
  static constexpr int STAGE_BYTES = K_BYTES + V_BYTES;
  static constexpr int P_BYTES = AQ * AKV * 2;
  static constexpr int X_BYTES = 2 * 2 * AQ * 4;                // row-max / row-sum exchange: [parity][half][row]
  static constexpr int SMEM = Q_BYTES + STAGES * STAGE_BYTES + P_BYTES + X_BYTES + 1024 + 256;
  static constexpr int TMEM_COLS = (D == 64) ? 128 : 512;      // NSB x 64 (S) + D (O), rounded to a power of two
  static constexpr int O_COL = NSB * AKV;
  static_assert(SMEM <= 232448, "shared memory budget");
};

__device__ __forceinline__ void pair_barrier(int quarter) {      // the two warps that own one TMEM lane quarter
  asm volatile("bar.sync %0, 64;" ::"r"(quarter + 1) : "memory");
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Up to ACTX independent key/value contexts share one launch (the four cross-attention contexts of the DiT block use the same
// queries): blockIdx.z = ctx * nsamp + sample.  Each context has its own K / V^T tensor maps, kv_div and output base.
constexpr int ACTX = 4;
struct AttnCtx {
  CUtensorMap tmK[ACTX], tmVt[ACTX];
  __nv_bfloat16* out[ACTX];
  __nv_bfloat16* out_lo[ACTX];     // low halves of the split output pair (DVD_PREC_BF16X3), or null
  int kv_div[ACTX];
};

// F16: Q, K, V^T and P are IEEE fp16 instead of bf16 (DVD_PREC_BF16X3: 2^-12 operand rounding; measured on the oracle, fp16
// attention inside an otherwise split-precision model moves the final map by 1.4e-6, bf16 attention by 1.1e-5)
template <int D, bool F16>
__global__ void __launch_bounds__(ATHREADS, D == 64 ? 3 : 1) k_attn_tc(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ AttnCtx cx, int nsamp,
                                                      int ldo, int T, int heads, float scale_log2) {
  using Cfg = AttnCfg<D>;
  constexpr int ST = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sKV = sQ + Cfg::Q_BYTES;
  uint8_t* sP = sKV + ST * Cfg::STAGE_BYTES;
  float* sX = reinterpret_cast<float*>(sP + Cfg::P_BYTES);       // [2][2][128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + Cfg::P_BYTES + Cfg::X_BYTES);
  uint64_t* q_full = bars;                 // 1
  uint64_t* k_full = bars + 1;             // ST
  uint64_t* k_empty = k_full + ST;         // ST
  uint64_t* v_full = k_empty + ST;         // ST
  uint64_t* v_empty = v_full + ST;         // ST
  uint64_t* s_full = v_empty + ST;         // 2
  uint64_t* s_empty = s_full + 2;          // 2
  uint64_t* p_full = s_empty + 2;          // 1
  uint64_t* pv_done = p_full + 1;          // 1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pv_done + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ctx = blockIdx.z / nsamp;
  const int q0 = blockIdx.x * AQ, h = blockIdx.y, n = blockIdx.z - ctx * nsamp, nkv = n / cx.kv_div[ctx];
  const int nt = T / AKV;
  const CUtensorMap& tmK = cx.tmK[ctx];
  const CUtensorMap& tmVt = cx.tmVt[ctx];
  __nv_bfloat16* __restrict__ O = cx.out[ctx];
  __nv_bfloat16* __restrict__ Olo = cx.out_lo[ctx];

  pdl_trigger();
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmQ); prefetch_tmap(&tmK); prefetch_tmap(&tmVt);
    mbar_init(q_full, 1);
    for (int s = 0; s < ST; ++s) { mbar_init(&k_full[s], 1); mbar_init(&k_empty[s], 1); mbar_init(&v_full[s], 1); mbar_init(&v_empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&s_full[b], 1); mbar_init(&s_empty[b], 256); }
    mbar_init(p_full, 256);
    mbar_init(pv_done, 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer: Q once, then the K and V^T rings
      mbar_expect_tx(q_full, Cfg::Q_BYTES);
#pragma unroll
      for (int j = 0; j < D / 64; ++j) tma_load_2d(sQ + j * (AQ * 128), &tmQ, q_full, h * D + 64 * j, n * T + q0);
      for (int t = 0; t < nt; ++t) {
        const int s = t % ST, u = t / ST;
        uint8_t* k = sKV + s * Cfg::STAGE_BYTES;
        mbar_wait(&k_empty[s], (u & 1) ^ 1);
        mbar_expect_tx(&k_full[s], Cfg::K_BYTES);
#pragma unroll
        for (int j = 0; j < D / 64; ++j) tma_load_2d(k + j * (AKV * 128), &tmK, &k_full[s], h * D + 64 * j, nkv * T + t * AKV);
        mbar_wait(&v_empty[s], (u & 1) ^ 1);
        mbar_expect_tx(&v_full[s], Cfg::V_BYTES);
        tma_load_2d(k + Cfg::K_BYTES, &tmVt, &v_full[s], t * AKV, (nkv * heads + h) * D);      // box: 64 keys x D rows of V^T
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    {
      // ===== MMA issuer: the whole warp runs the loop, one elected lane issues (tc_common.cuh)
      constexpr uint32_t idesc_qk = F16 ? make_idesc_f16(AQ, AKV) : make_idesc_bf16(AQ, AKV);     // 128 x 64
      constexpr uint32_t idesc_pv = F16 ? make_idesc_f16(AQ, D) : make_idesc_bf16(AQ, D);         // 128 x D
      const uint32_t tbase = __shfl_sync(0xffffffffu, tmem_base, 0);                             // warp-uniform for the compiler
      const uint64_t q_desc = make_desc_k_sw128(smem_u32(sQ)), p_desc = make_desc_k_sw128(smem_u32(sP));
      auto issue_qk = [&](int t) {
        const int s = t % ST, b = t % Cfg::NSB;
        mbar_wait(&k_full[s], (t / ST) & 1);
        mbar_wait(&s_empty[b], ((t / Cfg::NSB) & 1) ^ 1);
        fence_after_sync();
        const uint64_t k_desc = make_desc_k_sw128(smem_u32(sKV + s * Cfg::STAGE_BYTES));
#pragma unroll
        for (int k = 0; k < D / 16; ++k)                          // descriptor start field: 16-byte units
          mma_ss_elect(tbase + b * AKV, q_desc + (uint64_t)(((k >> 2) * (AQ * 128) + (k & 3) * 32) >> 4),
                       k_desc + (uint64_t)(((k >> 2) * (AKV * 128) + (k & 3) * 32) >> 4), idesc_qk, k ? 1u : 0u);
        mma_commit_elect(&s_full[b]);
        mma_commit_elect(&k_empty[s]);                            // K stage free as soon as QK^T(t) has read it
      };
      mbar_wait(q_full, 0);
      issue_qk(0);
      for (int t = 0; t < nt; ++t) {
        if (t + 1 < nt) issue_qk(t + 1);                          // S(t+1) overlaps softmax(t)
        mbar_wait(&v_full[t % ST], (t / ST) & 1);
        mbar_wait(p_full, t & 1);
        fence_after_sync();
        const uint64_t v_desc = make_desc_k_sw128(smem_u32(sKV + (t % ST) * Cfg::STAGE_BYTES + Cfg::K_BYTES));
#pragma unroll
        for (int k = 0; k < AKV / 16; ++k)
          mma_ss_elect(tbase + Cfg::O_COL, p_desc + (uint64_t)(k * 2), v_desc + (uint64_t)(k * 2), idesc_pv, (t | k) ? 1u : 0u);
        mma_commit_elect(&v_empty[t % ST]);                       // V^T stage free
        mma_commit_elect(pv_done);                                // P buffer free, O(t) complete
      }
    }
    __syncwarp();
  } else {
    // ===== softmax / correction / epilogue: row = TMEM lane; two threads (halves) per row
    const int quarter = warp & 3;
    const int half = (warp - 2) >> 2;                             // warps 2..5 -> keys [0,32), warps 6..9 -> keys [32,64) of each tile
    const int row = quarter * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
    float m = -INFINITY, l = 0.f;                                 // m is identical in both halves; l is this half's partial sum
    for (int t = 0; t < nt; ++t) {
      const int b = t % Cfg::NSB;
      mbar_wait(&s_full[b], (t / Cfg::NSB) & 1);
      fence_after_sync();
      uint32_t s0[32];
      tmem_ld_32x32(lane_base + b * AKV + half * 32, s0);
      tmem_ld_wait();
      fence_before_sync();
      mbar_arrive(&s_empty[b]);                                   // this half of S(b) is in registers
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(s0[j]));
      float* xch = sX + (t & 1) * 256;                            // double-buffered by tile parity (see the race note in DESIGN.md)
      xch[half * 128 + row] = mx;
      pair_barrier(quarter);
      mx = fmaxf(mx, xch[(half ^ 1) * 128 + row]);
      const float m_new = fmaxf(m, mx * scale_log2);
      // lazy rescale: keep the stale maximum while exp2 stays below 2^8
      const bool grow = (m_new - m) > 8.0f;                       // also true for t == 0 (m = -inf)
      const float alpha = (grow && t > 0) ? ex2(m - m_new) : 1.0f;
      if (grow) m = m_new;
      float sum = 0.f;
      uint32_t pk[16];                                            // 32 16-bit probabilities
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        const float a0 = ex2(fmaf(__uint_as_float(s0[j]), scale_log2, -m)), a1 = ex2(fmaf(__uint_as_float(s0[j + 1]), scale_log2, -m));
        if (F16) {
          const __half2 pa = __floats2half2_rn(a0, a1);
          sum += __low2float(pa) + __high2float(pa);              // the sum uses the rounded values the tensor core multiplies with
          pk[j >> 1] = *reinterpret_cast<const uint32_t*>(&pa);
        } else {
          const __nv_bfloat162 pa = __floats2bfloat162_rn(a0, a1);
          sum += __low2float(pa) + __high2float(pa);
          pk[j >> 1] = *reinterpret_cast<const uint32_t*>(&pa);
        }
      }
      l = l * alpha + sum;
      if (t > 0) {
        mbar_wait(pv_done, (t - 1) & 1);                          // PV(t-1) finished: P buffer reusable, O readable
        fence_after_sync();
        if (__any_sync(0xffffffffu, alpha != 1.0f)) {             // identical decision in both warps of the pair
#pragma unroll 1
          for (int c = half * (D / 2); c < (half + 1) * (D / 2); c += 32) {
            uint32_t o[32];
            tmem_ld_32x32(lane_base + Cfg::O_COL + c, o);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) o[j] = __float_as_uint(__uint_as_float(o[j]) * alpha);
            tmem_st_32x32(lane_base + Cfg::O_COL + c, o);
          }
          tmem_st_wait();
        }
      }
      // P half-row -> smem, K-major SWIZZLE_128B: 16-byte chunk c of row r lives at r*128 + ((c ^ (r & 7)) << 4)
      uint8_t* prow = sP + row * 128;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const uint4 v = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
        *reinterpret_cast<uint4*>(prow + (((half * 4 + c) ^ (row & 7)) << 4)) = v;
      }
      fence_proxy_async();                                        // generic-proxy writes -> visible to the UMMA (async proxy)
      fence_before_sync();
      mbar_arrive(p_full);
    }
    // ---- epilogue: total row sum = both halves' partial sums; each half stores D/2 columns
    float* xch = sX + (nt & 1) * 256;
    xch[half * 128 + row] = l;
    pair_barrier(quarter);
    const float inv = 1.0f / (l + xch[(half ^ 1) * 128 + row]);
    mbar_wait(pv_done, (nt - 1) & 1);
    fence_after_sync();
    const size_t ooff = (size_t)(n * T + q0 + row) * ldo + h * D;
#pragma unroll 1
    for (int c = half * (D / 2); c < (half + 1) * (D / 2); c += 32) {
      uint32_t o[32];
      tmem_ld_32x32(lane_base + Cfg::O_COL + c, o);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; j += 8) {
        uint4 u, l;
        split_bf16x2(__uint_as_float(o[j]) * inv, __uint_as_float(o[j + 1]) * inv, u.x, l.x);
        split_bf16x2(__uint_as_float(o[j + 2]) * inv, __uint_as_float(o[j + 3]) * inv, u.y, l.y);
        split_bf16x2(__uint_as_float(o[j + 4]) * inv, __uint_as_float(o[j + 5]) * inv, u.z, l.z);
        split_bf16x2(__uint_as_float(o[j + 6]) * inv, __uint_as_float(o[j + 7]) * inv, u.w, l.w);
        *reinterpret_cast<uint4*>(O + ooff + c + j) = u;
        if (Olo) *reinterpret_cast<uint4*>(Olo + ooff + c + j) = l;
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// V [nsamp, T, C] (row stride ldv) -> V^T [nsamp, C, T]; only used by the test hook (the denoiser's GEMM epilogue writes V^T directly)
__global__ void k_transpose_v(const uint16_t* __restrict__ v, int ldv, uint16_t* __restrict__ vt, int T, int C) {
  __shared__ uint16_t tile[32][34];
  const int n = blockIdx.z, t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += 8) tile[r][threadIdx.x] = v[((size_t)n * T + t0 + r) * ldv + c0 + threadIdx.x];
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) vt[((size_t)n * C + c0 + r) * T + t0 + threadIdx.x] = tile[threadIdx.x][r];
}
int transpose_v16(const void* v, int ldv, void* vt, int nsamp, int T, int C, cudaStream_t st) {
  DVD_REQUIRE(v && vt && T % 32 == 0 && C % 32 == 0, "transpose_v: bad args");
  k_transpose_v<<<dim3(T / 32, C / 32, nsamp), dim3(32, 8), 0, st>>>((const uint16_t*)v, ldv, (uint16_t*)vt, T, C);
  DVD_LAUNCH_CHECK("k_transpose_v");
  return 0;
}

template <int D, bool F16>
static int launch_attention_t(const CUtensorMap& tmQ, const AttnCtx& cx, int nctx, int ldo, int nsamp, int heads, int T, float scale,
                              cudaStream_t st) {
  auto kern = k_attn_tc<D, F16>;
  DVD_SET_MAX_SMEM(kern, AttnCfg<D>::SMEM);
  const float scale_log2 = scale * 1.4426950408889634f;
  dim3 grid(T / AQ, heads, nsamp * nctx);
  DVD_CUDA(launch_pdl(2, kern, grid, dim3(ATHREADS), (size_t)AttnCfg<D>::SMEM, st, tmQ, cx, nsamp, ldo, T, heads, scale_log2));
  DVD_LAUNCH_CHECK("k_attn_tc");
  return 0;
}

// nctx (<= 4) key/value contexts attended by the SAME queries in one launch; k[i]/vt[i]/o[i]/kv_div[i] describe context i.
int attention_tc_multi(const void* q, int ldq, const void* const* k, int ldk, const void* const* vt, __nv_bfloat16* const* o,
                       __nv_bfloat16* const* o_lo, int ldo, const int* kv_div, int nctx, int nsamp, int heads, int T, int d, float scale,
                       int f16, cudaStream_t st) {
  DVD_REQUIRE(q && k && vt && o && kv_div && nctx >= 1 && nctx <= ACTX, "attention_tc_multi: bad arguments");
  DVD_REQUIRE((d == 64 || d == 256) && T % 128 == 0 && nsamp > 0, "attention_tc: bad shape d=%d T=%d", d, T);
  DVD_REQUIRE(ldo % 8 == 0, "attention_tc: ldo %d is not a multiple of 8", ldo);
  DVD_REQUIRE((long long)nsamp * nctx <= 65535, "attention_tc: nsamp %d x nctx %d exceeds 65535 grid slices", nsamp, nctx);
  // every argument is checked before the first tensor map is encoded (a driver call)
  for (int i = 0; i < nctx; ++i) {
    DVD_REQUIRE(k[i] && vt[i] && o[i], "attention_tc: context %d: null pointer", i);
    DVD_REQUIRE(kv_div[i] > 0 && nsamp % kv_div[i] == 0, "attention_tc: context %d: nsamp %d is not a multiple of kv_div %d", i, nsamp, kv_div[i]);
    DVD_REQUIRE((reinterpret_cast<uintptr_t>(o[i]) & 15) == 0, "attention_tc: context %d: o must be 16-byte aligned", i);
    DVD_REQUIRE(!o_lo || (reinterpret_cast<uintptr_t>(o_lo[i]) & 15) == 0, "attention_tc: context %d: o_lo must be 16-byte aligned", i);
  }
  CUtensorMap tmQ;
  AttnCtx cx;
  memset(&cx, 0, sizeof(cx));
  // (fp16 and bf16 tiles are both plain 16-bit elements for TMA)
  int rc = make_tmap_bf16_2d(&tmQ, q, (uint64_t)nsamp * T, (uint64_t)heads * d, (uint64_t)ldq, AQ, 64); if (rc) return rc;
  for (int i = 0; i < nctx; ++i) {
    const int nkv = nsamp / kv_div[i];
    rc = make_tmap_bf16_2d(&cx.tmK[i], k[i], (uint64_t)nkv * T, (uint64_t)heads * d, (uint64_t)ldk, AKV, 64); if (rc) return rc;
    rc = make_tmap_bf16_2d(&cx.tmVt[i], vt[i], (uint64_t)nkv * heads * d, (uint64_t)T, (uint64_t)T, d, 64); if (rc) return rc;
    cx.out[i] = o[i]; cx.kv_div[i] = kv_div[i];
    cx.out_lo[i] = o_lo ? o_lo[i] : nullptr;
  }
  if (d == 64) return f16 ? launch_attention_t<64, true>(tmQ, cx, nctx, ldo, nsamp, heads, T, scale, st)
                          : launch_attention_t<64, false>(tmQ, cx, nctx, ldo, nsamp, heads, T, scale, st);
  return f16 ? launch_attention_t<256, true>(tmQ, cx, nctx, ldo, nsamp, heads, T, scale, st)
             : launch_attention_t<256, false>(tmQ, cx, nctx, ldo, nsamp, heads, T, scale, st);
}

int attention_tc(const void* q, int ldq, const void* k, int ldk, const void* vt, __nv_bfloat16* o, __nv_bfloat16* o_lo, int ldo, int nsamp,
                 int heads, int T, int d, float scale, int kv_div, int f16, cudaStream_t st) {
  DVD_REQUIRE(q && k && vt && o, "attention_tc: null pointer");
  if (attention_pair_supported(T, d, 1)) return attention_pair(q, ldq, k, ldk, vt, o, o_lo, ldo, nsamp, heads, T, scale, kv_div, f16, st);
  __nv_bfloat16* const* olo = o_lo ? &o_lo : nullptr;
  return attention_tc_multi(q, ldq, &k, ldk, &vt, &o, olo, ldo, &kv_div, 1, nsamp, heads, T, d, scale, f16, st);
}

}  // namespace dvd
