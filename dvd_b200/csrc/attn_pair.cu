// Decoder attention (head dim 256) on a CTA pair: O = softmax(scale * Q K^T) V for 256 queries of one (sample, head) per cluster of 2.
//
// Why a second kernel: the single-CTA kernel (attn_tc.cu) steps over 64 keys, and its one MMA-issuing thread needs 16 UMMAs of
// 128 x 64 x 16 per step for Q K^T: each is worth ~40 tensor clocks but costs more than that to issue, and the 2 x 64 KB of K / V per
// 128 keys next to the resident 64 KB Q tile leave no room for wider steps.  As a pair (cta_group::2):
//   * S = Q K^T  : UMMA M = 256 (128 queries per CTA) x N = 128 keys x K = 16; each CTA stages HALF of the key tile (64 keys x 256)
//   * O += P V   : UMMA M = 256 x N = 256 (head dim) x K = 16 keys; each CTA stages half of V^T (128 dims x 128 keys);
//                  P is the A operand read from TENSOR MEMORY: the softmax warps write the 16-bit probabilities over the S columns
//                  they have just read (tcgen05.st), so there is no P tile in shared memory and no generic->async proxy fence
//   * per CTA: Q 64 KB + 2 x (K 32 KB + V^T 32 KB) = 192 KB; TMEM 2 x 128 (S / P ping-pong) + 256 (O) = 512 columns
//   * one thread (leader CTA) issues 24 UMMAs per 128 keys for BOTH CTAs instead of 2 x 40
// The S buffers need no "empty" barrier: the tensor pipe executes in issue order, Q K^T(t+2) is issued after P V(t), which read the
// P that aliases that buffer.  Softmax: row = TMEM lane, two threads per row (64 keys each), lazy rescale as in attn_tc.cu.
// Warp roles per CTA: 0 = Q / K producer, 1 = MMA issuer (leader only), 2..9 = softmax / correction / epilogue, 10 = V^T producer (K and
// V^T have separate producers: behind one thread the K(t+2) request queued behind the wait for P V(t)'s V^T stage, and the late K tile
// delayed Q K^T(t+2) by 0.6 us per step, measured with tools/attn_bench.py --trace).  The output leaves through a per-warp staging
// tile in the (then idle) Q / K shared memory so that every global store covers whole 256-byte row segments: one thread per row
// storing 16 bytes at a time took 8.5 us of a 24 us launch.
#include "gemm_tc.cuh"
#include "tc_common.cuh"
#include "tc_epilogue.cuh"
#include <string.h>
#include <stdlib.h>

namespace dvd {
using namespace tc;

namespace {
constexpr int PQ = 128;        // queries per CTA
constexpr int PKV = 128;       // keys per step
constexpr int PD = 256;        // head dim
constexpr int PTHREADS = 352;   // warp 0: Q / K producer, 1: MMA issuer, 2..9: softmax, 10: V^T producer
constexpr int PST = 2;         // K / V^T ring depth

struct APCfg {
  static constexpr int Q_BYTES = PQ * PD * 2;                   // 64 KB: [d / 64][128 rows][128 B]
  static constexpr int K_BYTES = (PKV / 2) * PD * 2;            // 32 KB: this CTA's 64 keys, [d / 64][64 rows][128 B]
  static constexpr int V_BYTES = (PD / 2) * PKV * 2;            // 32 KB: this CTA's 128 dims, [keys / 64][128 rows][128 B]
  static constexpr int X_BYTES = 2 * 2 * PQ * 4;                // row-max / row-sum exchange [parity][half][row]
  static constexpr int K_OFF = Q_BYTES, V_OFF = K_OFF + PST * K_BYTES, X_OFF = V_OFF + PST * V_BYTES, BAR_OFF = X_OFF + X_BYTES;
  static constexpr int SMEM = BAR_OFF + 256 + 1024;
  static constexpr int S_COLS = PKV, O_COL = 2 * PKV, TMEM_COLS = 512;
  static_assert(SMEM <= 232448, "shared memory budget");
};

__device__ __forceinline__ void pair_barrier64(int quarter) {      // the two warps that own one TMEM lane quarter
  asm volatile("bar.sync %0, 64;" ::"r"(quarter + 1) : "memory");
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
#ifdef DVD_ATTN_TRACE
__device__ unsigned long long g_attn_trace[16][16];
__device__ __forceinline__ unsigned long long atime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define ATRACE(t, slot) do { if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && (t) < 16) g_attn_trace[t][slot] = atime(); } while (0)
#else
#define ATRACE(t, slot) do { } while (0)
#endif
}  // namespace

template <bool F16>
__global__ void __launch_bounds__(PTHREADS, 1)
k_attn_pair(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmVt,
            __nv_bfloat16* __restrict__ O, __nv_bfloat16* __restrict__ Olo, int ldo, int T, int heads, int kv_div, float scale_log2) {
  using Cfg = APCfg;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  float* sX = reinterpret_cast<float*>(smem + Cfg::X_OFF);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::BAR_OFF);
  uint64_t* q_full = bars;                 // 1   (leader's is used)
  uint64_t* k_full = bars + 1;             // PST (leader's)
  uint64_t* v_full = k_full + PST;         // PST (leader's)
  uint64_t* k_empty = v_full + PST;        // PST (own, multicast commit)
  uint64_t* v_empty = k_empty + PST;       // PST (own)
  uint64_t* s_full = v_empty + PST;        // 2   (own)
  uint64_t* p_full = s_full + 2;           // 1   (leader's: 8 softmax warps of each CTA)
  uint64_t* pv_done = p_full + 1;          // 1   (own)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pv_done + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int q0 = blockIdx.x * PQ, h = blockIdx.y, n = blockIdx.z, nkv = n / kv_div;
  const int nt = T / PKV;

  pdl_trigger();
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmQ); prefetch_tmap(&tmK); prefetch_tmap(&tmVt);
    mbar_init(q_full, 1);
    for (int s = 0; s < PST; ++s) { mbar_init(&k_full[s], 1); mbar_init(&v_full[s], 1); mbar_init(&k_empty[s], 1); mbar_init(&v_empty[s], 1); }
    mbar_init(&s_full[0], 1); mbar_init(&s_full[1], 1);
    mbar_init(p_full, 16);
    mbar_init(pv_done, 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc2(tmem_slot, Cfg::TMEM_COLS);
  fence_before_sync();
  cluster_sync_all();                                              // both CTAs' barriers exist before any remote arrive / TMA
  fence_after_sync();
  // The allocation covers all 512 columns of this SM's tensor memory, so its base address is 0 by construction; using the constant
  // lets the compiler keep every UMMA operand in uniform registers (a tensor-memory address held in a vector register costs an
  // elect / broadcast loop per instruction: ~100 clocks of issue per UMMA, measured with tools/attn_bench.py --trace).
  if (*tmem_slot != 0u) __trap();
  constexpr uint32_t tmem_base = 0u;
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer (both CTAs): own queries, own half of every K / V^T tile; all bytes are counted on the LEADER's barriers
      const uint32_t lq = mapa(smem_u32(q_full), 0);
      if (rank == 0) mbar_expect_tx(q_full, 2 * Cfg::Q_BYTES);
#pragma unroll
      for (int j = 0; j < PD / 64; ++j) tma_load_2d_pair(sQ + j * (PQ * 128), &tmQ, lq, h * PD + 64 * j, n * T + q0);
      for (int t = 0; t < nt; ++t) {
        const int s = t % PST, u = t / PST;
        uint8_t* k = smem + Cfg::K_OFF + s * Cfg::K_BYTES;
        const uint32_t lk = mapa(smem_u32(&k_full[s]), 0);
        mbar_wait(&k_empty[s], (u & 1) ^ 1);
        if (rank == 0) mbar_expect_tx(&k_full[s], 2 * Cfg::K_BYTES);
#pragma unroll
        for (int j = 0; j < PD / 64; ++j)
          tma_load_2d_pair(k + j * ((PKV / 2) * 128), &tmK, lk, h * PD + 64 * j, nkv * T + t * PKV + (int)rank * (PKV / 2));
      }
    }
    __syncwarp();
  } else if (warp == 10) {
    if (lane == 0) {
      // ===== V^T producer (both CTAs)
      for (int t = 0; t < nt; ++t) {
        const int s = t % PST, u = t / PST;
        uint8_t* v = smem + Cfg::V_OFF + s * Cfg::V_BYTES;
        const uint32_t lv = mapa(smem_u32(&v_full[s]), 0);
        mbar_wait(&v_empty[s], (u & 1) ^ 1);
        if (rank == 0) mbar_expect_tx(&v_full[s], 2 * Cfg::V_BYTES);
#pragma unroll
        for (int j = 0; j < PKV / 64; ++j)
          tma_load_2d_pair(v + j * ((PD / 2) * 128), &tmVt, lv, t * PKV + 64 * j, (nkv * heads + h) * PD + (int)rank * (PD / 2));
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (rank == 0) {
      // ===== MMA issuer (leader; the whole warp runs the loop, one elected lane issues): UMMA M = 256 across the pair
      constexpr uint32_t idesc_qk = F16 ? make_idesc_f16(2 * PQ, PKV) : make_idesc_bf16(2 * PQ, PKV);     // 256 x 128
      constexpr uint32_t idesc_pv = F16 ? make_idesc_f16(2 * PQ, PD) : make_idesc_bf16(2 * PQ, PD);       // 256 x 256
      const uint64_t q_desc = make_desc_k_sw128(smem_u32(sQ));
      auto issue_qk = [&](int t) {
        const int s = t % PST, b = t & 1;
        mbar_wait(&k_full[s], (t / PST) & 1);
        fence_after_sync();
        const uint64_t k_desc = make_desc_k_sw128(smem_u32(smem + Cfg::K_OFF + s * Cfg::K_BYTES));
#pragma unroll
        for (int k = 0; k < PD / 16; ++k)                          // descriptor start field is in 16-byte units
          mma_ss_pair_elect(tmem_base + b * Cfg::S_COLS, q_desc + (uint64_t)(((k >> 2) * (PQ * 128) + (k & 3) * 32) >> 4),
                            k_desc + (uint64_t)(((k >> 2) * ((PKV / 2) * 128) + (k & 3) * 32) >> 4), idesc_qk, k ? 1u : 0u);
        mma_commit_pair_elect(&s_full[b]);
        mma_commit_pair_elect(&k_empty[s]);                        // K stage free (both CTAs) as soon as Q K^T(t) has read it
        if (lane == 0) ATRACE(t, 0);
      };
      mbar_wait(q_full, 0);
      issue_qk(0);
      for (int t = 0; t < nt; ++t) {
        if (t + 1 < nt) issue_qk(t + 1);                           // S(t+1) overlaps softmax(t)
        const int s = t % PST, b = t & 1;
        mbar_wait(&v_full[s], (t / PST) & 1);
        mbar_wait(p_full, t & 1);
        if (lane == 0) ATRACE(t, 1);
        fence_after_sync();
        const uint64_t v_desc = make_desc_k_sw128(smem_u32(smem + Cfg::V_OFF + s * Cfg::V_BYTES));
#pragma unroll
        for (int k = 0; k < PKV / 16; ++k)                         // P: keys 16k.. live in columns (k / 4) * 64 + (k % 4) * 8 of the S buffer
          mma_ts_pair_elect(tmem_base + Cfg::O_COL, tmem_base + b * Cfg::S_COLS + (k >> 2) * 64 + (k & 3) * 8,
                            v_desc + (uint64_t)(((k >> 2) * ((PD / 2) * 128) + (k & 3) * 32) >> 4), idesc_pv, (t | k) ? 1u : 0u);
        mma_commit_pair_elect(&v_empty[s]);
        mma_commit_pair_elect(pv_done);
        if (lane == 0) ATRACE(t, 2);
      }
    }
    __syncwarp();
  } else {
    // ===== softmax / correction / epilogue: row = TMEM lane; two threads per row, 64 keys of every step each
    const int quarter = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row = quarter * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const uint32_t lp = mapa(smem_u32(p_full), 0);
    const bool tr = (warp == 2 && lane == 0);
    float m = -INFINITY, l = 0.f;
    for (int t = 0; t < nt; ++t) {
      const int b = t & 1;
      const uint32_t sp = lane_base + b * Cfg::S_COLS + half * 64;
      mbar_wait(&s_full[b], (t >> 1) & 1);
      if (tr) ATRACE(t, 3);
      fence_after_sync();
      uint32_t s0[32], s1[32];
      tmem_ld_32x32(sp, s0);
      tmem_ld_32x32(sp + 32, s1);
      tmem_ld_wait();
      if (tr) ATRACE(t, 4);
      float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
      for (int j = 0; j < 32; ++j) { mx0 = fmaxf(mx0, __uint_as_float(s0[j])); mx1 = fmaxf(mx1, __uint_as_float(s1[j])); }
      float mx = fmaxf(mx0, mx1);
      float* xch = sX + (t & 1) * 256;
      xch[half * 128 + row] = mx;
      pair_barrier64(quarter);
      mx = fmaxf(mx, xch[(half ^ 1) * 128 + row]);
      const float m_new = fmaxf(m, mx * scale_log2);
      const bool grow = (m_new - m) > 8.0f;                        // lazy rescale (also true for t == 0)
      const float alpha = (grow && t > 0) ? ex2f(m - m_new) : 1.0f;
      if (grow) m = m_new;
      float sum0 = 0.f, sum1 = 0.f;
      uint32_t pk[32];
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        const float a0 = ex2f(fmaf(__uint_as_float(s0[j]), scale_log2, -m)), a1 = ex2f(fmaf(__uint_as_float(s0[j + 1]), scale_log2, -m));
        const float c0 = ex2f(fmaf(__uint_as_float(s1[j]), scale_log2, -m)), c1 = ex2f(fmaf(__uint_as_float(s1[j + 1]), scale_log2, -m));
        if (F16) {
          const __half2 pa = __floats2half2_rn(a0, a1), pc = __floats2half2_rn(c0, c1);
          sum0 += a0 + a1; sum1 += c0 + c1;                        // (unrounded: round-to-nearest is unbiased, the sums agree to ~2^-12 / sqrt(keys))
          pk[j >> 1] = *reinterpret_cast<const uint32_t*>(&pa); pk[16 + (j >> 1)] = *reinterpret_cast<const uint32_t*>(&pc);
        } else {
          const __nv_bfloat162 pa = __floats2bfloat162_rn(a0, a1), pc = __floats2bfloat162_rn(c0, c1);
          sum0 += __low2float(pa) + __high2float(pa); sum1 += __low2float(pc) + __high2float(pc);
          pk[j >> 1] = *reinterpret_cast<const uint32_t*>(&pa); pk[16 + (j >> 1)] = *reinterpret_cast<const uint32_t*>(&pc);
        }
      }
      l = l * alpha + (sum0 + sum1);
      if (tr) ATRACE(t, 5);
      if (t > 0) {
        // Every phase of pv_done is waited for, in order, by every softmax thread (P V(t-1) was issued a whole softmax step ago, so this
        // does not stall): a parity wait may lag ONE phase at most, and the final wait below would otherwise be able to mistake the
        // completion of P V(nt-3) for that of P V(nt-1).
        mbar_wait(pv_done, (t - 1) & 1);                           // P V(t-1) finished: O readable
        fence_after_sync();
      }
      if (t > 0 && __any_sync(0xffffffffu, alpha != 1.0f)) {       // identical decision in both warps of the pair (same rows, same m)
#pragma unroll 1
        for (int c = half * (PD / 2); c < (half + 1) * (PD / 2); c += 32) {
          uint32_t o[32];
          tmem_ld_32x32(lane_base + Cfg::O_COL + c, o);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) o[j] = __float_as_uint(__uint_as_float(o[j]) * alpha);
          tmem_st_32x32(lane_base + Cfg::O_COL + c, o);
        }
      }
      tmem_st_32x32(sp, pk);                                       // P over the first 32 of this thread's own 64 S columns
      tmem_st_wait();
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(lp);
      if (tr) ATRACE(t, 6);
    }
    // ---- epilogue: total row sum = both halves' partial sums; each half stores 128 of the 256 columns
    float* xch = sX + (nt & 1) * 256;
    xch[half * 128 + row] = l;
    pair_barrier64(quarter);
    const float inv = 1.0f / (l + xch[(half ^ 1) * 128 + row]);
    mbar_wait(pv_done, (nt - 1) & 1);
    fence_after_sync();
    if (tr) ATRACE(0, 7);
    // this warp's 32 rows x 128 columns -> staging tile (hi: 32 x 256 B, lo: the same; 16-byte chunk c of row r at r * 256 +
    // ((c ^ (r & 15)) << 4): conflict-free both ways) -> global, 16 lanes per row
    uint8_t* stg = smem + (warp - 2) * 16384;                      // Q + K regions: every UMMA that read them has completed (pv_done)
#pragma unroll 1
    for (int cc = 0; cc < 4; ++cc) {
      uint32_t o[32];
      tmem_ld_32x32(lane_base + Cfg::O_COL + half * (PD / 2) + cc * 32, o);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; j += 8) {
        uint4 u, w;
        split_bf16x2(__uint_as_float(o[j]) * inv, __uint_as_float(o[j + 1]) * inv, u.x, w.x);
        split_bf16x2(__uint_as_float(o[j + 2]) * inv, __uint_as_float(o[j + 3]) * inv, u.y, w.y);
        split_bf16x2(__uint_as_float(o[j + 4]) * inv, __uint_as_float(o[j + 5]) * inv, u.z, w.z);
        split_bf16x2(__uint_as_float(o[j + 6]) * inv, __uint_as_float(o[j + 7]) * inv, u.w, w.w);
        const int off = lane * 256 + (((cc * 4 + (j >> 3)) ^ (lane & 15)) << 4);
        *reinterpret_cast<uint4*>(stg + off) = u;
        if (Olo) *reinterpret_cast<uint4*>(stg + 8192 + off) = w;
      }
    }
    __syncwarp();
    {
      const int c = lane & 15;
      const size_t obase = (size_t)(n * T + q0 + quarter * 32) * ldo + h * PD + half * (PD / 2) + c * 8;
#pragma unroll 4
      for (int i = 0; i < 16; ++i) {
        const int rr = 2 * i + (lane >> 4);
        const int off = rr * 256 + ((c ^ (rr & 15)) << 4);
        *reinterpret_cast<uint4*>(O + obase + (size_t)rr * ldo) = *reinterpret_cast<const uint4*>(stg + off);
        if (Olo) *reinterpret_cast<uint4*>(Olo + obase + (size_t)rr * ldo) = *reinterpret_cast<const uint4*>(stg + 8192 + off);
      }
    }
    if (tr) ATRACE(0, 8);
  }
  fence_before_sync();
  cluster_sync_all();                                              // the peer's smem / TMEM must outlive every MMA that reads it
  if (warp == 1) tmem_dealloc2(tmem_base, Cfg::TMEM_COLS);
}

bool attention_pair_supported(int T, int d, int nctx) {
  const char* v1 = getenv("DVD_ATTN_V1");                           // (read per call: tests switch kernels inside one process)
  const int off = v1 ? atoi(v1) : 0;
  return !off && d == PD && nctx == 1 && T % (2 * PQ) == 0 && T % PKV == 0;
}

template <bool F16>
static int launch_attention_pair(const CUtensorMap& tmQ, const CUtensorMap& tmK, const CUtensorMap& tmVt, __nv_bfloat16* o, __nv_bfloat16* o_lo,
                                 int ldo, int nsamp, int heads, int T, float scale, int kv_div, cudaStream_t st) {
  auto kern = k_attn_pair<F16>;
  DVD_SET_MAX_SMEM(kern, APCfg::SMEM);
  const float scale_log2 = scale * 1.4426950408889634f;
  DVD_CUDA(launch_pdl_cluster(2, kern, dim3(T / PQ, heads, nsamp), dim3(PTHREADS), (size_t)APCfg::SMEM, st, 2, 1, tmQ, tmK, tmVt, o, o_lo, ldo, T,
                              heads, kv_div, scale_log2));
  DVD_LAUNCH_CHECK("k_attn_pair");
  return 0;
}

int attention_pair(const void* q, int ldq, const void* k, int ldk, const void* vt, __nv_bfloat16* o, __nv_bfloat16* o_lo, int ldo, int nsamp,
                   int heads, int T, float scale, int kv_div, int f16, cudaStream_t st) {
  DVD_REQUIRE(q && k && vt && o, "attention_pair: null pointer");
  DVD_REQUIRE(nsamp > 0 && nsamp <= 65535, "attention_pair: nsamp %d outside 1..65535", nsamp);
  DVD_REQUIRE(kv_div > 0 && nsamp % kv_div == 0, "attention_pair: nsamp %d is not a multiple of kv_div %d", nsamp, kv_div);
  DVD_REQUIRE(T % (2 * PQ) == 0, "attention_pair: T %d is not a multiple of %d", T, 2 * PQ);
  DVD_REQUIRE(ldo % 8 == 0, "attention_pair: ldo %d is not a multiple of 8", ldo);
  DVD_REQUIRE((reinterpret_cast<uintptr_t>(o) & 15) == 0, "attention_pair: o must be 16-byte aligned");
  DVD_REQUIRE((reinterpret_cast<uintptr_t>(o_lo) & 15) == 0, "attention_pair: o_lo must be 16-byte aligned");
  const int nkv = nsamp / kv_div;
  CUtensorMap tmQ, tmK, tmVt;
  int rc = make_tmap_bf16_2d(&tmQ, q, (uint64_t)nsamp * T, (uint64_t)heads * PD, (uint64_t)ldq, PQ, 64); if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmK, k, (uint64_t)nkv * T, (uint64_t)heads * PD, (uint64_t)ldk, PKV / 2, 64); if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmVt, vt, (uint64_t)nkv * heads * PD, (uint64_t)T, (uint64_t)T, PD / 2, 64); if (rc) return rc;
  return f16 ? launch_attention_pair<true>(tmQ, tmK, tmVt, o, o_lo, ldo, nsamp, heads, T, scale, kv_div, st)
             : launch_attention_pair<false>(tmQ, tmK, tmVt, o, o_lo, ldo, nsamp, heads, T, scale, kv_div, st);
}

}  // namespace dvd

#ifdef DVD_ATTN_TRACE
extern "C" __attribute__((visibility("default"))) int dvd_debug_attn_trace(unsigned long long* out) {
  return (int)cudaMemcpyFromSymbol(out, dvd::g_attn_trace, sizeof(dvd::g_attn_trace));
}
#endif
