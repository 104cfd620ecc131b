// tcgen05 GEMM: C[M,N] = epilogue(A[M,K] * W[N,K]^T), 16-bit operands (both K-major, exactly the torch Linear layouts),
// fp32 accumulation in tensor memory.  This file: tensor maps, the dispatcher and the GENERIC single-CTA kernel (any
// M % 128 == 0, ragged N); the denoiser's shapes run on the persistent CTA-pair kernel of gemm_pair.cu.
//
//   * one CTA computes a 128 x BN output tile (UMMA M=128, N=BN, K=16; BN in {64, 128, 256}); 8 warps:
//       warp 0 / one lane : TMA producer  — cp.async.bulk.tensor 2-D boxes (128 x 64 bf16, SWIZZLE_128B) into a ring of stages
//       warp 1 / one lane : MMA issuer    — 4 (bf16) or 12 (split pair: hi*hi, lo*hi, hi*lo) tcgen05.mma per stage,
//                                           tcgen05.commit frees the stage / signals the epilogue
//       all 8 warps       : epilogue      — tcgen05.ld (32 lanes x 32 columns per warp), fused Epilogue, vector stores
//   * K tails (K = 1032 for the r-embedder) are zero-filled by TMA; N tails are masked in the epilogue.
#include "gemm_tc.cuh"
#include "tc_common.cuh"
#include "tc_epilogue.cuh"
#include <stdlib.h>
#include <algorithm>

namespace dvd {

using namespace tc;

// ---------------------------------------------------------------------------------------- tensor-map encode (driver entry point at run time)
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return DVD_E_NOTMA; }
  DVD_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (ld * 2) % 16 == 0, "tensor map: base/stride must be 16-byte aligned (ld=%llu)",
              (unsigned long long)ld);
  DVD_REQUIRE(box_cols * 2 == 128 && box_rows <= 256, "tensor map: box must be 128 bytes wide");
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstr[1] = {ld * 2};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu ld=%llu", (int)r, (unsigned long long)rows,
                                     (unsigned long long)cols, (unsigned long long)ld); return DVD_E_NOTMA; }
  return 0;
}

// 4-D bf16 NHWC activation [N, H, W, C]; box = 64 channels x 128 pixels of one image row (implicit-GEMM conv A operand).
// Out-of-bounds coordinates (x = -1 / W, y = -1 / H: the conv's zero padding) are zero-filled by TMA.
int make_tmap_bf16_nhwc(CUtensorMap* out, const void* base, uint64_t n, uint64_t h, uint64_t w, uint64_t c) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return DVD_E_NOTMA; }
  DVD_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && c % 64 == 0 && w % 128 == 0, "nhwc tensor map: need C %% 64 == 0 and W %% 128 == 0");
  cuuint64_t gdim[4] = {c, w, h, n};
  cuuint64_t gstr[3] = {c * 2, w * c * 2, h * w * c * 2};
  cuuint32_t box[4] = {64, 128, 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (nhwc) failed (%d)", (int)r); return DVD_E_NOTMA; }
  return 0;
}

// Plain (unswizzled) 3-D tile map over an image stack: dims {w, h, planes} of `elem_bytes`-sized elements (4 = fp32, 1 = uint8),
// box {box_w, box_h, box_p}.  Used by the unwarp kernel to stage source windows; OOB elements are zero-filled (= zeros padding).
int make_tmap_image3d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t w, uint64_t h, uint64_t planes, uint32_t box_w,
                      uint32_t box_h, uint32_t box_p) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return DVD_E_NOTMA; }
  DVD_REQUIRE(elem_bytes == 4 || elem_bytes == 1, "image tensor map: fp32 or uint8 only");
  DVD_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (w * elem_bytes) % 16 == 0 && (box_w * elem_bytes) % 16 == 0 && box_w <= 256 &&
                  box_h <= 256 && box_p <= 256, "image tensor map: alignment / box limits");
  cuuint64_t gdim[3] = {w, h, planes};
  cuuint64_t gstr[2] = {w * elem_bytes, w * h * elem_bytes};
  cuuint32_t box[3] = {box_w, box_h, box_p};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(out, elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void*>(base), gdim,
                   gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (image) failed (%d) w=%llu h=%llu", (int)r, (unsigned long long)w,
                                     (unsigned long long)h); return DVD_E_NOTMA; }
  return 0;
}

// ---------------------------------------------------------------------------------------- optional phase trace (-DDVD_GEMM_TRACE)
#ifdef DVD_GEMM_TRACE
__device__ unsigned long long g_gemm_trace[2048][8];
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define DVD_TRACE(slot) do { g_gemm_trace[((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) & 2047][slot] = gtime(); } while (0)
#else
#define DVD_TRACE(slot) do { } while (0)
#endif

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (!cached[dev]) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// ---------------------------------------------------------------------------------------- kernel
constexpr int TBM = 128, TBK = 64;
constexpr int TC_THREADS = 256;          // warp 0: TMA producer, warp 1: MMA issuer, all 8 warps: epilogue

template <int BN, bool X3>
struct TcCfg {
  static constexpr int NOP = X3 ? 2 : 1;                                   // hi (+ lo) copies of every operand tile
  static constexpr int STAGES = X3 ? (BN == 64 ? 3 : 2) : ((BN == 64) ? 4 : ((BN <= 128) ? 3 : 2));
  static constexpr int TMEM_COLS = BN <= 64 ? 64 : (BN <= 128 ? 128 : 256);  // power of two >= BN
  static constexpr int A_BYTES = TBM * TBK * 2, B_BYTES = BN * TBK * 2;    // one copy
  static constexpr int STAGE_BYTES = NOP * (A_BYTES + B_BYTES);            // [A_hi | A_lo | B_hi | B_lo]
  static constexpr int B_OFF = NOP * A_BYTES;
  static constexpr int CW = BN < 128 ? BN : 128;                          // columns per epilogue pass
  static constexpr int STAGE_LD = CW + 4;                                 // fp32 staging row stride (16-byte aligned, conflict-free)
  static constexpr int STAGING_BYTES = 4 * 32 * STAGE_LD * 4;             // 4 row groups x 32 rows
  static constexpr int RING_BYTES = STAGES * STAGE_BYTES;
  static_assert(STAGING_BYTES <= RING_BYTES, "epilogue staging must fit in the (drained) operand ring");
  static constexpr int SMEM = RING_BYTES + 1024 /*align slack*/ + 128 /*barriers*/;
  static constexpr int MIN_CTAS = SMEM <= 112 * 1024 ? 2 : 1;
  static_assert(SMEM <= 232448, "shared memory budget");
};

struct ConvGeom { int H, W, Cin; };      // CONV: A is an NHWC activation, K = 9 * Cin ordered [ky][kx][Cin]

template <int BN, bool CONV, bool X3>
__global__ void __launch_bounds__(TC_THREADS, TcCfg<BN, X3>::MIN_CTAS)
k_gemm_tc(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmAl, const __grid_constant__ CUtensorMap tmB,
          const __grid_constant__ CUtensorMap tmBl, int M, int N, int K, Epilogue e, ConvGeom cg) {
  using Cfg = TcCfg<BN, X3>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::RING_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tmem_full = empty + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // M tiles beyond the 65535 limit of gridDim.y (the 512x512 pyramid levels of >= 32 documents) are folded into gridDim.z
  const int m0 = (blockIdx.z * gridDim.y + blockIdx.y) * TBM, n0 = blockIdx.x * BN;
  if (m0 >= M) return;                                  // whole CTA (ragged last z-slice)
  const int nkb = (K + TBK - 1) / TBK;

  pdl_trigger();                                        // the next kernel of the stream may start its own prologue
  if (threadIdx.x == 0) {
    DVD_TRACE(0);                                       // CTA start
    prefetch_tmap(&tmA); prefetch_tmap(&tmB);
    if (X3) { prefetch_tmap(&tmAl); prefetch_tmap(&tmBl); }
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                                           // everything above overlapped the previous kernel's tail
  if (threadIdx.x == 0) DVD_TRACE(1);                   // prologue done, predecessor finished

  if (warp == 0) {
    if (lane == 0) {
      // ===== TMA producer
      int cn = 0, cy = 0, cx = 0, cblocks = 1;
      if (CONV) {
        const int hw = cg.H * cg.W;
        cn = m0 / hw; const int rem = m0 % hw; cy = rem / cg.W; cx = rem % cg.W;      // 128 consecutive pixels of one image row
        cblocks = cg.Cin / 64;
      }
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES, it = kb / STAGES;
        mbar_wait(&empty[s], (it & 1) ^ 1);
        uint8_t* a = smem + s * Cfg::STAGE_BYTES;
        mbar_expect_tx(&full[s], Cfg::STAGE_BYTES);
#pragma unroll
        for (int o = 0; o < Cfg::NOP; ++o) {
          const CUtensorMap* ta = o ? &tmAl : &tmA;
          const CUtensorMap* tb = o ? &tmBl : &tmB;
          uint8_t* ad = a + o * Cfg::A_BYTES;
          uint8_t* bd = a + Cfg::B_OFF + o * Cfg::B_BYTES;
          if (CONV) {
            const int tap = kb / cblocks, cb = kb % cblocks;
            tma_load_4d(ad, ta, &full[s], cb * 64, cx + tap % 3 - 1, cy + tap / 3 - 1, cn);
          } else {
            tma_load_2d(ad, ta, &full[s], kb * TBK, m0);
          }
          tma_load_2d(bd, tb, &full[s], kb * TBK, n0);
          if (BN == 256) tma_load_2d(bd + 128 * TBK * 2, tb, &full[s], kb * TBK, n0 + 128);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      // ===== MMA issuer
      constexpr uint32_t idesc = make_idesc_bf16(TBM, BN);
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES, it = kb / STAGES;
        mbar_wait(&full[s], it & 1);
        if (kb == 0) DVD_TRACE(2);                      // first stage landed
        if (kb == nkb - 1) DVD_TRACE(3);                // last stage landed
        fence_after_sync();
        const uint32_t a_addr = smem_u32(smem + s * Cfg::STAGE_BYTES), b_addr = a_addr + Cfg::B_OFF;
#pragma unroll
        for (int k = 0; k < TBK / 16; ++k) {
          // advancing K inside the 128-byte swizzle atom = +32 bytes on the start address
          const uint64_t ah = make_desc_k_sw128(a_addr + k * 32), bh = make_desc_k_sw128(b_addr + k * 32);
          mma_f16_ss(tmem_base, ah, bh, idesc, (kb | k) ? 1u : 0u);
          if (X3) {
            mma_f16_ss(tmem_base, make_desc_k_sw128(a_addr + Cfg::A_BYTES + k * 32), bh, idesc, 1u);       // lo * hi
            mma_f16_ss(tmem_base, ah, make_desc_k_sw128(b_addr + Cfg::B_BYTES + k * 32), idesc, 1u);       // hi * lo
          }
        }
        mma_commit(&empty[s]);                           // stage reusable once these MMAs have read it
      }
      mma_commit(tmem_full);                             // accumulator complete
    }
    __syncwarp();
  }

  // ===== epilogue.  tmem_full => every MMA has retired, so every TMA write has been consumed: the operand ring is dead
  // and is reused as an fp32 staging tile.  All 8 warps take part: warps w and w+4 own the same 32 rows (a warp can only read the
  // TMEM lanes 32*(w%4)..+31) and split the columns in phase 1 and the rows in phase 2, synchronised by a 64-thread named
  // barrier per row group.
  //   Phase 1 (thread = row, TMEM lane): TMEM -> registers -> staging (+ the transposed V^T store, which is naturally
  //   coalesced in this mapping).  Phase 2 (lane = 4 consecutive columns): staging -> fused epilogue -> fully coalesced
  //   512-byte row segments in global memory.
  mbar_wait(tmem_full, 0);
  if (threadIdx.x == 0) DVD_TRACE(4);                   // accumulator complete
  fence_after_sync();
  constexpr int CW = Cfg::CW, SLD = Cfg::STAGE_LD;
  static_assert((CW / 2) % 32 == 0, "each half of an epilogue pass is a whole number of 32-column TMEM loads");
  const int wq = warp & 3, wh = warp >> 2;               // row group (TMEM lane quarter), column / row half
  float* stage = reinterpret_cast<float*>(smem) + wq * 32 * SLD;
  const int row_t = m0 + wq * 32 + lane;                 // phase-1 row of this thread (M % 128 == 0 is checked on the host)
  auto pair_sync = [&]() { asm volatile("bar.sync %0, 64;" ::"r"(1 + wq) : "memory"); };
#pragma unroll 1
  for (int pass = 0; pass < BN / CW; ++pass) {
#pragma unroll 1
    for (int c0 = wh * (CW / 2); c0 < (wh + 1) * (CW / 2); c0 += 32) {
      uint32_t r[32];
      tmem_ld_32x32(tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(pass * CW + c0), r);
      tmem_ld_wait();
      float* srow = stage + lane * SLD + c0;
#pragma unroll
      for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(srow + j) = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]),
                                                                                         __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
      const int col0 = n0 + pass * CW + c0;
      if (e.vt_out && col0 >= e.vt_col0 && col0 + 31 < N) {
        // V^T (bias-only epilogue, checked on the host): the bias of the 32 columns is warp-uniform -> 8 vector loads up front
        float bv[32];
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 b4 = e.bias ? __ldg(reinterpret_cast<const float4*>(e.bias + col0 + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
          bv[j] = b4.x; bv[j + 1] = b4.y; bv[j + 2] = b4.z; bv[j + 3] = b4.w;
        }
        uint16_t* o = reinterpret_cast<uint16_t*>(e.vt_out) + ((size_t)(row_t >> 10) * (N - e.vt_col0) + (col0 - e.vt_col0)) * 1024 + (row_t & 1023);
#pragma unroll
        for (int j = 0; j < 32; ++j) o[(size_t)j * 1024] = cvt16(__uint_as_float(r[j]) + bv[j], e.out_f16);
      }
    }
    pair_sync();                                         // both column halves of the row group are staged
    // ---- phase 2: this warp finishes rows wh*16 .. wh*16+15 of the group
    const int col = n0 + pass * CW + 4 * lane;
    if (4 * lane < CW && col < N) {
      const EpiCols ec = load_epi_cols(e, col);
#pragma unroll 1
      for (int r0 = wh * 16; r0 < wh * 16 + 16; r0 += 8) {
        float4 a[8], q[8], p[8];
        // batch the loads of 8 rows (staging, residual, pos-embed) before any dependent math or store
#pragma unroll
        for (int i = 0; i < 8; ++i) a[i] = *reinterpret_cast<const float4*>(stage + (r0 + i) * SLD + 4 * lane);
        if (e.resid) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int row = m0 + wq * 32 + r0 + i;
            const int rr = e.resid_mod ? (row % e.resid_mod) : row;
            q[i] = *reinterpret_cast<const float4*>(e.resid + (size_t)rr * e.ldr + col);      // may alias e.out (in-place residual)
          }
        }
        if (e.pos) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int row = m0 + wq * 32 + r0 + i;
            p[i] = __ldg(reinterpret_cast<const float4*>(e.pos + (size_t)(row % e.pos_rows) * N + col));
          }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int row = m0 + wq * 32 + r0 + i;
          float v[4];
          apply_epi4(ec, a[i], e.pos != nullptr, p[i], e.resid != nullptr, q[i], v);
          int orow, ocol;
          epilogue_dest(e, row, col, orow, ocol);
          store_tc_out4(e, orow, ocol, v);
        }
      }
    }
    pair_sync();                                         // the staging rows may be overwritten by the next pass
  }
  fence_before_sync();
  __syncthreads();
  if (threadIdx.x == 0) DVD_TRACE(5);                   // epilogue done
  if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

template <int BN, bool CONV, bool X3>
static int launch_tc(const CUtensorMap& tmA, const CUtensorMap& tmAl, const CUtensorMap& tmB, const CUtensorMap& tmBl, int M, int N, int K,
                     const Epilogue& e, ConvGeom cg, cudaStream_t st) {
  using Cfg = TcCfg<BN, X3>;
  auto kern = k_gemm_tc<BN, CONV, X3>;
  DVD_SET_MAX_SMEM(kern, Cfg::SMEM);
  const int my = cdiv(M, TBM), gy = my > 32768 ? 32768 : my;
  dim3 grid(cdiv(N, BN), gy, cdiv(my, gy));
  DVD_CUDA(launch_pdl(1, k_gemm_tc<BN, CONV, X3>, grid, dim3(TC_THREADS), (size_t)Cfg::SMEM, st, tmA, tmAl, tmB, tmBl, M, N, K, e, cg));
  DVD_LAUNCH_CHECK("k_gemm_tc");
  return 0;
}

static int check_epilogue(const Epilogue& e, int N) {
  DVD_REQUIRE(N % 4 == 0, "gemm_tc: N must be a multiple of 4");
  auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  DVD_REQUIRE(al(e.bias) && al(e.scale) && al(e.shift) && al(e.gate) && al(e.pos) && al(e.resid) && al(e.out) &&
              (reinterpret_cast<uintptr_t>(e.out_bf16) & 7) == 0 && (reinterpret_cast<uintptr_t>(e.out_lo) & 7) == 0,
              "gemm_tc: epilogue pointers must be 16-byte aligned");
  DVD_REQUIRE(e.ldc % 4 == 0 && e.ldr % 4 == 0 && e.ldc_bf16 % 4 == 0 && e.group_col_stride % 4 == 0, "gemm_tc: epilogue leading dims %% 4");
  DVD_REQUIRE(!e.out_lo || (e.out_bf16 && !e.out_f16), "gemm_tc: out_lo needs out_bf16 (bf16 pair)");
  DVD_REQUIRE(!e.vt_out || (e.vt_col0 % 32 == 0 && N % 32 == 0 && !e.scale && !e.act && !e.pos && !e.gate && !e.resid),
              "gemm_tc: the V^T output supports a bias-only epilogue with vt_col0 %% 32 == 0");
  return 0;
}

static bool use_v1() {       // DVD_GEMM_V1=1: force the generic single-CTA kernel (A/B tests, tools/gemm_bench.py)
  static int v = -1;
  if (v < 0) { const char* s = getenv("DVD_GEMM_V1"); v = (s && s[0] == '1') ? 1 : 0; }
  return v == 1;
}

template <bool CONV, bool X3>
static int launch_tc_bn(int bn, const CUtensorMap& tmA, const CUtensorMap& tmAl, const CUtensorMap& tmB, const CUtensorMap& tmBl, int M, int N,
                        int K, const Epilogue& e, ConvGeom cg, cudaStream_t st) {
  if (bn == 256) return launch_tc<256, CONV, X3>(tmA, tmAl, tmB, tmBl, M, N, K, e, cg, st);
  if (bn == 64) return launch_tc<64, CONV, X3>(tmA, tmAl, tmB, tmBl, M, N, K, e, cg, st);
  return launch_tc<128, CONV, X3>(tmA, tmAl, tmB, tmBl, M, N, K, e, cg, st);
}

int gemm_tc(const TcMat& A, const TcMat& W, int M, int N, int K, const Epilogue& e, cudaStream_t st) {
  DVD_REQUIRE(A.hi && W.hi && (e.out || e.out_bf16), "gemm_tc: null pointer");
  DVD_REQUIRE(M > 0 && N > 0 && K > 0 && K % 8 == 0 && M % 128 == 0, "gemm_tc: bad shape M=%d N=%d K=%d (M must be a multiple of 128)", M, N, K);
  DVD_REQUIRE(A.f16 ? (!A.lo && W.lo) : ((A.lo != nullptr) == (W.lo != nullptr)),
              "gemm_tc: A and W must both be split pairs or both plain (or: fp16 A with a weight pair)");
  int rc = check_epilogue(e, N); if (rc) return rc;
  const bool periods_ok = e.resid_mod % 128 == 0 && e.pos_rows % 128 == 0 && e.group_rows % 128 == 0;
  if (!use_v1() && periods_ok && gemm_pair_supported(M, N, K, false)) return gemm_pair_dispatch(A, W, M, N, K, e, 0, 0, 0, 0, st);
  DVD_REQUIRE(!e.ln_stats && !e.stats_out, "gemm_tc: fused LayerNorm / row statistics need the CTA-pair kernel (M %% 256 == 0, N %% 64 == 0)");
  DVD_REQUIRE(!A.f16, "gemm_tc: the fp16-activation mode needs the CTA-pair kernel (M %% 256 == 0, N %% 64 == 0)");
  const bool x3 = A.lo != nullptr;
  // wide tiles only when they still fill the machine
  const bool wide = (N % 256 == 0) && ((long long)(M / 128) * (N / 256) * 100 >= 190LL * sm_count());
  const int bn = (N <= 64) ? 64 : (wide ? 256 : 128);
  CUtensorMap tmA, tmB, tmAl, tmBl;
  rc = make_tmap_bf16_2d(&tmA, A.hi, (uint64_t)M, (uint64_t)K, (uint64_t)A.ld, 128, 64); if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmB, W.hi, (uint64_t)N, (uint64_t)K, (uint64_t)W.ld, bn == 64 ? 64 : 128, 64); if (rc) return rc;
  tmAl = tmA; tmBl = tmB;
  if (x3) {
    rc = make_tmap_bf16_2d(&tmAl, A.lo, (uint64_t)M, (uint64_t)K, (uint64_t)A.ld, 128, 64); if (rc) return rc;
    rc = make_tmap_bf16_2d(&tmBl, W.lo, (uint64_t)N, (uint64_t)K, (uint64_t)W.ld, bn == 64 ? 64 : 128, 64); if (rc) return rc;
  }
  ConvGeom cg{0, 0, 0};
  return x3 ? launch_tc_bn<false, true>(bn, tmA, tmAl, tmB, tmBl, M, N, K, e, cg, st)
            : launch_tc_bn<false, false>(bn, tmA, tmAl, tmB, tmBl, M, N, K, e, cg, st);
}

// 3x3 / pad 1 / stride 1 convolution as an implicit GEMM: in NHWC [B,H,W,Cin], Wt [Cout, 9*Cin] ([ky][kx][Cin]),
// out NHWC [B,H,W,Cout] through the Epilogue (bias + ReLU, 16-bit and/or fp32).  Two operand forms: a bf16 activation with a bf16
// weight (one pass), or an fp16 activation with an fp16 weight pair (two passes).
int conv3x3_tc(const TcMat& in, const TcMat& Wt, int B, int H, int Wd, int Cin, int Cout, const Epilogue& e, cudaStream_t st) {
  DVD_REQUIRE(in.hi && Wt.hi && (e.out || e.out_bf16), "conv3x3_tc: null pointer");
  DVD_REQUIRE(Cin % 64 == 0 && Wd % 128 == 0 && (Cout == 64 || Cout % 128 == 0), "conv3x3_tc: unsupported shape Cin=%d W=%d Cout=%d", Cin, Wd, Cout);
  DVD_REQUIRE(!in.lo && (in.f16 ? Wt.lo != nullptr : Wt.lo == nullptr),
              "conv3x3_tc: bf16 activation with a bf16 weight, or fp16 activation with an fp16 weight pair");
  const int M = B * H * Wd, K = 9 * Cin;
  int rc = check_epilogue(e, Cout); if (rc) return rc;
  if (!use_v1() && gemm_pair_supported(M, Cout, K, true)) {
    TcMat w = Wt; w.ld = K;
    return gemm_pair_dispatch(in, w, M, Cout, K, e, B, H, Wd, Cin, st);
  }
  DVD_REQUIRE(!in.f16, "conv3x3_tc: the fp16-activation mode needs the CTA-pair kernel");
  const int bn = Cout == 64 ? 64 : ((Cout % 256 == 0 && (long long)(M / 128) * (Cout / 256) >= 2LL * sm_count()) ? 256 : 128);
  CUtensorMap tmA, tmB;
  rc = make_tmap_bf16_nhwc(&tmA, in.hi, (uint64_t)B, (uint64_t)H, (uint64_t)Wd, (uint64_t)Cin); if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmB, Wt.hi, (uint64_t)Cout, (uint64_t)K, (uint64_t)K, bn == 64 ? 64 : 128, 64); if (rc) return rc;
  ConvGeom cg{H, Wd, Cin};
  return launch_tc_bn<true, false>(bn, tmA, tmA, tmB, tmB, M, Cout, K, e, cg, st);
}

}  // namespace dvd

#ifdef DVD_GEMM_TRACE
extern "C" __attribute__((visibility("default"))) int dvd_debug_gemm_trace(unsigned long long* out, int n_ctas) {
  return (int)cudaMemcpyFromSymbol(out, dvd::g_gemm_trace, (size_t)n_ctas * 8 * sizeof(unsigned long long));
}
#endif
