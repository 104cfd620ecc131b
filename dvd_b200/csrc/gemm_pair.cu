// Persistent CTA-pair tcgen05 GEMM: the kernel every dense layer of the denoiser runs on.
//
//   C[M,N] = epilogue(A[M,K] * W[N,K]^T)      A, W K-major 16-bit: bf16 (1 tensor-core pass), bf16 hi + lo pairs on both sides (3 passes,
//                                             DVD_PREC_BF16X3), or ONE fp16 activation x fp16 weight pair (2 passes: the decoder's q|k|v GEMM)
//
// Shape of the machine: 74 clusters of two CTAs (the two SMs of a TPC), one cluster per TPC, each looping over work units.
//   * a unit = one 256 x BN output tile (UMMA M = 256 across the pair, tcgen05.mma.cta_group::2); units are dealt round-robin
//     (unit u -> pair u % npairs).  The M = 2048 problems of a single document have only 48..144 tiles: the host picks BN in
//     {64,128,192,256} from a cycle model so that the tile count fits the 74 pairs best (e.g. N = 1536 runs as 64 tiles of 256 x 192).
//     Split-K through global memory was implemented and measured (profiles/r2_gemm_sweep.txt): always slower - the partial tiles'
//     write / wait / read-back serialises two epilogues per tile - and was removed again.
//   * per SM the pair mode stages 128 A rows and only HALF of the W tile (BN/2 rows): 32 KB instead of 48 KB of L2 -> SM traffic per
//     k-block of a 128 x 256 tile, which is what bounds a one-SM-per-tile kernel (~13 TB/s of L2 reads at 1.1 PFLOP/s, DESIGN.md).
//   * warp 0 (one lane, both CTAs)  TMA producer: ring of 3..8 stages of [A_hi | A_lo | W_hi | W_lo] boxes (SWIZZLE_128B), continuous
//     across units; transaction bytes of both CTAs are counted on the LEADER's full barrier.
//   * warp 1 (leader; the whole warp runs the loop, one ELECTED lane issues)  MMA issuer: 4 / 12 / 8 UMMA 256 x BN x 16 per stage into one
//     of TWO TMEM accumulators; tcgen05.commit multicasts "stage free" / "accumulator ready" to both CTAs.
//   * warps 4..11 (both CTAs)       epilogue of the CTA's own 128 rows, overlapping the next unit's main loop: each warp owns a TMEM
//     lane quarter x half of the columns; tcgen05.ld 16x256b (mma-fragment layout: a quad holds one 32-byte sector of a row) -> fused
//     epilogue in registers -> sector-complete global accesses, no shared-memory staging (16-bit rows: 4 x 4 quad transpose -> 16-byte
//     stores).  The 32-column chunk body is ONE rolled copy of code, warmed by a dry pass while the first main loop runs (cold
//     instruction fetch was 3.3 us per chunk inside a step).
//   * CONV: A is an NHWC activation read through a 4-D tensor map (implicit GEMM of the 3x3 pyramid convolutions, zero padding = TMA
//     out-of-bounds fill); a pair covers 256 consecutive pixels of one image row.
#include "gemm_tc.cuh"
#include "tc_common.cuh"
#include "tc_epilogue.cuh"
#include <stdlib.h>

namespace dvd {
using namespace tc;

constexpr int PBM = 128, PBK = 64;
// 12 warps = 3 warpgroups: warpgroup 0 = {warp 0: TMA producer, warp 1: MMA issuer, warps 2-3: idle}, warpgroups 1-2 = 8 epilogue warps.
// The kernel is launched with 168 registers per thread (65536 / 384); after the set-up the first warpgroup gives registers back
// (setmaxnreg.dec 56) and the epilogue warpgroups take them (setmaxnreg.inc 224): their software-pipelined epilogue (accumulator fragment +
// two sets of prefetched residual / pos-embed / column vectors) spilled ~1 KB per thread under the flat 168-register budget.
constexpr int PP_THREADS = 384;
constexpr int PP_EPI_WARP0 = 4;           // first epilogue warp
constexpr int PP_EPI_WARPS = 8;
constexpr int PP_REGS_CTRL = 56, PP_REGS_EPI = 224;
static_assert(128 * PP_REGS_CTRL + 256 * PP_REGS_EPI <= 65536, "register budget after setmaxnreg");

// MODE: 0 = bf16 x bf16 (one pass); 1 = split pairs on both sides (hi*hi + lo*hi + hi*lo, DVD_PREC_BF16X3); 2 = ONE fp16 activation
// operand x fp16 weight pair (hi + lo): two passes, for the GEMMs whose activation tolerates fp16 rounding (oracle/precision_study.py
// --decoder-breakdown: it is the WEIGHT rounding that moves the map, the same perturbation for every token and step).  Everything is
// IEEE fp16 in this mode: kind::f16 rejects an fp16 A next to a bf16 B (illegal instruction, tried).
template <int BN, int MODE>
struct PairCfg {
  static constexpr int NA = MODE == 1 ? 2 : 1, NB = MODE >= 1 ? 2 : 1;
  static constexpr int A_BYTES = PBM * PBK * 2;                 // 16 KB: this CTA's 128 rows
  static constexpr int B_BYTES = (BN / 2) * PBK * 2;            // this CTA's half of the W tile
  static constexpr int STAGE_BYTES = NA * A_BYTES + NB * B_BYTES;
  static constexpr int B_OFF = NA * A_BYTES;
  static constexpr int FIXED = 1024 /*align slack*/ + 256 /*barriers*/;
  static constexpr int STAGES_FIT = (232448 - FIXED) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_FIT > 8 ? 8 : STAGES_FIT;
  static constexpr int RING_BYTES = STAGES * STAGE_BYTES;
  static constexpr int TMEM_COLS = (2 * BN <= 128) ? 128 : ((2 * BN <= 256) ? 256 : 512);
  static constexpr int SMEM = RING_BYTES + FIXED;
  static_assert(STAGES >= 2 && SMEM <= 232448, "shared memory budget");
  static_assert(A_BYTES % 1024 == 0 && B_BYTES % 1024 == 0, "SWIZZLE_128B tiles are 1024-byte aligned");
};

struct PairParams {
  int M, N, K;
  int tiles_n, units, npairs;
  int late_tile0;                 // column tiles >= late_tile0 are scheduled FIRST (0: natural order)
  int conv_h, conv_w, conv_cin;
  int epi;                        // epi_key(flags, out) of a compiled epilogue body, or EPI_GENERIC
};

// ---- optional phase trace (-DDVD_GEMM_TRACE, tools/gemm_trace.py): %globaltimer per CTA at the phase boundaries of its first two units
#ifdef DVD_GEMM_TRACE
__device__ unsigned long long g_pair_trace[512][16];
__device__ __forceinline__ unsigned long long ptime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
__device__ int g_pair_trace_n;   // != 0: record only launches with this N (catches ONE GEMM of a whole step: tools/step_trace.py)
#define PTRACE(slot) do { if ((slot) < 16 && (g_pair_trace_n == 0 || p.N == g_pair_trace_n)) g_pair_trace[blockIdx.x & 511][slot] = ptime(); } while (0)
#else
#define PTRACE(slot) do { } while (0)
#endif
#ifdef DVD_GEMM_TRACE2      // epilogue detail of (unit 0, chunk 0, warp 2) in slots 7..12 (single-unit shapes only)
#define ETRACE(slot) do { if (warp == PP_EPI_WARP0 && lane == 0 && it == 0 && ch == 0) PTRACE(slot); } while (0)
#else
#define ETRACE(slot) do { } while (0)
#endif

// ---- specialised epilogue bodies.  The generic Epilogue is a bag of run-time options; evaluating them per row costs ~600 warp
// instructions per 32 x 32 chunk, and with two epilogue warps per scheduler the epilogue of a 128 x 256 tile took 10 us (measured
// with tools/gemm_trace.py --epi).  The host classifies the Epilogue into a (flags, output kind) key; the combinations the denoiser
// uses are compiled as straight-line code, anything else takes the generic path.
enum { EF_SCALE = 1, EF_FLOOR = 2, EF_GATE = 4, EF_POS = 8, EF_RES = 16, EF_GELU = 32, EF_GELUX = 64, EF_LN = 128 };
// EO_F32X: fp32 residual stream + its 16-bit operand copy (bf16, or a pair when out_lo is set) + per-row partial statistics for a
// LayerNorm fused into the next GEMM
enum { EO_F32 = 0, EO_BF16 = 1, EO_PAIR = 2, EO_F16 = 3, EO_F32X = 4 };
constexpr int EPI_GENERIC = -1;
__host__ __device__ constexpr int epi_key(int flags, int out) { return (flags << 3) | out; }

struct LnRows { float m[4], rs[4]; };   // mean / rstd of this thread's four rows (fused-LN consumers)

// Register-fragment epilogue.  tcgen05.ld.16x256b.x4 hands a warp 16 TMEM lanes x 32 columns in the mma-fragment layout: thread t holds, for
// each 8-column block j, columns 8j + 2(t%4) + {0,1} of lanes t/4 and t/4 + 8.  Two loads (lanes +0 and +16) cover the warp's 32 lanes, so a
// thread owns rows t/4 + 8i (i = 0..3) x 4 column pairs.  A quad then holds 8 consecutive columns of a row = one 32-byte sector of an fp32
// output / residual row, so the global accesses are sector-complete WITHOUT a shared-memory transpose: no staging tile, no warp syncs,
// and the ring gets the 32 KB back.  (The first version staged through XOR-swizzled shared memory: 1.5 us per 32x32 chunk, see
// profiles/r2_gemm_trace_*.txt.)
struct EpiRowCtx { int col0, res_row0, pos_row0, orow0, ocol_add, N; };      // col0: first column of the chunk; *_row0: of the warp's 32 rows

struct Frag { uint32_t a[16], b[16]; };       // a: lanes 0..15 of the quarter, b: lanes 16..31
__device__ __forceinline__ float2 frag_val(const Frag& f, int i, int j) {     // row t/4 + 8i, columns 8j + 2(t%4) + {0,1}
  const uint32_t* r = (i < 2) ? f.a : f.b;
  const int o = 4 * j + 2 * (i & 1);
  return make_float2(__uint_as_float(r[o]), __uint_as_float(r[o + 1]));
}

// Everything the epilogue of one 32 x 32 chunk READS from global memory (per-column vectors, residual, pos-embed).  None of it depends on
// the accumulator, so the loads of chunk ch+1 are issued before chunk ch is processed (and those of a unit's first chunk before the
// wait for the accumulator): the L2 latency of the bias / residual fetch (~0.5 us, it used to be paid once per chunk and warp) is hidden.
template <int F>
struct EpiLoads {
  float2 cb[4], cs[4], ct[4], cg[4], cl[4];
  float2 qv[4][4], pv[4][4];
};
template <int F>
__device__ __forceinline__ void epi_load(const Epilogue& e, const EpiRowCtx& c, int lane, EpiLoads<F>& L) {
  const int tr = lane >> 2, tc2 = 2 * (lane & 3);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int col = c.col0 + 8 * j + tc2;
    L.cb[j] = e.bias ? __ldg(reinterpret_cast<const float2*>(e.bias + col)) : make_float2(0.f, 0.f);
    if (F & EF_SCALE) { L.cs[j] = __ldg(reinterpret_cast<const float2*>(e.scale + col)); L.ct[j] = __ldg(reinterpret_cast<const float2*>(e.shift + col)); }
    if (F & EF_GATE) L.cg[j] = __ldg(reinterpret_cast<const float2*>(e.gate + col));
    if (F & EF_LN) L.cl[j] = __ldg(reinterpret_cast<const float2*>(e.ln_colsum + col));
  }
  if (F & EF_RES) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float* rp = e.resid + (size_t)(c.res_row0 + tr + 8 * i) * e.ldr + c.col0 + tc2;       // may alias e.out (in-place residual)
#pragma unroll
      for (int j = 0; j < 4; ++j) L.qv[i][j] = *reinterpret_cast<const float2*>(rp + 8 * j);
    }
  }
  if (F & EF_POS) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float* pp = e.pos + (size_t)(c.pos_row0 + tr + 8 * i) * c.N + c.col0 + tc2;
#pragma unroll
      for (int j = 0; j < 4; ++j) L.pv[i][j] = __ldg(reinterpret_cast<const float2*>(pp + 8 * j));
    }
  }
}

// 4 x 4 transpose of 32-bit values inside a quad (lanes 4g .. 4g+3): lane q ends up with element q of every lane, in lane order.
// The mma-fragment layout leaves a lane with 2 adjacent columns of a row (4 bytes of 16-bit output) per 8-column group; after the
// transpose a lane holds 8 adjacent columns, so a 16-bit row segment leaves as ONE 16-byte store per lane and a quad covers 64
// contiguous bytes (two full sectors) instead of four 4-byte stores per lane (16 bytes per quad: half sectors).  Measured inside a
// step (tools/step_trace.py): the 4-byte stores of conv1's hi + lo tile took 8 us to drain the accumulator, 2.8 us in a bf16 microbench.
__device__ __forceinline__ void quad_transpose4(uint32_t (&v)[4], int q) {
  const bool b1 = (q & 2) != 0, b0 = (q & 1) != 0;
  uint32_t s0 = b1 ? v[0] : v[2], s1 = b1 ? v[1] : v[3];
  s0 = __shfl_xor_sync(0xffffffffu, s0, 2); s1 = __shfl_xor_sync(0xffffffffu, s1, 2);
  if (b1) { v[0] = s0; v[1] = s1; } else { v[2] = s0; v[3] = s1; }
  uint32_t t0 = b0 ? v[0] : v[1], t1 = b0 ? v[2] : v[3];
  t0 = __shfl_xor_sync(0xffffffffu, t0, 1); t1 = __shfl_xor_sync(0xffffffffu, t1, 1);
  if (b0) { v[0] = t0; v[2] = t1; } else { v[1] = t0; v[3] = t1; }
}

template <int F, int O>
__device__ __forceinline__ void epi_rows(const Epilogue& e, const Frag& f, const EpiRowCtx& c, int lane, const EpiLoads<F>& L, const LnRows& ln,
                                         const bool live) {                  // !live: instruction-cache warm-up pass, nothing is stored
  const int tr = lane >> 2, q = lane & 3, tc2 = 2 * q;
  constexpr bool OUT16 = (O != EO_F32);                       // a 16-bit tile is written (EO_F32X: next to the fp32 one)
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const size_t orow = (size_t)(c.orow0 + tr + 8 * i);
    const size_t o32 = orow * e.ldc + c.col0 + tc2 + c.ocol_add;
    float s1 = 0.f, s2 = 0.f;                                  // EO_F32X: this thread's share of the row's chunk statistics
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float2 a = frag_val(f, i, j);
      if (F & EF_LN) { a.x = ln.rs[i] * (a.x - ln.m[i] * L.cl[j].x); a.y = ln.rs[i] * (a.y - ln.m[i] * L.cl[j].y); }
      float v0 = a.x + L.cb[j].x, v1 = a.y + L.cb[j].y;
      if (F & EF_SCALE) { v0 = v0 * L.cs[j].x + L.ct[j].x; v1 = v1 * L.cs[j].y + L.ct[j].y; }
      if (F & EF_FLOOR) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
      if (F & EF_GELU) { v0 = gelu_tanh_fast(v0); v1 = gelu_tanh_fast(v1); }
      if (F & EF_GELUX) { v0 = gelu_tanh(v0); v1 = gelu_tanh(v1); }
      if (F & EF_POS) { v0 += L.pv[i][j].x; v1 += L.pv[i][j].y; }
      if (F & EF_GATE) { v0 *= L.cg[j].x; v1 *= L.cg[j].y; }
      if (F & EF_RES) { v0 += L.qv[i][j].x; v1 += L.qv[i][j].y; }
      if ((O == EO_F32 || O == EO_F32X) && live) *reinterpret_cast<float2*>(e.out + o32 + 8 * j) = make_float2(v0, v1);
      if (O == EO_F32X) { s1 += v0 + v1; s2 += v0 * v0 + v1 * v1; }
      if (O == EO_PAIR || (O == EO_F32X && e.out_lo)) split_bf16x2(v0, v1, hi[j], lo[j]);
      else if (O == EO_F16 || (O == EO_F32X && e.out_f16)) hi[j] = pack_f16x2(v0, v1);
      else if (OUT16) hi[j] = pack_bf16x2(v0, v1);
    }
    if (OUT16) {
      const size_t o16 = orow * e.ldc_bf16 + c.col0 + c.ocol_add + 8 * q;     // this lane's 8 columns after the transpose
      quad_transpose4(hi, q);
      if (live) *reinterpret_cast<uint4*>(e.out_bf16 + o16) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      if (O == EO_PAIR || (O == EO_F32X && e.out_lo)) {
        quad_transpose4(lo, q);
        if (live) *reinterpret_cast<uint4*>(e.out_lo + o16) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      }
    }
    if (O == EO_F32X) {
      // the quad holds the 32 columns of this chunk of row tr + 8i: fixed-order butterfly, then one (sum, sum of squares) per chunk
      s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
      s1 += __shfl_xor_sync(0xffffffffu, s1, 2); s2 += __shfl_xor_sync(0xffffffffu, s2, 2);
      if (q == 0 && live)
        *reinterpret_cast<float2*>(e.stats_out + ((size_t)(c.orow0 + tr + 8 * i) * (c.N >> 5) + ((c.col0 + c.ocol_add) >> 5)) * 2) = make_float2(s1, s2);
    }
  }
}

// any other Epilogue: run-time options (kept out of line: it is not on the denoiser's path)
__device__ __noinline__ void epi_rows_generic(const Epilogue& e, const Frag& f, const EpiRowCtx& c, int lane, const bool live) {
  const int tr = lane >> 2, tc2 = 2 * (lane & 3);
#pragma unroll 1
  for (int ij = 0; ij < 16; ++ij) {
    const int i = ij >> 2, j = ij & 3;
    const uint32_t* r = (i < 2) ? f.a : f.b;
    const int o = 4 * j + 2 * (i & 1);
    const int col = c.col0 + 8 * j + tc2, rr = tr + 8 * i;
    float v[2] = {__uint_as_float(r[o]), __uint_as_float(r[o + 1])};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      float x = v[k];
      if (e.bias) x += __ldg(e.bias + col + k);
      if (e.scale) x = x * __ldg(e.scale + col + k) + __ldg(e.shift + col + k);
      if (e.act == ACT_RELU) x = fmaxf(x, 0.f);
      else if (e.act == ACT_GELU) x = gelu_tanh_fast(x);
      else if (e.act == ACT_GELU_EXACT) x = gelu_tanh(x);
      else if (e.act == ACT_SIGMOID) x = sigmoidf_(x);
      if (e.pos) x += __ldg(e.pos + (size_t)(c.pos_row0 + rr) * c.N + col + k);
      if (e.gate) x *= __ldg(e.gate + col + k);
      if (e.resid) x += e.resid[(size_t)(c.res_row0 + rr) * e.ldr + col + k];
      v[k] = x;
    }
    const int orow = c.orow0 + rr, ocol = col + c.ocol_add;
    if (!live) continue;
    if (e.out) *reinterpret_cast<float2*>(e.out + (size_t)orow * e.ldc + ocol) = make_float2(v[0], v[1]);
    if (e.out_bf16) {
      const size_t off = (size_t)orow * e.ldc_bf16 + ocol;
      if (e.out_lo) {
        uint32_t hi, lo;
        split_bf16x2(v[0], v[1], hi, lo);
        *reinterpret_cast<uint32_t*>(e.out_bf16 + off) = hi;
        *reinterpret_cast<uint32_t*>(e.out_lo + off) = lo;
      } else {
        *reinterpret_cast<uint32_t*>(e.out_bf16 + off) = e.out_f16 ? pack_f16x2(v[0], v[1]) : pack_bf16x2(v[0], v[1]);
      }
    }
  }
}

// classification of an Epilogue (host): EPI_GENERIC when it is not one of the compiled combinations
static int classify_epilogue(const Epilogue& e) {
  int f = 0;
  if (e.scale) f |= EF_SCALE;
  if (e.act == ACT_RELU) f |= EF_FLOOR;
  else if (e.act == ACT_GELU) f |= EF_GELU;
  else if (e.act == ACT_GELU_EXACT) f |= EF_GELUX;
  else if (e.act != ACT_NONE) return EPI_GENERIC;
  if (e.gate) f |= EF_GATE;
  if (e.pos) f |= EF_POS;
  if (e.resid) f |= EF_RES;
  if (e.ln_stats) f |= EF_LN;
  int o;
  if (e.out && e.out_bf16 && e.stats_out && !(e.out_f16 && e.out_lo)) o = EO_F32X;      // 16-bit copy: bf16, bf16 pair or ONE fp16
  else if (e.stats_out) return EPI_GENERIC;                   // (rejected by the dispatcher: statistics need the compiled body)
  else if (e.out && !e.out_bf16) o = EO_F32;
  else if (!e.out && e.out_bf16) o = e.out_lo ? EO_PAIR : (e.out_f16 ? EO_F16 : EO_BF16);
  else return EPI_GENERIC;
  const int k = epi_key(f, o);
  switch (k) {
    case epi_key(0, EO_F32): case epi_key(0, EO_BF16): case epi_key(0, EO_PAIR): case epi_key(0, EO_F16):
    case epi_key(EF_POS, EO_BF16): case epi_key(EF_POS, EO_PAIR):
    case epi_key(EF_RES, EO_F32): case epi_key(EF_GATE | EF_RES, EO_F32):
    case epi_key(EF_GELU, EO_BF16): case epi_key(EF_GELUX, EO_PAIR):
    case epi_key(EF_SCALE | EF_FLOOR, EO_BF16): case epi_key(EF_SCALE | EF_FLOOR, EO_PAIR): case epi_key(EF_SCALE | EF_FLOOR | EF_RES, EO_F32):
    case epi_key(EF_FLOOR, EO_BF16): case epi_key(EF_FLOOR, EO_PAIR): case epi_key(EF_FLOOR, EO_F16):
    case epi_key(EF_LN, EO_F16): case epi_key(EF_LN, EO_BF16):
    case epi_key(EF_LN | EF_SCALE | EF_FLOOR, EO_PAIR): case epi_key(EF_LN | EF_SCALE | EF_FLOOR, EO_BF16):
    case epi_key(EF_RES, EO_F32X): case epi_key(EF_SCALE | EF_FLOOR | EF_RES, EO_F32X):
      return k;
    default:
      return EPI_GENERIC;
  }
}

// 16 TMEM lanes x 32 fp32 columns, mma-fragment layout (see Frag)
__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

struct PairUnit { int m0, n0, kb0, kb1; };
__device__ __forceinline__ PairUnit decode_unit(const PairParams& p, int u, int nkb, int bn) {
  PairUnit q;
  int mt, nt;
  if (p.late_tile0 > 0) {
    // q|k|v with a transposed V store: the V tiles' epilogue (2-byte scattered stores on top of the normal ones) is the slow one, so all
    // V tiles are dealt first - they land in the first wave, where the epilogue overlaps the pair's next main loop
    const int nv = p.tiles_n - p.late_tile0, first = nv * (p.M / (2 * PBM));
    if (u < first) { mt = u / nv; nt = p.late_tile0 + (u - mt * nv); }
    else { const int v = u - first; mt = v / p.late_tile0; nt = v - mt * p.late_tile0; }
  } else {
    mt = u / p.tiles_n; nt = u - mt * p.tiles_n;
  }
  q.m0 = mt * (2 * PBM); q.n0 = nt * bn;
  q.kb0 = 0; q.kb1 = nkb;
  return q;
}

// The epilogue warps' loop over the units of their pair (F < 0: generic run-time-option body).
template <int BN, int F, int O>
__device__ __forceinline__ void epilogue_loop(const PairParams& p, const Epilogue& e, uint32_t tmem_base, uint64_t* acc_full, uint64_t* acc_empty,
                                              int warp, int lane, uint32_t rank, int pair, int nkb) {
  constexpr int FF = F < 0 ? 0 : F;
  const int quarter = warp & 3, half = (warp - PP_EPI_WARP0) >> 2;
  const uint32_t lead_acc_empty0 = mapa(smem_u32(&acc_empty[0]), 0);
  constexpr int NCH = BN / 64;                               // 32-column chunks per warp and unit
  int it = 0;
  for (int u = pair; u < p.units; u += p.npairs, ++it) {
    const PairUnit q = decode_unit(p, u, nkb, BN);
    const int buf = it & 1;
    const int rbase = q.m0 + (int)rank * PBM + quarter * 32;  // first global row of this warp
    // row bookkeeping once per unit (the 32 rows of a warp never straddle a residual / pos-embed / stream boundary: the host checks
    // that those periods are multiples of 128), so the per-row work is address increments only
    EpiRowCtx rc;
    rc.res_row0 = e.resid_mod ? rbase % e.resid_mod : rbase;
    rc.pos_row0 = e.pos_rows ? rbase % e.pos_rows : 0;
    rc.orow0 = rbase; rc.ocol_add = 0; rc.N = p.N;
    if (e.group_rows) { rc.orow0 = rbase % e.group_rows; rc.ocol_add = (rbase / e.group_rows) * e.group_col_stride; }
    rc.col0 = q.n0 + half * (BN / 2);
    EpiLoads<FF> cur, nxt;
    if (F >= 0) epi_load<FF>(e, rc, lane, cur);               // first chunk's operands: in flight while the main loop still runs
    LnRows ln;
    if (FF & EF_LN) {
      // fused LayerNorm: lane r sums the partial (sum, sum of squares) of row rbase + r in chunk order (deterministic), then every
      // thread fetches the mean / rstd of its four rows
      const float4* sp = reinterpret_cast<const float4*>(e.ln_stats + (size_t)(rbase + lane) * e.ln_chunks * 2);
      float s1 = 0.f, s2 = 0.f;
      for (int k = 0; k < (e.ln_chunks >> 1); ++k) { const float4 t = __ldg(sp + k); s1 += t.x; s2 += t.y; s1 += t.z; s2 += t.w; }
      const float inv_c = 1.0f / (float)(e.ln_chunks * 32);
      const float mean = s1 * inv_c;
      const float rstd = rsqrtf(fmaxf(s2 * inv_c - mean * mean, 0.f) + e.ln_eps);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        ln.m[i] = __shfl_sync(0xffffffffu, mean, (lane >> 2) + 8 * i);
        ln.rs[i] = __shfl_sync(0xffffffffu, rstd, (lane >> 2) + 8 * i);
      }
    }
    const uint32_t tacc = tmem_base + buf * BN + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * (BN / 2));
    // The chunk body is ONE copy of code run NCH times (not unrolled), and the pair's first unit runs it once more up front as a
    // dry pass (pass -1: garbage accumulator, stores predicated off) while the main loop is still busy.  A launch executes an
    // epilogue body it has not run for ~100 us; the instruction fetch of the cold, straight-line code took 3.3 us per chunk inside a
    // step against 0.6 us in a back-to-back micro-benchmark (tools/step_trace.py: conv1's 4 chunks 14 us vs 2.8 us) - the dry pass
    // pulls the body into the instruction caches for free.
#pragma unroll 1
    for (int pass = (it == 0 ? -1 : 0); pass < NCH; ++pass) {
      const bool live = pass >= 0;
      const int ch = live ? pass : 0;
      if (pass == 0) {
        mbar_wait(&acc_full[buf], (it >> 1) & 1);
        if (warp == PP_EPI_WARP0 && lane == 0 && it < 2) PTRACE(4 + 5 * it);          // accumulator complete
        fence_after_sync();
      }
      rc.col0 = q.n0 + half * (BN / 2) + ch * 32;
      Frag f;
      tmem_ld_16x256b_x4(tacc + (uint32_t)(ch * 32), f.a);
      tmem_ld_16x256b_x4(tacc + (16u << 16) + (uint32_t)(ch * 32), f.b);
      if (F >= 0 && live && ch + 1 < NCH) {                   // next chunk's operands
        EpiRowCtx rn = rc; rn.col0 = rc.col0 + 32;
        epi_load<FF>(e, rn, lane, nxt);
      }
      tmem_ld_wait();
      if (live && warp == PP_EPI_WARP0 && lane == 0 && it == 0 && ch == 0) PTRACE(7);
      if (live && ch == NCH - 1) {                            // accumulator fully copied out: hand the buffer back to the MMA warp
        if (warp == PP_EPI_WARP0 && lane == 0 && it < 2) PTRACE(5 + 5 * it);      // TMEM drained
        fence_before_sync();
        __syncwarp();
        // (nobody waits for the buffers of a pair's last two units)
        if (lane == 0 && u + 2 * p.npairs < p.units) mbar_arrive_cluster(lead_acc_empty0 + (uint32_t)buf * 8u);
      }
      if (e.vt_out && rc.col0 >= e.vt_col0) {
        // transposed V^T [sample][column][token] (bias-only epilogue, host check): per column the 8 threads of equal t%4 write 8
        // consecutive tokens (16 bytes)
        const int tr = lane >> 2, tc2 = 2 * (lane & 3);
        uint16_t* vt = reinterpret_cast<uint16_t*>(e.vt_out);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int col = rc.col0 + 8 * j + tc2;
          const float2 b2 = e.bias ? __ldg(reinterpret_cast<const float2*>(e.bias + col)) : make_float2(0.f, 0.f);
          float2 c2 = make_float2(0.f, 0.f);
          if (FF & EF_LN) c2 = __ldg(reinterpret_cast<const float2*>(e.ln_colsum + col));
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int row = rbase + tr + 8 * i;
            float2 a = frag_val(f, i, j);
            if (FF & EF_LN) { a.x = ln.rs[i] * (a.x - ln.m[i] * c2.x); a.y = ln.rs[i] * (a.y - ln.m[i] * c2.y); }
            uint16_t* o = vt + ((size_t)(row >> 10) * (p.N - e.vt_col0) + (col - e.vt_col0)) * 1024 + (row & 1023);
            if (live) {
              o[0] = cvt16(a.x + b2.x, e.out_f16);
              o[1024] = cvt16(a.y + b2.y, e.out_f16);
            }
          }
        }
      }
      if (F >= 0) epi_rows<FF, O>(e, f, rc, lane, cur, ln, live);
      else epi_rows_generic(e, f, rc, lane, live);
      if (live && warp == PP_EPI_WARP0 && lane == 0 && it == 0 && ch == 0) PTRACE(11);
      if (F >= 0 && live && ch + 1 < NCH) cur = nxt;
    }
    if (warp == PP_EPI_WARP0 && lane == 0 && it < 2) PTRACE(6 + 5 * it);          // epilogue of the unit done (this warp)
  }
}

template <int BN, int MODE, bool CONV>
__global__ void __launch_bounds__(PP_THREADS, 1)
k_gemm_pair(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmAl, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmBl, const PairParams p, const Epilogue e) {
  using Cfg = PairCfg<BN, MODE>;
  constexpr int ST = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + Cfg::RING_BYTES);
  uint64_t* empty = full + ST;
  uint64_t* acc_full = empty + ST;        // 2
  uint64_t* acc_empty = acc_full + 2;     // 2 (the leader's are used)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();                   // 0 = leader
  const int pair = blockIdx.x >> 1;
  const int nkb = (p.K + PBK - 1) / PBK;

  pdl_trigger();
  if (threadIdx.x == 0) {
    PTRACE(0);                                               // CTA start
    prefetch_tmap(&tmA); prefetch_tmap(&tmB);
    if (MODE == 1) prefetch_tmap(&tmAl);
    if (MODE >= 1) prefetch_tmap(&tmBl);
    for (int s = 0; s < ST; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }       // full: the leader's arrive.expect_tx; both CTAs' TMA bytes
    for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 2 * PP_EPI_WARPS); }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc2(tmem_slot, Cfg::TMEM_COLS);
  fence_before_sync();
  cluster_sync_all();                                        // the barriers of BOTH CTAs exist before any remote arrive / TMA
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) PTRACE(1);                           // prologue done (the dependency wait follows per role)

  // (each role's code is dominated by its own setmaxnreg, so that ptxas applies the right register budget to it)
  if (warp >= PP_EPI_WARP0) {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(PP_REGS_EPI));
    // ===== epilogue warps (both CTAs): TMEM lane quarter = warp % 4, column half = (warp - 4) / 4
    pdl_wait();
#define DVD_EPI_CASE(F, O) case epi_key(F, O): epilogue_loop<BN, F, O>(p, e, tmem_base, acc_full, acc_empty, warp, lane, rank, pair, nkb); break;
    switch (p.epi) {
      DVD_EPI_CASE(0, EO_F32) DVD_EPI_CASE(0, EO_BF16) DVD_EPI_CASE(0, EO_PAIR) DVD_EPI_CASE(0, EO_F16)
      DVD_EPI_CASE(EF_POS, EO_BF16) DVD_EPI_CASE(EF_POS, EO_PAIR)
      DVD_EPI_CASE(EF_RES, EO_F32) DVD_EPI_CASE(EF_GATE | EF_RES, EO_F32)
      DVD_EPI_CASE(EF_GELU, EO_BF16) DVD_EPI_CASE(EF_GELUX, EO_PAIR)
      DVD_EPI_CASE(EF_SCALE | EF_FLOOR, EO_BF16) DVD_EPI_CASE(EF_SCALE | EF_FLOOR, EO_PAIR) DVD_EPI_CASE(EF_SCALE | EF_FLOOR | EF_RES, EO_F32)
      DVD_EPI_CASE(EF_FLOOR, EO_BF16) DVD_EPI_CASE(EF_FLOOR, EO_PAIR) DVD_EPI_CASE(EF_FLOOR, EO_F16)
      DVD_EPI_CASE(EF_LN, EO_F16) DVD_EPI_CASE(EF_LN, EO_BF16)
      DVD_EPI_CASE(EF_LN | EF_SCALE | EF_FLOOR, EO_PAIR) DVD_EPI_CASE(EF_LN | EF_SCALE | EF_FLOOR, EO_BF16)
      DVD_EPI_CASE(EF_RES, EO_F32X) DVD_EPI_CASE(EF_SCALE | EF_FLOOR | EF_RES, EO_F32X)
      default: epilogue_loop<BN, -1, 0>(p, e, tmem_base, acc_full, acc_empty, warp, lane, rank, pair, nkb); break;
    }
#undef DVD_EPI_CASE
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(PP_REGS_CTRL));
    if (warp == 0) {
      if (lane == 0) {
        // ===== TMA producer (both CTAs): own 128 A rows, own half of the W tile; the bytes of both CTAs are counted on the LEADER's full
        // barrier, which only the leader arrives on (expect_tx of both CTAs' bytes): a follower-side arrive per k-block would put a
        // cluster-scope fence on the producer's critical path.  The follower refills a stage only after ITS empty barrier fired, i.e. after
        // the previous phase of the leader's full barrier completed, so bytes never land in the wrong phase.
        // The W tiles do not depend on the previous kernel: the first ring-full of them is requested BEFORE griddepcontrol.wait, so that
        // under programmatic dependent launch the weight fetch (HBM: a step streams more weights than the L2 holds) overlaps the
        // predecessor's tail; the A tiles follow after the wait.
        uint32_t g = 0;
        const int cblocks = CONV ? p.conv_cin / 64 : 1;
        bool waited_pdl = false;
        for (int u = pair; u < p.units; u += p.npairs) {
          const PairUnit q = decode_unit(p, u, nkb, BN);
          const int m0 = q.m0 + (int)rank * PBM, nb = q.n0 + (int)rank * (BN / 2);
          int cn = 0, cy = 0, cx = 0;
          if (CONV) {
            const int hw = p.conv_h * p.conv_w;
            cn = m0 / hw; const int rem = m0 - cn * hw; cy = rem / p.conv_w; cx = rem - cy * p.conv_w;   // 128 consecutive pixels of one image row
          }
          auto load_b = [&](int kb, uint32_t gg) {
            const int s = gg % ST;
            uint8_t* a = smem + s * Cfg::STAGE_BYTES;
            const uint32_t lead_full = mapa(smem_u32(&full[s]), 0);
            if (rank == 0) mbar_expect_tx(&full[s], 2 * Cfg::STAGE_BYTES);        // both CTAs' loads of this stage
  #pragma unroll
            for (int o = 0; o < Cfg::NB; ++o) tma_load_2d_pair(a + Cfg::B_OFF + o * Cfg::B_BYTES, o ? &tmBl : &tmB, lead_full, kb * PBK, nb);
          };
          auto load_a = [&](int kb, uint32_t gg) {
            const int s = gg % ST;
            uint8_t* a = smem + s * Cfg::STAGE_BYTES;
            const uint32_t lead_full = mapa(smem_u32(&full[s]), 0);
  #pragma unroll
            for (int o = 0; o < Cfg::NA; ++o) {
              if (CONV) {
                const int tap = kb / cblocks, cb = kb - tap * cblocks;
                tma_load_4d_pair(a + o * Cfg::A_BYTES, o ? &tmAl : &tmA, lead_full, cb * 64, cx + tap % 3 - 1, cy + tap / 3 - 1, cn);
              } else {
                tma_load_2d_pair(a + o * Cfg::A_BYTES, o ? &tmAl : &tmA, lead_full, kb * PBK, m0);
              }
            }
          };
          int kb = q.kb0;
          if (!waited_pdl) {                                     // first unit: W tiles of the first ring-full ahead of the dependency wait
            const int npre = (q.kb1 - q.kb0) < ST ? (q.kb1 - q.kb0) : ST;
            for (int i = 0; i < npre; ++i) load_b(q.kb0 + i, g + i);
            pdl_wait();
            waited_pdl = true;
            for (int i = 0; i < npre; ++i) load_a(q.kb0 + i, g + i);
            kb += npre; g += npre;
          }
          for (; kb < q.kb1; ++kb, ++g) {
            mbar_wait(&empty[g % ST], ((g / ST) & 1) ^ 1);
            load_b(kb, g);
            load_a(kb, g);
          }
        }
        if (!waited_pdl) pdl_wait();
      } else {
        pdl_wait();
      }
      __syncwarp();
    } else if (warp == 1) {
      pdl_wait();
      if (rank == 0) {
        // ===== MMA issuer (leader only): UMMA M = 256 across the pair, accumulator buffer = unit parity.  The whole warp runs the loop
        // and one elected lane issues (tc_common.cuh: inside an `if (lane == 0)` region every UMMA costs an elect / branch loop).
        constexpr uint32_t idesc = MODE == 2 ? make_idesc_f16(2 * PBM, BN) : make_idesc_bf16(2 * PBM, BN);
        const uint32_t tbase = __shfl_sync(0xffffffffu, tmem_base, 0);       // warp-uniform for the compiler
        uint32_t g = 0;
        int it = 0;
        for (int u = pair; u < p.units; u += p.npairs, ++it) {
          const PairUnit q = decode_unit(p, u, nkb, BN);
          const int buf = it & 1;
          mbar_wait(&acc_empty[buf], ((it >> 1) & 1) ^ 1);       // both CTAs' epilogue warps have drained this accumulator
          fence_after_sync();
          const uint32_t tacc = tbase + buf * BN;
          for (int kb = q.kb0; kb < q.kb1; ++kb, ++g) {
            const int s = g % ST;
            mbar_wait(&full[s], (g / ST) & 1);
            if (lane == 0) {
              if (kb == q.kb0) if (it < 2) PTRACE(2 + 5 * it);              // first stage of the unit landed
              if (kb == q.kb1 - 1) if (it < 2) PTRACE(3 + 5 * it);          // last stage landed
            }
            fence_after_sync();
            const uint32_t a_addr = smem_u32(smem + s * Cfg::STAGE_BYTES);
            const uint64_t ad = make_desc_k_sw128(a_addr), bd = make_desc_k_sw128(a_addr + Cfg::B_OFF);   // start field: 16-byte units
  #pragma unroll
            for (int k = 0; k < PBK / 16; ++k) {
              const uint64_t ah = ad + (uint64_t)(k * 2), bh = bd + (uint64_t)(k * 2);
              mma_ss_pair_elect(tacc, ah, bh, idesc, (kb > q.kb0 || k > 0) ? 1u : 0u);
              if (MODE == 1) mma_ss_pair_elect(tacc, ah + (uint64_t)(Cfg::A_BYTES >> 4), bh, idesc, 1u);    // lo * hi
              if (MODE >= 1) mma_ss_pair_elect(tacc, ah, bh + (uint64_t)(Cfg::B_BYTES >> 4), idesc, 1u);    // hi * lo
            }
            mma_commit_pair_elect(&empty[s]);                    // frees stage s in both CTAs
          }
          mma_commit_pair_elect(&acc_full[buf]);                 // the accumulators of both CTAs are complete
        }
      }
      __syncwarp();
    }
  }
  if (threadIdx.x == 32 * PP_EPI_WARP0) PTRACE(14);                          // this CTA's epilogue warps are done
  fence_before_sync();
  cluster_sync_all();                                          // the peer's smem / TMEM must outlive every MMA that reads it
  if (warp == 1) tmem_dealloc2(tmem_base, Cfg::TMEM_COLS);
  if (threadIdx.x == 32) PTRACE(15);                          // exit
}

// ---------------------------------------------------------------------------------------- host side
static int g_force_bn = -1, g_debug = 0;
static void read_env() {
  if (g_force_bn >= 0) return;
  const char* b = getenv("DVD_GEMM_BN"); g_force_bn = b ? atoi(b) : 0;
  const char* d = getenv("DVD_GEMM_DEBUG"); g_debug = d ? atoi(d) : 0;
}

bool gemm_pair_supported(int M, int N, int K, bool conv) {
  (void)K; (void)conv;
  return M % 256 == 0 && N % 64 == 0;
}
// the epilogue computes residual / pos-embed / stream-concat row offsets once per 32-row group
static bool epilogue_periods_ok(const Epilogue& e) {
  return (e.resid_mod % 128 == 0) && (e.pos_rows % 128 == 0) && (e.group_rows % 128 == 0);
}

template <int BN, int MODE, bool CONV>
static int max_pairs() {           // co-resident clusters of this instantiation on the current device (cached per device)
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
  if (cached[dev]) return cached[dev];
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * 256); cfg.blockDim = dim3(PP_THREADS); cfg.dynamicSmemBytes = PairCfg<BN, MODE>::SMEM;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, k_gemm_pair<BN, MODE, CONV>, &cfg) != cudaSuccess || n <= 0) { cudaGetLastError(); n = sm_count() / 2 - 2; }
  if (n > sm_count() / 2) n = sm_count() / 2;
  cached[dev] = n;
  return n;
}

// Cycle model used to pick the tile width.  Per k-block and CTA: tensor time (UMMA 256 x bn x 16 on a pair = bn/2 clocks, 4 per k-block,
// x3 in split-precision mode) against the L2 -> SM operand stream (~43 B/clk per SM when every SM pulls: 12.5 TB/s measured with
// tools/gemm_trace.py).  Per unit a fixed pipeline-fill cost, per launch the exposed last epilogue.  Calibrated against
// profiles/r2_gemm_sweep.txt (all denoiser shapes x {128,192,256}).
static double unit_kb_cycles(int bn, int mode) {
  const double mma = (mode == 1 ? 3.0 : mode == 2 ? 2.0 : 1.0) * 4.0 * (bn / 2.0) * 1.15;
  const double bytes = (mode == 1 ? 2.0 : 1.0) * 16384.0 + (mode >= 1 ? 2.0 : 1.0) * bn * 64.0;
  const double mem = bytes / 43.0;
  return mma > mem ? mma : mem;
}

static int pick_bn(int M, int N, int K, int mode, int npairs) {
  const int nkb = (K + PBK - 1) / PBK;
  double best = -1.0;
  int bn_out = 64;
  const int bns[4] = {256, 192, 128, 64};
  for (int bi = 0; bi < 4; ++bi) {
    const int bn = bns[bi];
    if (N % bn) continue;
    if (g_force_bn > 0 && bn != g_force_bn && N % g_force_bn == 0) continue;
    const long long units = (long long)(M / 256) * (N / bn);
    const long long waves = (units + npairs - 1) / npairs;
    const double cost = waves * (nkb * unit_kb_cycles(bn, mode) + 700.0) + (900.0 + 9.0 * bn);
    if (best < 0 || cost < best) { best = cost; bn_out = bn; }
  }
  return bn_out;
}

template <int BN, int MODE, bool CONV>
static int launch_pair(const TcMat& A, const TcMat& W, int M, int N, int K, const Epilogue& e, int conv_b, int conv_h, int conv_w, int conv_cin,
                       cudaStream_t st) {
  using Cfg = PairCfg<BN, MODE>;
  auto kern = k_gemm_pair<BN, MODE, CONV>;
  DVD_SET_MAX_SMEM(kern, Cfg::SMEM);
  const int npairs_max = max_pairs<BN, MODE, CONV>();
  DVD_REQUIRE(npairs_max > 0, "gemm_pair: no co-resident cluster available");
  CUtensorMap tmA, tmB, tmAl, tmBl;
  int rc;
  if (CONV) rc = make_tmap_bf16_nhwc(&tmA, A.hi, (uint64_t)conv_b, (uint64_t)conv_h, (uint64_t)conv_w, (uint64_t)conv_cin);
  else rc = make_tmap_bf16_2d(&tmA, A.hi, (uint64_t)M, (uint64_t)K, (uint64_t)A.ld, 128, 64);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmB, W.hi, (uint64_t)N, (uint64_t)K, (uint64_t)W.ld, (uint32_t)(BN / 2), 64); if (rc) return rc;
  tmAl = tmA; tmBl = tmB;
  if (MODE == 1) {
    if (CONV) rc = make_tmap_bf16_nhwc(&tmAl, A.lo, (uint64_t)conv_b, (uint64_t)conv_h, (uint64_t)conv_w, (uint64_t)conv_cin);
    else rc = make_tmap_bf16_2d(&tmAl, A.lo, (uint64_t)M, (uint64_t)K, (uint64_t)A.ld, 128, 64);
    if (rc) return rc;
  }
  if (MODE >= 1) {
    rc = make_tmap_bf16_2d(&tmBl, W.lo, (uint64_t)N, (uint64_t)K, (uint64_t)W.ld, (uint32_t)(BN / 2), 64); if (rc) return rc;
  }
  PairParams p;
  p.M = M; p.N = N; p.K = K;
  p.tiles_n = N / BN;
  const long long units = (long long)(M / 256) * p.tiles_n;
  DVD_REQUIRE(units < (1LL << 31), "gemm_pair: too many work units");
  p.units = (int)units;
  p.npairs = units < npairs_max ? (int)units : npairs_max;
  p.conv_h = conv_h; p.conv_w = conv_w; p.conv_cin = conv_cin;
  p.epi = classify_epilogue(e);
  p.late_tile0 = (e.vt_out && e.vt_col0 > 0 && e.vt_col0 % BN == 0 && e.vt_col0 < N) ? e.vt_col0 / BN : 0;
  if (g_debug) fprintf(stderr, "[gemm_pair] M=%d N=%d K=%d mode=%d conv=%d bn=%d units=%d npairs=%d (max %d) stages=%d smem=%d\n", M, N, K,
                       MODE, (int)CONV, BN, p.units, p.npairs, npairs_max, Cfg::STAGES, Cfg::SMEM);
  DVD_CUDA(launch_pdl_cluster(1, kern, dim3(2 * p.npairs), dim3(PP_THREADS), (size_t)Cfg::SMEM, st, 2, 1, tmA, tmAl, tmB, tmBl, p, e));
  DVD_LAUNCH_CHECK("k_gemm_pair");
  return 0;
}

template <int MODE, bool CONV>
static int launch_pair_bn(int bn, const TcMat& A, const TcMat& W, int M, int N, int K, const Epilogue& e, int conv_b, int conv_h, int conv_w,
                          int conv_cin, cudaStream_t st) {
  switch (bn) {
    case 256: return launch_pair<256, MODE, CONV>(A, W, M, N, K, e, conv_b, conv_h, conv_w, conv_cin, st);
    case 192: return launch_pair<192, MODE, CONV>(A, W, M, N, K, e, conv_b, conv_h, conv_w, conv_cin, st);
    case 128: return launch_pair<128, MODE, CONV>(A, W, M, N, K, e, conv_b, conv_h, conv_w, conv_cin, st);
    default:  return launch_pair<64, MODE, CONV>(A, W, M, N, K, e, conv_b, conv_h, conv_w, conv_cin, st);
  }
}

// A: 2-D [M,K] or, when conv_h > 0, NHWC [B,H,W,Cin] with K = 9*Cin; W: [N,K] K-major.  W must not be written by the kernel that
// immediately precedes this launch in the stream if that kernel triggers programmatic dependent launch (the weight tiles are
// requested ahead of griddepcontrol.wait); the denoiser's weights are static.
int gemm_pair_dispatch(const TcMat& A, const TcMat& W, int M, int N, int K, const Epilogue& e, int conv_b, int conv_h, int conv_w, int conv_cin,
                       cudaStream_t st) {
  read_env();
  const bool conv = conv_h > 0;
  const int mode = A.lo ? 1 : (A.f16 ? 2 : 0);
  DVD_REQUIRE(mode == 0 || W.lo, "gemm_pair: the weight's low half is missing");
  DVD_REQUIRE(gemm_pair_supported(M, N, K, conv), "gemm_pair: unsupported shape M=%d N=%d K=%d", M, N, K);
  DVD_REQUIRE(epilogue_periods_ok(e), "gemm_pair: resid_mod / pos_rows / group_rows must be multiples of 128");
  DVD_REQUIRE((!e.ln_stats && !e.stats_out) || classify_epilogue(e) != EPI_GENERIC, "gemm_pair: fused-LN / row-statistics epilogue combination not compiled");
  DVD_REQUIRE(!e.ln_stats || (e.ln_colsum && e.ln_chunks > 0 && e.ln_chunks % 2 == 0 && (reinterpret_cast<uintptr_t>(e.ln_stats) & 15) == 0),
              "gemm_pair: fused LN needs ln_colsum and an even number of 32-column chunks");
  DVD_REQUIRE(!e.stats_out || (N % 32 == 0 && !e.group_rows), "gemm_pair: row statistics need N %% 32 == 0 and no stream remap");
  DVD_REQUIRE(!conv || (conv_w % 128 == 0 && conv_cin % 64 == 0 && K == 9 * conv_cin), "gemm_pair: bad conv geometry");
  DVD_REQUIRE(!e.out_bf16 || (e.ldc_bf16 % 8 == 0 && e.group_col_stride % 8 == 0 && (reinterpret_cast<uintptr_t>(e.out_bf16) & 15) == 0 &&
                              (reinterpret_cast<uintptr_t>(e.out_lo) & 15) == 0),
              "gemm_pair: 16-bit outputs are stored 16 bytes at a time (ld %% 8, 16-byte aligned bases)");
  DVD_REQUIRE(!conv || mode != 1, "gemm_pair: the implicit convolution takes a bf16 activation or an fp16 one, not a split pair");
  const int bn = pick_bn(M, N, K, mode, sm_count() / 2);
  if (conv) return mode == 2 ? launch_pair_bn<2, true>(bn, A, W, M, N, K, e, conv_b, conv_h, conv_w, conv_cin, st)
                             : launch_pair_bn<0, true>(bn, A, W, M, N, K, e, conv_b, conv_h, conv_w, conv_cin, st);
  if (mode == 2) return launch_pair_bn<2, false>(bn, A, W, M, N, K, e, 0, 0, 0, 0, st);
  return mode ? launch_pair_bn<1, false>(bn, A, W, M, N, K, e, 0, 0, 0, 0, st)
              : launch_pair_bn<0, false>(bn, A, W, M, N, K, e, 0, 0, 0, 0, st);
}

}  // namespace dvd

#ifdef DVD_GEMM_TRACE
extern "C" __attribute__((visibility("default"))) int dvd_debug_pair_trace_filter(int n) {
  return (int)cudaMemcpyToSymbol(dvd::g_pair_trace_n, &n, sizeof(int));
}
extern "C" __attribute__((visibility("default"))) int dvd_debug_pair_trace(unsigned long long* out, int n_ctas) {
  return (int)cudaMemcpyFromSymbol(out, dvd::g_pair_trace, (size_t)n_ctas * 16 * sizeof(unsigned long long));
}
#endif
