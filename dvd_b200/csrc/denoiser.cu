// Host-side orchestration of the denoiser forward and the DDIM loop (all launches asynchronous on
// the caller's stream, no allocation, no sync -> CUDA-graph capturable).
//
// What is hoisted relative to the reference (SURVEY.md §2.3):
//   * DiT blocks 0..10 are never executed (their outputs are discarded at CM:614-616).
//   * pyramid, c/m/l patch embeds and the cross-attention K/V of the three static contexts run
//     once per DOCUMENT (dvd_static_forward), not once per step and hypothesis.
//   * the cross-attention query LN(x)*Wq is computed once, not four times (CM:237-265).
//   * timestep MLP / adaLN projections come from a precomputed table (dvd_tables_init).
//   * the DDIM posterior update is the 2-scalar epilogue of the final layer (GD:445-491, eta=0).
#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "misc.cuh"
#include <string.h>
#include <vector>

namespace dvd {

struct B16 { __nv_bfloat16* hi = nullptr; __nv_bfloat16* lo = nullptr; };

struct Workspace {
  // static, per document
  float *y4, *pyrP, *pyrQ, *feat, *a_stat, *ctx[3], *kv_static[3];
  // per step
  float *a_r, *xe, *r, *qn, *q, *kv_r, *xo, *xs, *hmod, *qkv, *h1, *X, *pe, *hd, *qkv_d, *att_d, *f1, *f2, *S;
  float *flow[2], *xbuf[2], *pred;
  float* final_flow;                       // [docs * n_hyp, 2, 64, 64]: last pred_xstart of every hypothesis (input of the mean)
  // 16-bit GEMM operand staging (tensor modes): plain bf16, or bf16 hi + lo pairs in DVD_PREC_BF16X3
  B16 a_stat16, ctx16[3], a_r16, r16, qn16, xo16, hmod16, h116, hd16, att_d16, f116, f216;
  B16 X16;                                 // decoder residual stream as a GEMM operand (fused-LayerNorm path, DVD_PREC_BF16X3)
  float* lnstats;                          // [M][48][2] partial row statistics of X for the LayerNorm fused into the next GEMM
  // attention operands: bf16 (DVD_PREC_BF16) or fp16 (DVD_PREC_BF16X3)
  __nv_bfloat16 *q16, *kv_static16[3], *kv_r16, *qkv16, *qkv_d16;       // Q, K row-major
  __nv_bfloat16 *vt_static16[3], *vt_r16, *vt_qkv16, *vt_d16;            // V^T [sample, C_v, 1024] written by the GEMM epilogues
  size_t s_floats;
  size_t step_off;                         // offset of the per-step region
  size_t total_bytes;
};

constexpr size_t kSChunkSamples = 8;      // (sample, 6 heads) pairs per fp32 attention chunk

struct Carver {
  char* base; size_t off;
  char* take(size_t bytes) { size_t o = off; off += (bytes + 255) & ~size_t(255); return base ? base + o : nullptr; }
  float* F(size_t n) { return (float*)take(n * 4); }
  __nv_bfloat16* H(size_t n) { return (__nv_bfloat16*)take(n * 2); }
  B16 P(size_t n, bool pair) { B16 b; b.hi = H(n); b.lo = pair ? H(n) : nullptr; return b; }
};

// per-document buffers (written by static_forward, read by every step of every hypothesis) + the gathered final flows
static void carve_static(Carver& k, Workspace& w, int docs, int n_hyp, bool tc, bool x3) {
  const size_t Md = (size_t)docs * 1024;
  w.y4 = k.F((size_t)docs * 512 * 512 * 4);
  w.pyrP = k.F((size_t)docs * 512 * 512 * 64);
  w.pyrQ = k.F((size_t)docs * 512 * 512 * 64);
  w.feat = k.F((size_t)docs * 4096 * 256);
  w.a_stat = k.F(Md * 1536);
  for (int i = 0; i < 3; ++i) w.ctx[i] = k.F(Md * 384);
  for (int i = 0; i < 3; ++i) w.kv_static[i] = k.F(Md * 768);
  w.final_flow = k.F((size_t)docs * n_hyp * 8192);
  if (tc) {
    w.a_stat16 = k.P(Md * 1536, x3);
    for (int i = 0; i < 3; ++i) w.ctx16[i] = k.P(Md * 384, x3);
    for (int i = 0; i < 3; ++i) w.kv_static16[i] = k.H(Md * 768);
    for (int i = 0; i < 3; ++i) w.vt_static16[i] = k.H(Md * 384);
  }
}

// per-step buffers of a group of docs * n_hyp samples
static void carve_step(Carver& k, Workspace& w, int docs, int n_hyp, bool tc, bool x3) {
  const size_t N = (size_t)docs * n_hyp, M = N * 1024;
  w.a_r = k.F(M * 1032);
  w.xe = k.F(M * 384); w.r = k.F(M * 384); w.qn = k.F(M * 384); w.q = k.F(M * 384);
  w.kv_r = k.F(M * 768);
  w.xo = k.F(4 * M * 384); w.xs = k.F(4 * M * 384); w.hmod = k.F(4 * M * 384);
  w.qkv = k.F(4 * M * 1152);
  w.h1 = k.F(4 * M * 1536);
  w.X = k.F(M * 1536);
  w.pe = k.F(N * 1536 * (1 + 32 + 4));      // mean | 32 partials | hs1 hs ws1 ws
  w.hd = k.F(M * 1536); w.qkv_d = k.F(M * 4608); w.att_d = k.F(M * 1536);
  w.f1 = k.F(M * 2048); w.f2 = k.F(M * 2048);
  size_t chunk = N < kSChunkSamples ? N : kSChunkSamples;
  w.s_floats = tc ? 0 : (size_t)4 * chunk * kHeads * 1024 * 1024;        // up to 4 streams x chunk samples
  w.S = k.F(w.s_floats);
  for (int i = 0; i < 2; ++i) { w.flow[i] = k.F(N * 8192); w.xbuf[i] = k.F(N * 8192); }
  w.pred = k.F(N * 8192);
  if (tc) {
    w.a_r16 = k.P(M * 1032, x3);
    w.r16 = k.P(M * 384, x3); w.qn16 = k.P(M * 384, x3); w.xo16 = k.P(4 * M * 384, x3); w.hmod16 = k.P(4 * M * 384, x3);
    w.h116 = k.P(4 * M * 1536, x3); w.hd16 = k.P(M * 1536, x3); w.att_d16 = k.P(M * 1536, x3); w.f116 = k.P(M * 2048, x3);
    w.f216 = k.P(M * 2048, x3);
    w.q16 = k.H(M * 384); w.kv_r16 = k.H(M * 768); w.qkv16 = k.H(4 * M * 1152); w.qkv_d16 = k.H(M * 4608);
    w.vt_r16 = k.H(M * 384); w.vt_qkv16 = k.H(4 * M * 384); w.vt_d16 = k.H(M * 1536);
    if (x3) { w.X16 = k.P(M * 1536, true); w.lnstats = k.F(M * 48 * 2); }
  }
}

static Workspace carve(void* base, int docs, int n_hyp, int precision) {
  Workspace w{};
  const bool tc = precision != DVD_PREC_FP32, x3 = precision == DVD_PREC_BF16X3;
  Carver k{(char*)base, 0};
  carve_static(k, w, docs, n_hyp, tc, x3);
  w.step_off = k.off;
  carve_step(k, w, docs, n_hyp, tc, x3);
  w.total_bytes = k.off;
  return w;
}

// ------------------------------------------------------------------------------------------ fp32 attention (GEMM + softmax + GEMM)
// q/k/v are row-major with leading dims ldq/ldk/ldv; head h occupies columns [h*d, (h+1)*d).
// sample n of q/o uses rows [n*T, (n+1)*T); k/v use sample n / kv_div.
static int attention_f32(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, float* o, int ldo, int nsamp,
                         int heads, int T, int d, float scale, int kv_div, float* S, size_t s_floats, cudaStream_t st) {
  size_t per = (size_t)heads * T * T;
  size_t chunk = s_floats / per;
  DVD_REQUIRE(chunk >= (size_t)kv_div, "attention_f32: scratch too small");
  chunk = (chunk / kv_div) * kv_div;
  for (size_t n0 = 0; n0 < (size_t)nsamp; n0 += chunk) {
    int nc = (int)(((size_t)nsamp - n0) < chunk ? (size_t)nsamp - n0 : chunk);
    GemmParams p;
    p.A = q + n0 * T * ldq; p.lda = ldq; p.sAn = (long long)T * ldq; p.sAh = d;
    p.B = k + (n0 / kv_div) * T * ldk; p.ldb = ldk; p.sBn = (long long)T * ldk; p.sBh = d; p.bdiv = kv_div;
    p.M = T; p.N = T; p.K = d; p.heads = heads; p.alpha = scale;
    p.e.out = S; p.e.ldc = T; p.sCn = (long long)per; p.sCh = (long long)T * T;
    int rc = gemm_f32(p, A_DIRECT, B_NK, nc * heads, st);
    if (rc) return rc;
    rc = softmax_rows(S, (long long)nc * heads * T, T, st);
    if (rc) return rc;
    GemmParams g;
    g.A = S; g.lda = T; g.sAn = (long long)per; g.sAh = (long long)T * T;
    g.B = v + (n0 / kv_div) * T * ldv; g.ldb = ldv; g.sBn = (long long)T * ldv; g.sBh = d; g.bdiv = kv_div;
    g.M = T; g.N = d; g.K = T; g.heads = heads;
    g.e.out = o + n0 * T * ldo; g.e.ldc = ldo; g.sCn = (long long)T * ldo; g.sCh = d;
    rc = gemm_f32(g, A_DIRECT, B_KN, nc * heads, st);
    if (rc) return rc;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------ kernel-class profiler
// When enabled (dvd_profile_begin) every dense contraction is bracketed by CUDA events on the launch stream so that
// bench.py can report the share and the achieved FLOP/s of each kernel class measured inside a real step.
enum { PC_GEMM = 0, PC_ATTN = 1, PC_CONV = 2, PC_COUNT = 3 };
struct Profiler {
  bool on = false;
  std::vector<cudaEvent_t> ev[PC_COUNT];      // start/stop pairs
  double flops[PC_COUNT] = {0, 0, 0};         // algorithmic (2 M N K)
  double exec_flops[PC_COUNT] = {0, 0, 0};    // what the tensor pipe executes: x3 / x2 in the split-precision passes
  long long launches[PC_COUNT] = {0, 0, 0};
};
static thread_local Profiler g_prof;
struct ProfScope {
  int cls; cudaStream_t st; bool on;
  ProfScope(int c, cudaStream_t s, double flops, int passes = 1) : cls(c), st(s), on(g_prof.on) {
    if (!on) return;
    cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); g_prof.ev[cls].push_back(e);
    g_prof.flops[cls] += flops; g_prof.exec_flops[cls] += flops * passes; g_prof.launches[cls] += 1;
  }
  ~ProfScope() {
    if (!on) return;
    cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); g_prof.ev[cls].push_back(e);
  }
};

// ------------------------------------------------------------------------------------------ precision dispatch helpers
struct Ctx {
  const dvd_weights_t* w;
  Workspace ws;
  int docs, n_hyp, prec;
  cudaStream_t st;
  bool tc() const { return prec != DVD_PREC_FP32; }
  bool x3() const { return prec == DVD_PREC_BF16X3; }
};

// 16-bit destinations of an epilogue: the operand of the next GEMM (plain bf16 or split pair) ...
static void out_operand(Epilogue& e, const B16& dst, int ld) { e.out_bf16 = dst.hi; e.out_lo = dst.lo; e.ldc_bf16 = ld; }
// ... or an operand of the attention kernel (bf16, fp16 in the split-precision mode)
static void out_attn(const Ctx& c, Epilogue& e, __nv_bfloat16* dst, int ld) { e.out_bf16 = dst; e.out_lo = nullptr; e.ldc_bf16 = ld; e.out_f16 = c.x3() ? 1 : 0; }

// C = epi(A * W[row0 : row0+N, :]^T)
// a_f16 (DVD_PREC_BF16X3 only): A16.hi holds ONE fp16 value per element -> two tensor passes (fp16 A x weight hi, x weight lo)
static int linear(const Ctx& c, const float* A32, const B16& A16, int lda, const dvd_mat_t& W, int row0, int M, int N,
                  const Epilogue& e, bool a_f16 = false) {
  ProfScope ps(PC_GEMM, c.st, 2.0 * M * N * W.k, c.x3() ? (a_f16 ? 2 : 3) : 1);
  if (c.tc()) {
    DVD_REQUIRE(A16.hi && W.bf16 && (!c.x3() || ((A16.lo || a_f16) && W.bf16_lo)), "linear: 16-bit operands missing");
    TcMat a, w;
    a.hi = A16.hi; a.lo = (c.x3() && !a_f16) ? A16.lo : nullptr; a.ld = lda; a.f16 = c.x3() && a_f16;
    w.hi = (const __nv_bfloat16*)W.bf16 + (size_t)row0 * W.k; w.ld = W.k;
    w.lo = c.x3() ? (const __nv_bfloat16*)W.bf16_lo + (size_t)row0 * W.k : nullptr;
    return gemm_tc(a, w, M, N, W.k, e, c.st);
  }
  GemmParams p = linear_params(A32, lda, W.f32 + (size_t)row0 * W.k, M, N, W.k);
  p.e = e;
  return gemm_f32(p, A_DIRECT, B_NK, 1, c.st);
}

#define DVD_TRY(x) do { int _rc = (x); if (_rc) return _rc; } while (0)

static int conv3x3(const Ctx& c, const float* in, float* out, int B, int H, int W, int Cin, const dvd_mat_t& Wt, const float* bias) {
  // fp32 mode: implicit GEMM on the FFMA path
  ProfScope ps(PC_CONV, c.st, 2.0 * B * H * W * Wt.n * 9.0 * Cin);
  GemmParams p;
  p.A = in; p.convH = H; p.convW = W; p.convC = Cin;
  p.B = Wt.f32; p.ldb = 9 * Cin; p.M = B * H * W; p.N = Wt.n; p.K = 9 * Cin;
  p.e.bias = bias; p.e.act = ACT_RELU; p.e.out = out; p.e.ldc = Wt.n;
  return gemm_f32(p, A_CONV3, B_NK, 1, c.st);
}

static TcMat weight_op(const Ctx& c, const dvd_mat_t& W) {
  TcMat w;
  w.hi = (const __nv_bfloat16*)W.bf16; w.lo = c.x3() ? (const __nv_bfloat16*)W.bf16_lo : nullptr; w.ld = W.k;
  return w;
}

static int static_forward(const Ctx& c, const float* y512, const float* mask_cat, const float* mask_y512, const float* line_msk) {
  const dvd_weights_t& w = *c.w; const Workspace& s = c.ws; cudaStream_t st = c.st;
  const int B = c.docs, Md = B * 1024;
  const bool tc = c.tc(), x3 = c.x3();
  // ---- K1 pyramid (CM:83-95): 7 x conv3x3+ReLU, 3 x maxpool, NHWC
  DVD_TRY(pack_y4(y512, mask_cat, s.y4, B, st));
  if (tc) {
    // level_0 (Cin = 4): the 3x3x4 patch of every pixel is written once as a K = 64 (36 valid + zero padding) 16-bit row
    // (im2col, 128 B per pixel) and multiplied by the K-padded weight on tcgen05; the six wide convs run as implicit GEMMs
    // directly on the NHWC activations; the last pool writes the fp32 feature map the rest of the model consumes.
    // DVD_PREC_BF16X3 runs on the fp16 weight pairs (dvd_weights_t::pyr_h): the activations are ONE fp16 value per element and every
    // conv runs two tensor passes (oracle/precision_study.py --two-pass: "only pyramid: fp16 activation x weight pair" moves the final
    // map by nothing measurable, 1.25e-6 vs 1.44e-6 for bf16 pairs on both sides).
    const int passes = x3 ? 2 : 1, pf = x3 ? 1 : 0;
    __nv_bfloat16* P = (__nv_bfloat16*)s.pyrP;
    __nv_bfloat16* Q = (__nv_bfloat16*)s.pyrQ;
    auto op = [&](__nv_bfloat16* a) { TcMat m; m.hi = a; m.ld = 64; m.f16 = x3; return m; };
    auto wop = [&](int layer) {
      if (!x3) return weight_op(c, w.pyr[layer]);
      TcMat m; m.hi = (const __nv_bfloat16*)w.pyr_h[layer].bf16; m.lo = (const __nv_bfloat16*)w.pyr_h[layer].bf16_lo; m.ld = w.pyr_h[layer].k;
      return m;
    };
    auto out16 = [&](Epilogue& e, __nv_bfloat16* dst, int ld) { e.out_bf16 = dst; e.ldc_bf16 = ld; e.out_f16 = pf; };
    {
      ProfScope ps(PC_CONV, st, 2.0 * B * 512 * 512 * 64 * 36.0, passes);
      TcMat wt = wop(0); wt.ld = 64;
      DVD_REQUIRE(wt.hi && (!x3 || wt.lo), "pyramid level_0 16-bit (K-padded) weight missing");
      DVD_TRY(im2col3x3_c4_bf16(s.y4, Q, B, 512, 512, st, pf));     // Q: [B*512*512, 64]
      Epilogue e; e.bias = w.pyr_b[0]; e.act = ACT_RELU; out16(e, P, 64);
      DVD_TRY(gemm_tc(op(Q), wt, B * 512 * 512, 64, 64, e, st));
    }
    auto conv = [&](__nv_bfloat16* in, __nv_bfloat16* out, int H, int Cin, int layer) -> int {
      const int Cout = w.pyr[layer].n;
      ProfScope ps(PC_CONV, st, 2.0 * B * H * H * Cout * 9.0 * Cin, passes);
      Epilogue e; e.bias = w.pyr_b[layer]; e.act = ACT_RELU; out16(e, out, Cout);
      const TcMat wt = wop(layer);
      DVD_REQUIRE(wt.hi && (!x3 || wt.lo), "pyramid 16-bit weights missing");
      return conv3x3_tc(op(in), wt, B, H, H, Cin, Cout, e, st);
    };
    DVD_TRY(conv(P, Q, 512, 64, 1));
    DVD_TRY(maxpool2_nhwc_bf16(Q, P, nullptr, B, 512, 512, 64, st, pf));
    DVD_TRY(conv(P, Q, 256, 64, 2));
    DVD_TRY(conv(Q, P, 256, 128, 3));
    DVD_TRY(maxpool2_nhwc_bf16(P, Q, nullptr, B, 256, 256, 128, st, pf));
    DVD_TRY(conv(Q, P, 128, 128, 4));
    DVD_TRY(conv(P, Q, 128, 256, 5));
    DVD_TRY(conv(Q, P, 128, 256, 6));
    DVD_TRY(maxpool2_nhwc_bf16(P, nullptr, s.feat, B, 128, 128, 256, st, pf));
  } else {
    DVD_TRY(conv3x3(c, s.y4, s.pyrP, B, 512, 512, 4, w.pyr[0], w.pyr_b[0]));
    DVD_TRY(conv3x3(c, s.pyrP, s.pyrQ, B, 512, 512, 64, w.pyr[1], w.pyr_b[1]));
    DVD_TRY(maxpool2_nhwc(s.pyrQ, s.pyrP, B, 512, 512, 64, st));
    DVD_TRY(conv3x3(c, s.pyrP, s.pyrQ, B, 256, 256, 64, w.pyr[2], w.pyr_b[2]));
    DVD_TRY(conv3x3(c, s.pyrQ, s.pyrP, B, 256, 256, 128, w.pyr[3], w.pyr_b[3]));
    DVD_TRY(maxpool2_nhwc(s.pyrP, s.pyrQ, B, 256, 256, 128, st));
    DVD_TRY(conv3x3(c, s.pyrQ, s.pyrP, B, 128, 128, 128, w.pyr[4], w.pyr_b[4]));
    DVD_TRY(conv3x3(c, s.pyrP, s.pyrQ, B, 128, 128, 256, w.pyr[5], w.pyr_b[5]));
    DVD_TRY(conv3x3(c, s.pyrQ, s.pyrP, B, 128, 128, 256, w.pyr[6], w.pyr_b[6]));
    DVD_TRY(maxpool2_nhwc(s.pyrP, s.feat, B, 128, 128, 256, st));
  }
  // ---- K2 static patch embeds (c: CM:594, m: CM:585, l: CM:605), + bias + pos
  Epilogue e; e.pos = w.pos; e.pos_rows = 1024;
  for (int i = 0; i < 3; ++i) {
    const int emb = 2 + i;                       // emb[] order: obs, r, c, m, l
    const int C = i == 0 ? 256 : (i == 1 ? 384 : 64);
    if (i == 0) DVD_TRY(patchify_nhwc(s.feat, tc ? nullptr : s.a_stat, s.a_stat16.hi, s.a_stat16.lo, 4 * C, B, C, st));
    else DVD_TRY(patchify_nchw(i == 1 ? mask_y512 : line_msk, tc ? nullptr : s.a_stat, s.a_stat16.hi, s.a_stat16.lo, 4 * C, B, C, st));
    Epilogue ee = e; ee.bias = w.emb_b[emb]; ee.out = tc ? nullptr : s.ctx[i]; ee.ldc = 384;
    if (tc) out_operand(ee, s.ctx16[i], 384);
    DVD_TRY(linear(c, s.a_stat, s.a_stat16, 4 * C, w.emb[emb], 0, Md, 384, ee));
    // ---- static cross-attention K,V (in_proj rows 384..1151)
    Epilogue ek; ek.bias = w.xattn_in_b + 384; ek.out = tc ? nullptr : s.kv_static[i]; ek.ldc = 768;
    if (tc) { out_attn(c, ek, s.kv_static16[i], 768); ek.vt_out = s.vt_static16[i]; ek.vt_col0 = 384; }
    DVD_TRY(linear(c, s.ctx[i], s.ctx16[i], 384, w.xattn_in, 384, Md, 768, ek));
  }
  return 0;
}

static int attention(const Ctx& c, const float* q, const __nv_bfloat16* q16, int ldq, const float* k, const __nv_bfloat16* k16, int ldk,
                     const float* v, const __nv_bfloat16* vt16, int ldv, float* o, const B16& o16, int ldo, int nsamp, int d,
                     float scale, int kv_div) {
  ProfScope ps(PC_ATTN, c.st, 4.0 * nsamp * kHeads * 1024.0 * 1024.0 * d);
  if (c.tc()) return attention_tc(q16, ldq, k16, ldk, vt16, o16.hi, o16.lo, ldo, nsamp, kHeads, 1024, d, scale, kv_div, c.x3() ? 1 : 0, c.st);
  return attention_f32(q, ldq, k, ldk, v, ldv, o, ldo, nsamp, kHeads, 1024, d, scale, kv_div, c.ws.S, c.ws.s_floats, c.st);
}

// test hook (dvd_debug_stop_after): leave denoise_step after a stage so that the stage's output can be read from the workspace
//   1 = after the DiT block ("X" = x1|x2|x3|x4), 2 = after the adaptive positional encoding, 3 + l = after decoder layer l
static thread_local int g_stop_after = 0;

static int denoise_step(const Ctx& c, const float* x_t, const float* init_flow, const float* init_feat_nchw, int init_feat_div,
                        int feat_mode, const float* trow, float da, float db, float* pred, float* x_prev) {
  const dvd_weights_t& w = *c.w; const Workspace& s = c.ws; cudaStream_t st = c.st;
  const int N = c.docs * c.n_hyp, M = N * 1024;
  const bool tc = c.tc();
  // DVD_PREC_BF16X3 folds every LayerNorm of the decoder into the GEMM that consumes it (producers emit row statistics + the raw rows as
  // a 16-bit operand, the consumer normalises in its epilogue): norm2 -> conv1 (raw rows as a bf16 pair, three passes) and norm1 ->
  // q|k|v (raw rows as ONE fp16 value against the fp16 pair qkv_ln, two passes; q, k and v are rounded to fp16 for the attention anyway;
  // oracle: 1.2e-6 -> 1.8e-6 mean map error).  Measured against separate LayerNorm kernels in profiles/r2_ln_fusion.txt.  Before the
  // GEMM epilogue's cold-code fix the fused variants lost: every instruction added to an epilogue that ran cold cost several times its
  // warm price.
  const bool lnf = c.x3();
  const float* ada = trow + 384;                 // shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp
  const float* fin = trow + 384 + 2304;          // shift[1536], scale[1536]
  // ---- obs embed (CM:571) and r embed (CM:602-603) with the fused feature warp (GD:618-624)
  DVD_TRY(obs_embed(x_t, w.emb[0].f32, w.emb_b[0], w.pos, s.xe, N, st));
  const int lda_r = 1032;                       // 258*4; TMA zero-fills the K tail of the last 64-wide box
  DVD_TRY(build_r_operand(init_flow, s.feat, init_feat_nchw, init_feat_div, feat_mode, tc ? nullptr : s.a_r, s.a_r16.hi, s.a_r16.lo,
                          lda_r, N, c.n_hyp, st));
  {
    Epilogue e; e.bias = w.emb_b[1]; e.pos = w.pos; e.pos_rows = 1024; e.out = tc ? nullptr : s.r; e.ldc = 384;
    if (tc) out_operand(e, s.r16, 384);
    DVD_TRY(linear(c, s.a_r, s.a_r16, lda_r, w.emb[1], 0, M, 384, e));
  }
  // ---- cross attention (CM:237-265): one shared query, four contexts
  DVD_TRY(layernorm(s.xe, 384, tc ? nullptr : s.qn, 384, s.qn16.hi, s.qn16.lo, 384, M, 384, 1e-6f, nullptr, nullptr, nullptr, nullptr, st));
  {
    Epilogue e; e.bias = w.xattn_in_b; e.out = tc ? nullptr : s.q; e.ldc = 384;
    if (tc) out_attn(c, e, s.q16, 384);
    DVD_TRY(linear(c, s.qn, s.qn16, 384, w.xattn_in, 0, M, 384, e));
    Epilogue ek; ek.bias = w.xattn_in_b + 384; ek.out = tc ? nullptr : s.kv_r; ek.ldc = 768;
    if (tc) { out_attn(c, ek, s.kv_r16, 768); ek.vt_out = s.vt_r16; ek.vt_col0 = 384; }
    DVD_TRY(linear(c, s.r, s.r16, 384, w.xattn_in, 384, M, 768, ek));
  }
  if (tc) {
    // the four contexts (stream order x1..x4 = cond, msk6, msk_line, r; CM:243-265) share the queries: ONE launch of 4 x N x 6 x 8 CTAs
    ProfScope ps(PC_ATTN, st, 4.0 * 4.0 * N * kHeads * 1024.0 * 1024.0 * 64);
    const void* kk[4] = {s.kv_static16[0], s.kv_static16[1], s.kv_static16[2], s.kv_r16};
    const void* vv[4] = {s.vt_static16[0], s.vt_static16[1], s.vt_static16[2], s.vt_r16};
    __nv_bfloat16* oo[4]; __nv_bfloat16* ol[4];
    for (int i = 0; i < 4; ++i) { oo[i] = s.xo16.hi + (size_t)i * M * 384; ol[i] = s.xo16.lo ? s.xo16.lo + (size_t)i * M * 384 : nullptr; }
    const int dv[4] = {c.n_hyp, c.n_hyp, c.n_hyp, 1};
    DVD_TRY(attention_tc_multi(s.q16, 384, kk, 768, vv, oo, s.xo16.lo ? ol : nullptr, 384, dv, 4, N, kHeads, 1024, 64, 0.125f, c.x3() ? 1 : 0, st));
  } else {
    for (int i = 0; i < 4; ++i) {                // stream order x1..x4 = cond, msk6, msk_line, r  (CM:243-265)
      const float* kv = i < 3 ? s.kv_static[i] : s.kv_r;
      DVD_TRY(attention(c, s.q, nullptr, 384, kv, nullptr, 768, kv + 384, nullptr, 768, s.xo + (size_t)i * M * 384, B16(), 384, N, 64,
                        0.125f, i < 3 ? c.n_hyp : 1));
    }
  }
  {
    Epilogue e; e.bias = w.xattn_out_b; e.resid = s.xe; e.ldr = 384; e.resid_mod = M; e.out = s.xs; e.ldc = 384;
    DVD_TRY(linear(c, s.xo, s.xo16, 384, w.xattn_out, 0, 4 * M, 384, e));
  }
  // ---- adaLN self-attention on the 4 streams (CM:268-292), shared weights
  DVD_TRY(layernorm(s.xs, 384, tc ? nullptr : s.hmod, 384, s.hmod16.hi, s.hmod16.lo, 384, 4 * M, 384, 1e-6f, nullptr, nullptr, ada + 0,
                    ada + 384, st));
  {
    Epilogue e; e.bias = w.blk_qkv_b; e.out = tc ? nullptr : s.qkv; e.ldc = 1152;
    if (tc) { out_attn(c, e, s.qkv16, 1152); e.vt_out = s.vt_qkv16; e.vt_col0 = 768; }
    DVD_TRY(linear(c, s.hmod, s.hmod16, 384, w.blk_qkv, 0, 4 * M, 1152, e));
  }
  DVD_TRY(attention(c, s.qkv, s.qkv16, 1152, s.qkv + 384, tc ? s.qkv16 + 384 : nullptr, 1152, s.qkv + 768, s.vt_qkv16, 1152,
                    s.xo, s.xo16, 384, 4 * N, 64, 0.125f, 1));
  {
    Epilogue e; e.bias = w.blk_proj_b; e.gate = ada + 768; e.resid = s.xs; e.ldr = 384; e.out = s.xs; e.ldc = 384;
    DVD_TRY(linear(c, s.xo, s.xo16, 384, w.blk_proj, 0, 4 * M, 384, e));
  }
  // ---- adaLN MLP; fc2 writes straight into the concatenated decoder input (CM:623)
  DVD_TRY(layernorm(s.xs, 384, tc ? nullptr : s.hmod, 384, s.hmod16.hi, s.hmod16.lo, 384, 4 * M, 384, 1e-6f, nullptr, nullptr, ada + 1152,
                    ada + 1536, st));
  {
    Epilogue e; e.bias = w.blk_fc1_b; e.act = c.x3() ? ACT_GELU_EXACT : ACT_GELU; e.out = tc ? nullptr : s.h1; e.ldc = 1536;
    if (tc) out_operand(e, s.h116, 1536);
    DVD_TRY(linear(c, s.hmod, s.hmod16, 384, w.blk_fc1, 0, 4 * M, 1536, e));
    Epilogue f; f.bias = w.blk_fc2_b; f.gate = ada + 1920; f.resid = s.xs; f.ldr = 384; f.out = s.X; f.ldc = 1536;
    f.group_rows = M; f.group_col_stride = 384;
    DVD_TRY(linear(c, s.h1, s.h116, 1536, w.blk_fc2, 0, 4 * M, 384, f));
  }
  if (g_stop_after == 1) return 0;
  // ---- decoder: adaptive 2-D positional encoding (CA:143-157)
  {
    float* mean = s.pe; float* hs1 = s.pe + (size_t)N * 1536 * 33; float* hs = hs1 + (size_t)N * 1536;
    float* ws1 = hs + (size_t)N * 1536; float* wsv = ws1 + (size_t)N * 1536;
    DVD_TRY(token_mean(s.X, mean, N, 1536, st));
    // h- and w-branch side by side: conv1x1 + ReLU, then conv1x1 + sigmoid (CA:143-157)
    DVD_TRY(gemv_pair(mean, mean, 1536, w.h_scale0.f32, w.w_scale0.f32, w.h_scale0_b, w.w_scale0_b, hs1, ws1, 1536, N, 1536, 1536, 1, st));
    DVD_TRY(gemv_pair(hs1, ws1, 1536, w.h_scale2.f32, w.w_scale2.f32, w.h_scale2_b, w.w_scale2_b, hs, wsv, 1536, N, 1536, 1536, 3, st));
    // bf16x3: all twelve LayerNorms of the decoder are folded into the GEMMs that consume them (no LN kernel, no normalised copy):
    // every producer of the residual stream X also writes X as a 16-bit operand and the rows' partial (sum, sum of squares); the QKV /
    // conv1 GEMMs multiply the RAW rows by gamma-scaled weights and normalise in the epilogue (Epilogue::ln_*).  Accuracy checked on
    // the oracle first (oracle/precision_study.py --ln-fusion: 1.44e-6 -> 1.53e-6 mean map error).
    if (lnf) DVD_TRY(posenc_add_ln(s.X, hs, wsv, w.dec_hpe, w.dec_wpe, N, 1536, s.X16.hi, s.lnstats, 48, st));
    else DVD_TRY(posenc_add(s.X, hs, wsv, w.dec_hpe, w.dec_wpe, N, 1536, st));
  }
  if (g_stop_after == 2) return 0;
  // ---- 6 decoder layers (CA:377-396)
  for (int l = 0; l < 6; ++l) {
    const dvd_dec_layer_t& L = w.dec[l];
    if (!lnf) DVD_TRY(layernorm(s.X, 1536, tc ? nullptr : s.hd, 1536, s.hd16.hi, s.hd16.lo, 1536, M, 1536, 1e-5f, L.n1_w, L.n1_b, nullptr, nullptr, st));
    {
      Epilogue e; e.out = tc ? nullptr : s.qkv_d; e.ldc = 4608;
      if (tc) { out_attn(c, e, s.qkv_d16, 4608); e.vt_out = s.vt_d16; e.vt_col0 = 3072; }
      if (lnf) {
        e.ln_stats = s.lnstats; e.ln_colsum = L.qkv_colsum; e.ln_chunks = 48; e.ln_eps = 1e-5f; e.bias = L.qkv_cvec;
        DVD_TRY(linear(c, nullptr, s.X16, 1536, L.qkv_ln, 0, M, 4608, e, true));
      } else {
        DVD_TRY(linear(c, s.hd, s.hd16, 1536, L.qkv, 0, M, 4608, e));
      }
    }
    DVD_TRY(attention(c, s.qkv_d, s.qkv_d16, 4608, s.qkv_d + 1536, tc ? s.qkv_d16 + 1536 : nullptr, 4608, s.qkv_d + 3072, s.vt_d16, 4608,
                      s.att_d, s.att_d16, 1536, N, 256, 0.0625f, 1));
    {
      Epilogue e; e.resid = s.X; e.ldr = 1536; e.out = s.X; e.ldc = 1536;
      if (lnf) { out_operand(e, s.X16, 1536); e.stats_out = s.lnstats; }
      DVD_TRY(linear(c, s.att_d, s.att_d16, 1536, L.fc, 0, M, 1536, e));
    }
    if (!lnf) DVD_TRY(layernorm(s.X, 1536, tc ? nullptr : s.hd, 1536, s.hd16.hi, s.hd16.lo, 1536, M, 1536, 1e-5f, L.n2_w, L.n2_b, nullptr, nullptr, st));
    {
      Epilogue e; e.scale = L.bn1_scale; e.shift = L.bn1_shift; e.act = ACT_RELU; e.out = tc ? nullptr : s.f1; e.ldc = 2048;
      if (tc) out_operand(e, s.f116, 2048);
      if (lnf) {
        e.ln_stats = s.lnstats; e.ln_colsum = L.conv1_colsum; e.ln_chunks = 48; e.ln_eps = 1e-5f; e.bias = L.conv1_cvec;
        DVD_TRY(linear(c, nullptr, s.X16, 1536, L.conv1_ln, 0, M, 2048, e));
      } else {
        DVD_TRY(linear(c, s.hd, s.hd16, 1536, L.conv1, 0, M, 2048, e));
      }
    }
    if (tc) DVD_TRY(dwconv3x3_bn_relu_bf16(s.f116.hi, s.f116.lo, L.dw_w, L.bn2_scale, L.bn2_shift, s.f216.hi, s.f216.lo, N, 2048, st));
    else DVD_TRY(dwconv3x3_bn_relu(s.f1, L.dw_w, L.bn2_scale, L.bn2_shift, s.f2, nullptr, N, 2048, st));
    {
      Epilogue e; e.scale = L.bn3_scale; e.shift = L.bn3_shift; e.act = ACT_RELU; e.resid = s.X; e.ldr = 1536; e.out = s.X; e.ldc = 1536;
      if (lnf) { e.out_bf16 = s.X16.hi; e.out_lo = nullptr; e.ldc_bf16 = 1536; e.out_f16 = 1; e.stats_out = s.lnstats; }     // raw rows as ONE fp16
      DVD_TRY(linear(c, s.f2, s.f216, 2048, L.conv2, 0, M, 1536, e));
    }
    if (g_stop_after == 3 + l) return 0;
  }
  // ---- final layer + unpatchify + init_flow + DDIM update (one kernel)
  DVD_TRY(final_layer(s.X, w.dec_ln_w, w.dec_ln_b, fin, fin + 1536, w.fin.f32, w.fin_b, init_flow, x_t, da, db, pred, x_prev, N, st));
  return 0;
}

static int make_ctx(Ctx& c, const dvd_weights_t* w, void* workspace, size_t bytes, int docs, int n_hyp, int precision, void* stream) {
  DVD_REQUIRE(w && workspace, "null weights/workspace");
  DVD_REQUIRE(docs > 0 && n_hyp > 0, "docs and n_hyp must be positive");
  DVD_REQUIRE(precision == DVD_PREC_FP32 || precision == DVD_PREC_BF16 || precision == DVD_PREC_BF16X3, "bad precision %d", precision);
  DVD_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
  if (precision == DVD_PREC_BF16X3) {            // the packs only this precision reads (include/dvd_b200.h)
    for (int i = 0; i < 7; ++i) {
      DVD_REQUIRE(w->pyr_h[i].bf16, "bf16x3 weight table: pyr_h[%d].bf16 is NULL", i);
      DVD_REQUIRE(w->pyr_h[i].bf16_lo, "bf16x3 weight table: pyr_h[%d].bf16_lo is NULL", i);
    }
    for (int l = 0; l < 6; ++l) {
      const dvd_dec_layer_t& L = w->dec[l];
      const struct { const void* p; const char* name; } need[] = {
          {L.qkv_ln.bf16, "qkv_ln.bf16"}, {L.qkv_ln.bf16_lo, "qkv_ln.bf16_lo"}, {L.qkv_colsum, "qkv_colsum"}, {L.qkv_cvec, "qkv_cvec"},
          {L.conv1_ln.bf16, "conv1_ln.bf16"}, {L.conv1_ln.bf16_lo, "conv1_ln.bf16_lo"}, {L.conv1_colsum, "conv1_colsum"},
          {L.conv1_cvec, "conv1_cvec"}};
      for (const auto& f : need) DVD_REQUIRE(f.p, "bf16x3 weight table: dec[%d].%s is NULL", l, f.name);
    }
  }
  c.w = w; c.docs = docs; c.n_hyp = n_hyp; c.prec = precision; c.st = (cudaStream_t)stream;
  c.ws = carve(workspace, docs, n_hyp, precision);
  if (c.ws.total_bytes > bytes) {
    set_error("workspace too small: need %zu bytes, got %zu", c.ws.total_bytes, bytes);
    return DVD_E_WORKSPACE;
  }
  return 0;
}

}  // namespace dvd

using namespace dvd;

extern "C" size_t dvd_workspace_bytes(int docs, int n_hyp, int precision) {
  if (docs <= 0 || n_hyp <= 0) return 0;
  return carve(nullptr, docs, n_hyp, precision).total_bytes;
}

extern "C" const float* dvd_workspace_feat(void* workspace, int docs, int n_hyp, int precision) {
  if (!workspace || docs <= 0 || n_hyp <= 0) return nullptr;
  return carve(workspace, docs, n_hyp, precision).feat;
}

// name -> fp32 buffer inside the workspace (stage-level parity tests)
extern "C" const float* dvd_workspace_tensor(void* workspace, int docs, int n_hyp, int precision, const char* name, long long* numel) {
  if (!workspace || !name || docs <= 0 || n_hyp <= 0) return nullptr;
  Workspace w = carve(workspace, docs, n_hyp, precision);
  const long long N = (long long)docs * n_hyp, M = N * 1024, Md = (long long)docs * 1024;
  struct { const char* n; const float* p; long long c; } tab[] = {
      {"feat", w.feat, (long long)docs * 4096 * 256}, {"cond", w.ctx[0], Md * 384}, {"msk6", w.ctx[1], Md * 384},
      {"msk_line", w.ctx[2], Md * 384}, {"kv_cond", w.kv_static[0], Md * 768}, {"xe", w.xe, M * 384}, {"r", w.r, M * 384},
      {"q", w.q, M * 384}, {"kv_r", w.kv_r, M * 768}, {"xo", w.xo, 4 * M * 384}, {"xs", w.xs, 4 * M * 384},
      {"qkv", w.qkv, 4 * M * 1152}, {"X", w.X, M * 1536}, {"qkv_d", w.qkv_d, M * 4608}, {"att_d", w.att_d, M * 1536},
      {"f1", w.f1, M * 2048}, {"a_r", w.a_r, M * 1032}, {"pe", w.pe, N * 1536 * 37}};
  for (auto& t : tab)
    if (!strcmp(t.n, name)) { if (numel) *numel = t.c; return t.p; }
  return nullptr;
}

extern "C" int dvd_tables_init(const dvd_weights_t* w, const float* t_values_host, int n_steps, float* tables, void* stream) {
  DVD_REQUIRE(w && t_values_host && tables && n_steps > 0, "tables_init: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  for (int s = 0; s < n_steps; ++s) {
    float* row = tables + (size_t)s * DVD_TABLE_ROW;
    float* fin = row + 384 + 2304;
    float* tval = fin + 1024;                    // scratch inside the row, overwritten last
    float* freq = fin;                           // [256]
    float* h = fin + 256;                        // [384]
    DVD_CUDA(cudaMemcpyAsync(tval, t_values_host + s, sizeof(float), cudaMemcpyHostToDevice, st));
    DVD_TRY(timestep_embedding(tval, freq, 1, st));
    DVD_TRY(gemv(freq, 256, w->t_mlp0.f32, w->t_mlp0_b, h, 384, 1, 384, 256, 0, 0, 4, st));        // Linear + SiLU (CM:104-108)
    DVD_TRY(gemv(h, 384, w->t_mlp2.f32, w->t_mlp2_b, row, 384, 1, 384, 384, 0, 0, 0, st));
    DVD_TRY(gemv(row, 384, w->blk_ada.f32, w->blk_ada_b, row + 384, 2304, 1, 2304, 384, 1, 0, 0, st));   // CM:175-177,209-211
    DVD_TRY(gemv(row, 384, w->fin_ada.f32, w->fin_ada_b, fin, 3072, 1, 3072, 1536, 1, 384, 0, st));      // CM:325-331 t.repeat(1,4)
  }
  return 0;
}

extern "C" int dvd_static_forward(const dvd_weights_t* w, void* workspace, size_t workspace_bytes, int docs, int n_hyp, int precision,
                                  const float* y512, const float* mask_cat, const float* mask_y512, const float* line_msk, void* stream) {
  Ctx c;
  DVD_TRY(make_ctx(c, w, workspace, workspace_bytes, docs, n_hyp, precision, stream));
  DVD_REQUIRE(y512 && mask_cat && mask_y512 && line_msk, "static_forward: null input");
  return static_forward(c, y512, mask_cat, mask_y512, line_msk);
}

extern "C" int dvd_denoise_step(const dvd_weights_t* w, void* workspace, size_t workspace_bytes, int docs, int n_hyp, int precision,
                                const float* x_t, const float* init_flow, const float* init_feat, int feat_is_init, const float* table_row,
                                float ddim_a, float ddim_b, float* pred_x0, float* x_prev, void* stream) {
  Ctx c;
  DVD_TRY(make_ctx(c, w, workspace, workspace_bytes, docs, n_hyp, precision, stream));
  DVD_REQUIRE(x_t && init_flow && table_row && pred_x0, "denoise_step: null argument");
  const int mode = feat_is_init ? FEAT_ASIS : (init_feat ? FEAT_EXPLICIT_OR_ZERO : FEAT_WARP);
  return denoise_step(c, x_t, init_flow, init_feat, 1, mode, table_row, ddim_a, ddim_b, pred_x0, x_prev);
}

extern "C" int dvd_debug_stop_after(int stage) { g_stop_after = stage; return 0; }

extern "C" int dvd_profile_begin(void) {
  for (auto& v : g_prof.ev) { for (auto e : v) cudaEventDestroy(e); v.clear(); }
  for (int i = 0; i < PC_COUNT; ++i) { g_prof.flops[i] = 0; g_prof.exec_flops[i] = 0; g_prof.launches[i] = 0; }
  g_prof.on = true;
  return 0;
}
// ms[3], flops[3], launches[3], executed_flops[3] for the classes {gemm, attention, pyramid conv}; synchronises the device.
extern "C" int dvd_profile_end(double* ms, double* flops, long long* launches, double* executed_flops) {
  g_prof.on = false;
  DVD_CUDA(cudaDeviceSynchronize());
  for (int c = 0; c < PC_COUNT; ++c) {
    double tot = 0;
    for (size_t i = 0; i + 1 < g_prof.ev[c].size(); i += 2) {
      float t = 0; cudaEventElapsedTime(&t, g_prof.ev[c][i], g_prof.ev[c][i + 1]); tot += t;
    }
    if (ms) ms[c] = tot;
    if (flops) flops[c] = g_prof.flops[c];
    if (executed_flops) executed_flops[c] = g_prof.exec_flops[c];
    if (launches) launches[c] = g_prof.launches[c];
    for (auto e : g_prof.ev[c]) cudaEventDestroy(e);
    g_prof.ev[c].clear();
  }
  return 0;
}

extern "C" int dvd_hyp_mean_clamp(const float* pred_x0, float* out, int docs, int n_hyp, void* stream) {
  return hyp_mean_clamp(pred_x0, out, docs, n_hyp, (cudaStream_t)stream);
}

// The S-step DDIM loop of one group of hypotheses (GD:574-633); leaves the last pred_xstart of the group in `final_flow`.
static int sample_group(const Ctx& c, const float* x_T, const float* init_flow0, const float* tables, const float* t_scaled_host,
                        const float* ddim_a_host, const float* ddim_b_host, int S, const float* init_feat0, float* final_flow, int it_begin,
                        int it_end, const float*& x, int& cur) {
  const Workspace& s = c.ws; cudaStream_t st = c.st;
  const int n_hyp = c.n_hyp;
  if (it_begin == 0) {
    // GD:574: every kwarg (incl. init_flow) is repeated n_hyp times
    for (int d = 0; d < c.docs; ++d)
      for (int h = 0; h < n_hyp; ++h)
        DVD_CUDA(cudaMemcpyAsync(s.flow[0] + ((size_t)d * n_hyp + h) * 8192, init_flow0 + (size_t)d * 8192, 8192 * sizeof(float),
                                 cudaMemcpyDeviceToDevice, st));
    x = x_T; cur = 0;
  }
  for (int it = it_begin; it < it_end; ++it) {
    // CM:597-598: while the rescaled t > 600 the model overrides init_feat with the un-warped feature.
    // GD:618-624: from the second iteration on, init_flow = previous pred_xstart and init_feat = warp(feat).
    // First iteration with t <= 600 (only possible for S < 3): the caller's init_feat (zeros at EV:167) is used.
    // CM:599-601: with more than one sample per call, entries whose rescaled t equals 2 exactly also take the un-warped feature (the
    // reference compares the float timestep with the integer label 2: only reachable at S = 1000, t index 2).
    const bool asis = t_scaled_host[it] > 600.0f || (t_scaled_host[it] == 2.0f && n_hyp > 1);
    int feat_mode = asis ? FEAT_ASIS : (it == 0 ? FEAT_EXPLICIT_OR_ZERO : FEAT_WARP);
    float* xn = s.xbuf[it & 1];
    float* pred = (it + 1 == S) ? final_flow : s.flow[cur ^ 1];      // pred of this step is init_flow of the next one
    DVD_TRY(denoise_step(c, x, s.flow[cur], feat_mode == FEAT_EXPLICIT_OR_ZERO ? init_feat0 : nullptr, n_hyp, feat_mode,
                         tables + (size_t)it * DVD_TABLE_ROW, ddim_a_host[it], ddim_b_host[it], pred, it + 1 < S ? xn : nullptr));
    x = xn; cur ^= 1;
  }
  return 0;
}

extern "C" int dvd_sample(const dvd_weights_t* w, void* workspace, size_t workspace_bytes, int docs, int n_hyp, int precision,
                          const float* x_T, const float* init_flow0, const float* tables, const float* t_scaled_host,
                          const float* ddim_a_host, const float* ddim_b_host, int S, const float* init_feat0, float* map_out,
                          void* stream) {
  Ctx c;
  DVD_TRY(make_ctx(c, w, workspace, workspace_bytes, docs, n_hyp, precision, stream));
  DVD_REQUIRE(x_T && init_flow0 && tables && t_scaled_host && ddim_a_host && ddim_b_host && map_out && S > 0, "sample: bad args");
  cudaStream_t st = c.st;
  const float* x = nullptr; int cur = 0;
  DVD_TRY(sample_group(c, x_T, init_flow0, tables, t_scaled_host, ddim_a_host, ddim_b_host, S, init_feat0, c.ws.final_flow, 0, S, x, cur));
  return hyp_mean_clamp(c.ws.final_flow, map_out, docs, n_hyp, st);
}
