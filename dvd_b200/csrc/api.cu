// C-ABI plumbing: version, thread-local error text, device check, launch counter, test hooks.
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "misc.cuh"

namespace dvd {

static thread_local char g_err[512] = "";
static thread_local long long g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return (int)e;
}
void count_launch(int n) { g_launches += n; }
bool pdl_enabled(int kind) {
  static int mask = -1;
  if (mask < 0) {
    const char* off = getenv("DVD_NO_PDL");
    const char* m = getenv("DVD_PDL_MASK");
    mask = (off && off[0] == '1') ? 0 : (m ? atoi(m) : 0x1F);
  }
  return (mask & kind) != 0;
}
// Timing ablation only (results are garbage): DVD_DEBUG_SKIP=<mask> drops every launch of the given kernel kinds, so that the
// difference in ms/step is the true in-graph cost of that class (ncu durations are cold-cache and serialised).
bool debug_skip(int kind) {
  static int mask = -1;
  if (mask < 0) { const char* m = getenv("DVD_DEBUG_SKIP"); mask = m ? atoi(m) : 0; }
  return (mask & kind) != 0;
}

}  // namespace dvd

using namespace dvd;

extern "C" int dvd_version(void) { return DVD_ABI_VERSION; }
extern "C" const char* dvd_last_error(void) { return g_err; }
extern "C" long long dvd_launch_count(int reset) {
  long long v = g_launches;
  if (reset) g_launches = 0;
  return v;
}
extern "C" int dvd_check_device(void) {
  int dev = 0;
  DVD_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp p;
  DVD_CUDA(cudaGetDeviceProperties(&p, dev));
  if (p.major != 10) {
    set_error("device %d is sm_%d%d; libdvd_b200 is built for sm_100a only", dev, p.major, p.minor);
    return DVD_E_ARCH;
  }
  return 0;
}

// A[M,K] fp32, W[N,K] fp32 -> C[M,N] = A W^T + bias.  In the tensor modes the operands are first converted into `scratch`
// (bf16: (M+N)*K*2 bytes; bf16x3: twice that) and the tcgen05 kernels are used.
extern "C" int dvd_test_gemm(const float* A, const float* W, const float* bias, float* C, int M, int N, int K, int precision,
                             void* scratch, size_t scratch_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  DVD_REQUIRE(A && W && C, "test_gemm: null");
  Epilogue e; e.bias = bias; e.out = C; e.ldc = N;
  if (precision == DVD_PREC_FP32) {
    GemmParams p = linear_params(A, K, W, M, N, K);
    p.e = e;
    return gemm_f32(p, A_DIRECT, B_NK, 1, st);
  }
  const bool a16 = precision == 3;                // test-only code: ONE fp16 activation x fp16 weight pair (the decoder's q|k|v GEMM in DVD_PREC_BF16X3)
  const bool x3 = precision == DVD_PREC_BF16X3 || a16;
  auto al = [](size_t b) { return (b + 255) & ~size_t(255); };
  const size_t a_b = al((size_t)M * K * 2), w_b = al((size_t)N * K * 2);
  const size_t ops = (x3 ? 2 : 1) * (a_b + w_b);
  DVD_REQUIRE(scratch && scratch_bytes >= ops, "test_gemm: scratch needs %zu bytes", ops);
  char* base = (char*)scratch;
  TcMat a, w;
  a.hi = (__nv_bfloat16*)base; w.hi = (__nv_bfloat16*)(base + a_b); a.ld = K; w.ld = K;
  int rc;
  if (x3) {
    a.lo = (__nv_bfloat16*)(base + a_b + w_b); w.lo = (__nv_bfloat16*)(base + 2 * a_b + w_b);
    if (a16) { rc = f32_to_f16(A, (void*)a.hi, (long long)M * K, st); a.lo = nullptr; a.f16 = true; }
    else rc = f32_split_bf16(A, (__nv_bfloat16*)a.hi, (__nv_bfloat16*)a.lo, (long long)M * K, st);
    if (rc) return rc;
    rc = a16 ? f32_split_f16(W, (void*)w.hi, (void*)w.lo, (long long)N * K, st)
             : f32_split_bf16(W, (__nv_bfloat16*)w.hi, (__nv_bfloat16*)w.lo, (long long)N * K, st);
    if (rc) return rc;
  } else {
    rc = f32_to_bf16(A, (__nv_bfloat16*)a.hi, (long long)M * K, st); if (rc) return rc;
    rc = f32_to_bf16(W, (__nv_bfloat16*)w.hi, (long long)N * K, st); if (rc) return rc;
  }
  return gemm_tc(a, w, M, N, K, e, st);
}

// q,k,v,o: [batch, T, heads*d] fp32.  fp32 mode: scratch holds the [batch*heads, T, T] scores.
extern "C" int dvd_test_attention(const float* q, const float* k, const float* v, float* o, int batch, int heads, int T, int d,
                                  float scale, int precision, void* scratch, size_t scratch_bytes, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  DVD_REQUIRE(q && k && v && o && scratch, "test_attention: null");
  const int ld = heads * d;
  if (precision == DVD_PREC_FP32) {
    size_t per = (size_t)heads * T * T;
    DVD_REQUIRE(scratch_bytes >= per * batch * 4, "test_attention: scratch needs %zu bytes", per * batch * 4);
    float* S = (float*)scratch;
    GemmParams p;
    p.A = q; p.lda = ld; p.sAn = (long long)T * ld; p.sAh = d;
    p.B = k; p.ldb = ld; p.sBn = (long long)T * ld; p.sBh = d;
    p.M = T; p.N = T; p.K = d; p.heads = heads; p.alpha = scale;
    p.e.out = S; p.e.ldc = T; p.sCn = (long long)per; p.sCh = (long long)T * T;
    int rc = gemm_f32(p, A_DIRECT, B_NK, batch * heads, st); if (rc) return rc;
    rc = softmax_rows(S, (long long)batch * heads * T, T, st); if (rc) return rc;
    GemmParams g;
    g.A = S; g.lda = T; g.sAn = (long long)per; g.sAh = (long long)T * T;
    g.B = v; g.ldb = ld; g.sBn = (long long)T * ld; g.sBh = d;
    g.M = T; g.N = d; g.K = T; g.heads = heads;
    g.e.out = o; g.e.ldc = ld; g.sCn = (long long)T * ld; g.sCh = d;
    return gemm_f32(g, A_DIRECT, B_KN, batch * heads, st);
  }
  // tensor modes: bf16 operands (DVD_PREC_BF16) or fp16 operands + split-pair output (DVD_PREC_BF16X3)
  const bool x3 = precision == DVD_PREC_BF16X3;
  size_t n = (size_t)batch * T * ld;
  DVD_REQUIRE(scratch_bytes >= n * 2 * 6, "test_attention: scratch needs %zu bytes", n * 12);
  __nv_bfloat16* q16 = (__nv_bfloat16*)scratch; __nv_bfloat16* k16 = q16 + n; __nv_bfloat16* v16 = k16 + n; __nv_bfloat16* o16 = v16 + n;
  __nv_bfloat16* vt16 = o16 + n; __nv_bfloat16* olo = vt16 + n;
  int rc;
  if (x3) {
    rc = f32_to_f16(q, q16, n, st); if (rc) return rc;
    rc = f32_to_f16(k, k16, n, st); if (rc) return rc;
    rc = f32_to_f16(v, v16, n, st); if (rc) return rc;
  } else {
    rc = f32_to_bf16(q, q16, n, st); if (rc) return rc;
    rc = f32_to_bf16(k, k16, n, st); if (rc) return rc;
    rc = f32_to_bf16(v, v16, n, st); if (rc) return rc;
  }
  rc = transpose_v16(v16, ld, vt16, batch, T, ld, st); if (rc) return rc;
  rc = attention_tc(q16, ld, k16, ld, vt16, o16, x3 ? olo : nullptr, ld, batch, heads, T, d, scale, 1, x3 ? 1 : 0, st); if (rc) return rc;
  return pair_to_f32(o16, x3 ? olo : nullptr, o, n, st);
}

// The decoder's depthwise 3x3 + folded BN + ReLU of the tensor modes on its own: [N,1024,C] bf16 (in_lo non-NULL: bf16 pairs) in and
// out, the same launch dvd_denoise_step makes.
extern "C" int dvd_test_dwconv(const void* in_hi, const void* in_lo, const float* w9, const float* scale, const float* shift, void* out_hi,
                               void* out_lo, int N, int C, void* stream) {
  return dwconv3x3_bn_relu_bf16((const __nv_bfloat16*)in_hi, (const __nv_bfloat16*)in_lo, w9, scale, shift, (__nv_bfloat16*)out_hi,
                                (__nv_bfloat16*)out_lo, N, C, (cudaStream_t)stream);
}

// Plain tensor-core GEMM entry point (tuning / micro-benchmarks): out = A W^T + bias, bf16 output (and optional fp32 output).
// A16_lo / W16_lo non-null: split-precision pairs (three passes).
extern "C" int dvd_gemm_bf16(const void* A16, const void* A16_lo, int lda, const void* W16, const void* W16_lo, int ldw, const float* bias,
                             void* out16, float* out32, int M, int N, int K, void* stream) {
  Epilogue e; e.bias = bias; e.out_bf16 = (__nv_bfloat16*)out16; e.ldc_bf16 = N; e.out = out32; e.ldc = N;
  TcMat a, w;
  a.hi = (const __nv_bfloat16*)A16; a.lo = (const __nv_bfloat16*)A16_lo; a.ld = lda;
  a.f16 = !A16_lo && W16_lo;                      // a lone A next to a weight pair is fp16: the two-pass mode
  w.hi = (const __nv_bfloat16*)W16; w.lo = (const __nv_bfloat16*)W16_lo; w.ld = ldw;
  return gemm_tc(a, w, M, N, K, e, (cudaStream_t)stream);
}

// Same with the epilogue pieces the decoder uses (tuning / micro-benchmarks): folded BN scale / shift, ReLU, a split-pair 16-bit output
// (out16_lo) and an fp32 residual added in place of `out32` (resid may alias out32).
extern "C" int dvd_gemm_tune(const void* A16, const void* A16_lo, int lda, const void* W16, const void* W16_lo, int ldw, const float* bias,
                             const float* scale, const float* shift, int relu, void* out16, void* out16_lo, float* out32, const float* resid,
                             int M, int N, int K, void* stream) {
  Epilogue e; e.bias = bias; e.scale = scale; e.shift = shift; e.act = relu ? ACT_RELU : ACT_NONE;
  e.out_bf16 = (__nv_bfloat16*)out16; e.out_lo = (__nv_bfloat16*)out16_lo; e.ldc_bf16 = N; e.out = out32; e.ldc = N;
  e.resid = resid; e.ldr = N;
  TcMat a, w;
  a.hi = (const __nv_bfloat16*)A16; a.lo = (const __nv_bfloat16*)A16_lo; a.ld = lda;
  a.f16 = !A16_lo && W16_lo;
  w.hi = (const __nv_bfloat16*)W16; w.lo = (const __nv_bfloat16*)W16_lo; w.ld = ldw;
  return gemm_tc(a, w, M, N, K, e, (cudaStream_t)stream);
}
