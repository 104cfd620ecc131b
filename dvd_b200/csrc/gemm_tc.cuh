// tcgen05 / TMEM / TMA tensor-core path (DVD_PREC_BF16 and DVD_PREC_BF16X3): dense GEMM with the shared Epilogue and
// flash attention.  Implemented in gemm_tc.cu (tensor maps, dispatch, single-CTA kernel), gemm_pair.cu (persistent CTA-pair
// kernel) and attn_tc.cu.
#pragma once
#include "gemm_simt.cuh"

namespace dvd {

// One K-major 16-bit operand matrix (row-major, K contiguous, leading dimension ld in elements).  lo == nullptr: plain bf16.
// lo != nullptr: split-precision pair, value = hi + lo (both bf16); a GEMM whose A and W are both pairs runs three tensor-core
// passes per k-step (hi*hi + lo*hi + hi*lo: fp32-accurate to ~2^-16, the lo*lo term is dropped).
struct TcMat {
  const __nv_bfloat16* hi = nullptr;
  const __nv_bfloat16* lo = nullptr;
  int ld = 0;
  bool f16 = false;      // A: `hi` holds ONE IEEE fp16 value per element (two-pass mode; lo must be null, and W must be an fp16 pair)
};

// C[M,N] = epilogue(A[M,K] * W[N,K]^T), fp32 accumulate in TMEM.  M % 128 == 0, K % 8 == 0, N % 4 == 0.
int gemm_tc(const TcMat& A, const TcMat& W, int M, int N, int K, const Epilogue& e, cudaStream_t st);
inline int gemm_tc_bf16(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, int ldw, int M, int N, int K, const Epilogue& e,
                        cudaStream_t st) {
  TcMat a; a.hi = A; a.ld = lda;
  TcMat w; w.hi = W; w.ld = ldw;
  return gemm_tc(a, w, M, N, K, e, st);
}

// 3x3 / pad 1 conv as implicit GEMM on tcgen05 (TMA boxes over the NHWC activation, zero padding by OOB fill):
// in [B,H,W,Cin] (plain bf16 with a plain bf16 Wt, or fp16 with an fp16 pair Wt), Wt [Cout, 9*Cin] ordered [ky][kx][Cin]; output
// through the Epilogue as [B*H*W, Cout].
int conv3x3_tc(const TcMat& in, const TcMat& Wt, int B, int H, int Wd, int Cin, int Cout, const Epilogue& e, cudaStream_t st);

// softmax(scale * Q K^T) V per (sample, head); 16-bit in/out (bf16, or fp16 when f16 != 0), fp32 softmax statistics and accumulation.
// q/k/o row-major with leading dims ld*, head h at columns [h*d, (h+1)*d); vt is V TRANSPOSED: [nsamp/kv_div, heads*d, T]
// (written by the QKV GEMM epilogue, Epilogue::vt_out).  k/vt of sample n come from sample n / kv_div.
// The output is always bf16: o (and, when o_lo != nullptr, the low half of the split pair o + o_lo).  d in {64, 256}, T % 128 == 0.
int attention_tc(const void* q, int ldq, const void* k, int ldk, const void* vt, __nv_bfloat16* o, __nv_bfloat16* o_lo, int ldo,
                 int nsamp, int heads, int T, int d, float scale, int kv_div, int f16, cudaStream_t st);

// Same, for up to 4 key/value contexts that share the queries (one launch): context i uses k[i], vt[i], kv_div[i], writes o[i] (+ o_lo[i]).
int attention_tc_multi(const void* q, int ldq, const void* const* k, int ldk, const void* const* vt, __nv_bfloat16* const* o,
                       __nv_bfloat16* const* o_lo, int ldo, const int* kv_div, int nctx, int nsamp, int heads, int T, int d, float scale,
                       int f16, cudaStream_t st);

// ---- internal: head dim 256 on a CTA pair (attn_pair.cu), 128-key steps, P read from tensor memory.  DVD_ATTN_V1=1 disables it.
bool attention_pair_supported(int T, int d, int nctx);
int attention_pair(const void* q, int ldq, const void* k, int ldk, const void* vt, __nv_bfloat16* o, __nv_bfloat16* o_lo, int ldo, int nsamp,
                   int heads, int T, float scale, int kv_div, int f16, cudaStream_t st);

// V [nsamp, T, C] (row stride ldv) -> V^T [nsamp, C, T], any 16-bit type  (test hook only)
int transpose_v16(const void* v, int ldv, void* vt, int nsamp, int T, int C, cudaStream_t st);

int sm_count();       // SMs of the current device (cached per device)

// ---- internal: persistent CTA-pair kernel (gemm_pair.cu); conv_h > 0 selects the implicit-GEMM mode
bool gemm_pair_supported(int M, int N, int K, bool conv);
int gemm_pair_dispatch(const TcMat& A, const TcMat& W, int M, int N, int K, const Epilogue& e, int conv_b, int conv_h, int conv_w,
                       int conv_cin, cudaStream_t st);

}  // namespace dvd
