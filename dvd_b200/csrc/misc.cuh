// Small fused kernels around the dense contractions (all bandwidth-trivial next to the GEMMs).
#pragma once
#include "common.cuh"

namespace dvd {

// rows x C layer norm (two-pass in registers, one warp per row), optional affine, optional
// adaLN modulate:  out = (LN(x)*w + b) * (1 + mod_scale) + mod_shift.   C in {384, 1536}.
// Writes fp32 (out) and/or bf16 (out_bf16); either may be null.
// bf16 destinations throughout this header: `x16` alone is plain bf16; with a non-null `x16_lo` the value is stored as the split
// pair hi = bf16(v), lo = bf16(v - hi) (operand of a 3-pass GEMM in DVD_PREC_BF16X3).
int layernorm(const float* in, int ldin, float* out, int ldo, __nv_bfloat16* out_bf16, __nv_bfloat16* out_bf16_lo, int ldo16, int rows, int C,
              float eps, const float* w, const float* b, const float* mod_shift, const float* mod_scale, cudaStream_t st);

// y512 [B,3,512,512] + mask [B,1,512,512] (NCHW) -> NHWC [B,512,512,4]        (CM:586-587)
int pack_y4(const float* y512, const float* mask, float* out, int B, cudaStream_t st);
// 2x2 max pool on NHWC fp32
int maxpool2_nhwc(const float* in, float* out, int B, int H, int W, int C, cudaStream_t st);
// 3x3 / pad 1 im2col of a 4-channel NHWC fp32 image into bf16 rows of 64 (k = tap*4 + c, k >= 36 zero): [B*H*W, 64]
// (out_f16 != 0: ONE IEEE fp16 value per element instead of bf16)
int im2col3x3_c4_bf16(const float* in, __nv_bfloat16* out, int B, int H, int W, cudaStream_t st, int out_f16);
int maxpool2_nhwc_bf16(const __nv_bfloat16* in, __nv_bfloat16* out16, float* out32, int B, int H, int W, int C, cudaStream_t st,
                       int f16);      // f16: input and 16-bit output are single fp16 values (else bf16)
// fp32 NHWC -> NCHW (feat for the drop-in model() return value) and back
int nhwc_to_nchw(const float* in, float* out, int B, int H, int W, int C, cudaStream_t st);

// patchify (timm PatchEmbed's conv k=2,s=2 as a GEMM A operand): A[(b,h,w), c*4+p*2+q] = in[b,c,2h+p,2w+q]
// NCHW source [B,C,64,64] -> A [B*1024, lda] (fp32 and/or bf16)
int patchify_nchw(const float* in, float* A, __nv_bfloat16* A16, __nv_bfloat16* A16_lo, int lda, int B, int C, cudaStream_t st);
// NHWC source [B,64,64,C]
int patchify_nhwc(const float* in, float* A, __nv_bfloat16* A16, __nv_bfloat16* A16_lo, int lda, int B, int C, cudaStream_t st);

// A operand of the r-embedder (CM:602-603) fused with the inter-step feature warp (GD:618-624):
//   channels 0..1  = init_flow[n]        (NCHW [N,2,64,64])
//   channels 2..257 = warp ? grid_sample(feat[n/n_hyp], (init_flow[n]+base64)*2-1) : feat[n/n_hyp]
//   or, when init_feat_nchw != NULL, that explicit tensor [N,256,64,64].
// feat is NHWC [docs,64,64,256].  A [N*1024, lda>=1032].
enum { FEAT_ASIS = 0, FEAT_WARP = 1, FEAT_EXPLICIT_OR_ZERO = 2 };
// mode FEAT_EXPLICIT_OR_ZERO: init_feat_nchw[n / init_feat_div] if non-NULL, else zeros (EV:167).
int build_r_operand(const float* init_flow, const float* feat_nhwc, const float* init_feat_nchw, int init_feat_div, int mode,
                    float* A, __nv_bfloat16* A16, __nv_bfloat16* A16_lo, int lda, int N, int n_hyp, cudaStream_t st);

// obs patch embed (K = 8, CM:571) done directly: xe[n,tok,:] = W[384,8] * patch + bias + pos
int obs_embed(const float* x, const float* W, const float* bias, const float* pos, float* out, int N, cudaStream_t st);

// row softmax in place over [rows, n] (n <= 1024, multiple of 32), one warp per row
int softmax_rows(float* S, long long rows, int n, cudaStream_t st);

// small dense layer for N_rows <= 8: out[r, j] = act( dot(f(in[r, :]), W[j, :]) + b[j] ),
// f = SiLU if silu_in; input index taken modulo in_mod (t.repeat(1,4), CM:331) if in_mod > 0.
int gemv(const float* in, int ldin, const float* W, const float* b, float* out, int ldo, int rows, int N, int K,
         int silu_in, int in_mod, int act, cudaStream_t st);
int gemv_pair(const float* in0, const float* in1, int ldin, const float* W0, const float* W1, const float* b0, const float* b1, float* out0,
              float* out1, int ldo, int rows, int N, int K, int act, cudaStream_t st);

// sinusoidal timestep embedding (CM:111-134): out[r, 0:128]=cos, [128:256]=sin
int timestep_embedding(const float* t, float* out, int rows, cudaStream_t st);

// mean over the 1024 tokens of X [N,1024,C] -> [N,C]                      (CA:146 AdaptiveAvgPool2d)
int token_mean(const float* X, float* out, int N, int C, cudaStream_t st);
// X[n,tok,c] += hs[n,c]*hpe[tok/32,c] + ws[n,c]*wpe[tok%32,c]              (CA:148-153)
int posenc_add(float* X, const float* hs, const float* ws, const float* hpe, const float* wpe, int N, int C, cudaStream_t st);

// same + the row as ONE IEEE fp16 value per element in x16 (the raw-row operand of the two-pass q|k|v GEMM) + per-row (sum, sum of
// squares) in `stats` [N*1024][chunks][2] (slot 0), for the LayerNorm fused into that GEMM's epilogue (Epilogue::ln_stats).
// C = 1536, chunks = C / 32.
int posenc_add_ln(float* X, const float* hs, const float* ws, const float* hpe, const float* wpe, int N, int C, __nv_bfloat16* x16,
                  float* stats, int chunks, cudaStream_t st);

// depthwise 3x3 (pad 1) over the 32x32 token grid + folded BN + ReLU, token-major [N,1024,C]  (CA:33-41)
int dwconv3x3_bn_relu(const float* in, const float* w9c, const float* scale, const float* shift, float* out,
                      __nv_bfloat16* out16, int N, int C, cudaStream_t st);

int dwconv3x3_bn_relu_bf16(const __nv_bfloat16* in, const __nv_bfloat16* in_lo, const float* w9c, const float* scale, const float* shift,
                           __nv_bfloat16* out, __nv_bfloat16* out_lo, int N, int C, cudaStream_t st);

// decoder.layer_norm (affine, 1e-5) -> norm_final (1e-6) -> modulate -> Linear 1536->8 -> unpatchify
// -> += init_flow -> pred ; x_prev = a*pred + b*x_t          (CA:457, CM:329-336,553-566,645-646, GD:470-489)
int final_layer(const float* X, const float* ln_w, const float* ln_b, const float* shift, const float* scale,
                const float* W8, const float* b8, const float* init_flow, const float* x_t, float a, float b,
                float* pred, float* x_prev, int N, cudaStream_t st);

int hyp_mean_clamp(const float* pred, float* out, int docs, int n_hyp, cudaStream_t st);

int f32_to_bf16(const float* in, __nv_bfloat16* out, long long n, cudaStream_t st);

}  // namespace dvd
namespace dvd {
int bf16_to_f32(const __nv_bfloat16* in, float* out, long long n, cudaStream_t st);
int f32_split_bf16(const float* in, __nv_bfloat16* hi, __nv_bfloat16* lo, long long n, cudaStream_t st);
int f32_to_f16(const float* in, void* out, long long n, cudaStream_t st);
int f32_split_f16(const float* in, void* hi, void* lo, long long n, cudaStream_t st);      // IEEE fp16 pair (test hook)
int pair_to_f32(const __nv_bfloat16* hi, const __nv_bfloat16* lo, float* out, long long n, cudaStream_t st);
}
