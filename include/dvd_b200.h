/*
 * dvd_b200.h — C ABI of libdvd_b200.so: the B200 (sm_100a) implementation of DvD's sampling +
 * unwarp hot path.
 *
 * The reference (hanquansanren/DvD) is pure Python/PyTorch and has no FFI of its own; this is the
 * thin native boundary its Python call sites bind through ctypes (see INTEGRATION.md).  Each
 * entry point names the reference lines it replaces (paths relative to the reference root):
 *   GD = train_settings/dvd/improved_diffusion/gaussian_diffusion.py
 *   CM = train_settings/dvd/improved_diffusion/cross_model.py
 *   CA = train_settings/dvd/improved_diffusion/cross_attn.py
 *   EV = train_settings/dvd/evaluation.py
 *   WP = datasets/utils/warping.py
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless the name ends in _host.
 *   - the caller owns every buffer (weights, workspace, inputs, outputs); the library allocates
 *     no device memory and keeps no pointer past a call.
 *   - all work is enqueued asynchronously on `stream` (a cudaStream_t passed as void*); no
 *     implicit device synchronisation, so every call is CUDA-graph capturable.
 *   - return value: 0 = ok, >0 = cudaError_t, <0 = DVD_E_* ; text via dvd_last_error()
 *     (thread local).  No C++ exception crosses the boundary.
 */
#ifndef DVD_B200_H
#define DVD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVD_ABI_VERSION 5

#if defined(__GNUC__)
#define DVD_API __attribute__((visibility("default")))
#else
#define DVD_API
#endif

#define DVD_E_BADARG   (-1)   /* null pointer, bad shape, misalignment               */
#define DVD_E_ARCH     (-2)   /* device is not sm_100                                 */
#define DVD_E_WORKSPACE (-3)  /* workspace too small                                  */
#define DVD_E_NOTMA    (-4)   /* driver entry point for tensor maps unavailable       */

/* precision of the denoiser's dense contractions */
#define DVD_PREC_FP32  0      /* fp32 FFMA reference mode (bit-for-bit reproducible)   */
#define DVD_PREC_BF16  1      /* bf16 operands, fp32 accumulate on tcgen05 / TMEM (fast, reduced accuracy)        */
#define DVD_PREC_BF16X3 2     /* fp32-accurate tensor-core mode: GEMM operands are bf16 pairs hi+lo and run three */
                              /* tcgen05 passes (hi*hi + lo*hi + hi*lo, error ~2^-16); the pyramid and the        */
                              /* decoder's q|k|v run two (fp16 activation x fp16 weight pair); attention in fp16   */

/* One dense weight matrix W[n][k] (row-major, K contiguous == torch Linear layout). */
typedef struct dvd_mat {
  const float* f32;           /* always present                                       */
  const void*  bf16;          /* bf16(W) for the tensor modes (may be NULL in fp32)    */
  const void*  bf16_lo;       /* bf16(W - bf16(W)) where a precision runs this matrix on bf16 pairs (DVD_PREC_BF16X3), else NULL */
  int32_t n, k;
} dvd_mat_t;

typedef struct dvd_dec_layer {          /* CA:343-396 DecoderLayer, CA:13-57 feed-forward */
  const float *n1_w, *n1_b;             /* norm1 (eps 1e-5)                               */
  dvd_mat_t qkv;                        /* [4608,1536] = linear_q ‖ linear_k ‖ linear_v   */
  dvd_mat_t fc;                         /* [1536,1536]                                    */
  const float *n2_w, *n2_b;
  dvd_mat_t conv1;                      /* [2048,1536]                                    */
  const float *bn1_scale, *bn1_shift;   /* eval-mode BN folded: y = x*scale + shift       */
  const float *dw_w;                    /* depthwise 3x3 weights, tap-major [9][2048]     */
  const float *bn2_scale, *bn2_shift;
  dvd_mat_t conv2;                      /* [1536,2048]                                    */
  const float *bn3_scale, *bn3_shift;
  /* LayerNorm folded into the consumer GEMM, required for DVD_PREC_BF16X3 (which reads these instead of qkv / conv1): W' = W * gamma
   * (per input channel), colsum[n] = sum_k W'[n][k] of the ROUNDED pair, cvec = W beta.  The epilogue computes
   * rstd * (x W'^T - mean * colsum) + cvec from the raw residual rows. */
  dvd_mat_t qkv_ln;                     /* [4608,1536] = qkv * norm1.weight, as an IEEE fp16 hi / lo pair (two-pass GEMM on fp16 raw rows) */
  const float *qkv_colsum, *qkv_cvec;   /* [4608]                                         */
  dvd_mat_t conv1_ln;                   /* [2048,1536] = conv1 * norm2.weight             */
  const float *conv1_colsum, *conv1_cvec;   /* [2048]                                     */
} dvd_dec_layer_t;

/* Packed weights of the live part of DiT-S/2 (tv=True): CM:361-459.  Blocks 0..10 are dead
 * (CM:614-616 never re-assigns x) and are not part of this table. */
typedef struct dvd_weights {
  const float* pos;                     /* noised_obs_pos_embed [1024,384]                 */
  dvd_mat_t pyr[7];                     /* conv3x3 weights repacked [Cout][ky][kx][Cin]    */
  const float* pyr_b[7];
  dvd_mat_t emb[5];                     /* obs, r, c, m, l patch-embed  [384, 4C]          */
  const float* emb_b[5];
  dvd_mat_t t_mlp0, t_mlp2;  const float *t_mlp0_b, *t_mlp2_b;          /* CM:97-139       */
  dvd_mat_t blk_ada;         const float* blk_ada_b;                   /* [2304,384]       */
  dvd_mat_t xattn_in;        const float* xattn_in_b;                  /* [1152,384] q‖k‖v */
  dvd_mat_t xattn_out;       const float* xattn_out_b;
  dvd_mat_t blk_qkv;         const float* blk_qkv_b;                   /* [1152,384]       */
  dvd_mat_t blk_proj;        const float* blk_proj_b;
  dvd_mat_t blk_fc1;         const float* blk_fc1_b;                   /* [1536,384]       */
  dvd_mat_t blk_fc2;         const float* blk_fc2_b;                   /* [384,1536]       */
  const float *dec_hpe, *dec_wpe;       /* sinusoid tables, position-major [32][1536]      */
  dvd_mat_t h_scale0, h_scale2, w_scale0, w_scale2;                    /* CA:136-141       */
  const float *h_scale0_b, *h_scale2_b, *w_scale0_b, *w_scale2_b;
  dvd_dec_layer_t dec[6];
  const float *dec_ln_w, *dec_ln_b;     /* decoder.layer_norm (eps 1e-5)                   */
  dvd_mat_t fin;             const float* fin_b;                       /* [8,1536]         */
  dvd_mat_t fin_ada;         const float* fin_ada_b;                   /* [3072,1536]      */
  /* Required for DVD_PREC_BF16X3: the pyramid weights (same packing as pyr[], level 0 K-padded to 64) as IEEE fp16 hi / lo pairs in
   * the bf16 / bf16_lo slots.  That precision runs the pyramid in two tensor passes (ONE fp16 activation x weight pair; the oracle study
   * finds no measurable map error from fp16 pyramid activations) and reads pyr[].bf16 / .bf16_lo not at all. */
  dvd_mat_t pyr_h[7];
} dvd_weights_t;

/* Per-step conditioning table row (floats): temb[384] ‖ block adaLN[2304] ‖ final adaLN[3072]. */
#define DVD_TABLE_ROW (384 + 2304 + 3072)

DVD_API int         dvd_version(void);
DVD_API const char* dvd_last_error(void);
/* 0 if the current device can run this library (compute capability 10.x). */
DVD_API int         dvd_check_device(void);

/* ---- unwarp: EV:300-306 (upsample map + base ramp + 0.987 affine) fused with WP:73 grid_sample.
 * photo [B,C,H,W] fp32, map [B,2,mh,mw] fp32 displacement field in [-1,1]; out [B,C,H,W] fp32.  */
DVD_API int dvd_unwarp_f32(const float* photo, const float* map, float* out, int B, int C, int H, int W,
                   int mh, int mw, float affine, void* stream);
/* uint8 variant: photo/out are HWC uint8 [B,H,W,C] (C<=4); the result is truncated like
 * visualization_utils.py:76-77 `.astype(np.uint8)`. */
DVD_API int dvd_unwarp_u8(const uint8_t* photo, const float* map, uint8_t* out, int B, int C, int H, int W,
                  int mh, int mw, float affine, void* stream);
/* fp32 NCHW photo in, uint8 HWC out (the reference's tensor types at both ends of visualize_dewarping). */
DVD_API int dvd_unwarp_f32_u8(const float* photo, const float* map, uint8_t* out, int B, int C, int H, int W,
                      int mh, int mw, float affine, void* stream);
/* Mixed-size uint8 HWC batch: documents of different sizes in ONE launch (same result, byte for byte, as dvd_unwarp_u8 on each
 * document alone).  The caller owns a table in device memory: dvd_unwarp_u8_plan fills it in HOST memory (pinned, for an async
 * upload; no CUDA call, so it can run while earlier work is in flight), the caller copies it to the device, and dvd_unwarp_u8_mixed
 * launches.  The launch reads the table on the device only, so a CUDA graph captured once serves every composition planned into
 * the same device table.  Document d reads map row d of map [n_docs,2,mh,mw]; empty documents (H or W = 0) are allowed. */
typedef struct dvd_unwarp_doc {
  const uint8_t* photo;                 /* [H,W,C] uint8, device (NULL allowed when H or W is 0) */
  uint8_t* out;                         /* [H,W,C] uint8, device                                 */
  int32_t H, W;
} dvd_unwarp_doc_t;
/* bytes of a table for up to max_docs documents */
DVD_API size_t dvd_unwarp_table_bytes(int max_docs);
/* host only: validates (C in 1..4, H,W >= 0, H*W*C < 2^31, non-NULL pointers of non-empty documents, table_bytes large enough) and
 * fills table_host; *total_tiles (may be NULL) = the number of 128x8 tiles of the batch. */
DVD_API int dvd_unwarp_u8_plan(const dvd_unwarp_doc_t* docs_host, int n_docs, int C, int mh, int mw, float affine,
                               void* table_host, size_t table_bytes, long long* total_tiles);
/* one launch; table = the uploaded plan; C must equal the planned C (a table planned for another C is ignored: nothing is written) */
DVD_API int dvd_unwarp_u8_mixed(const void* table, int C, const float* map, void* stream);
/* Sized uint8 HWC batch: document d dewarps its H x W photo into an Ho x Wo output (any size, per document) in ONE launch, with
 * the table design of the mixed-size batch above (host plan -> device copy -> launch; a graph captured once serves every plan).
 * With supersampling factor s the output is the mean of each s x s block of the reference chain evaluated at s*Ho x s*Wo:
 *   out = trunc(avg_pool2d(grid_sample(photo, fullres_grid(map[d], s*Ho, s*Wo)), s))
 * s = 1 and Ho x Wo = H x W is dvd_unwarp_u8, byte for byte.  supersample = 0 picks s = min(8, max(1, ceil(H/Ho), ceil(W/Wo))).
 * A document with H, W, Ho or Wo = 0 is empty (owns no tile; its pointers may be NULL). */
typedef struct dvd_unwarp_sized_doc {
  const uint8_t* photo;                 /* [H,W,C] uint8, device   */
  uint8_t* out;                         /* [Ho,Wo,C] uint8, device */
  int32_t H, W;                         /* photo                   */
  int32_t Ho, Wo;                       /* output                  */
  int32_t supersample;                  /* 0 = auto, 1..8          */
  int32_t pad;
} dvd_unwarp_sized_doc_t;
/* bytes of a sized table for up to max_docs documents */
DVD_API size_t dvd_unwarp_sized_table_bytes(int max_docs);
/* host only: validates (C in 1..4, sizes >= 0, supersample in 0..8, H*W*C and Ho*Wo*C < 2^31, non-NULL pointers of non-empty
 * documents, table_bytes large enough, map size) and fills table_host; *total_tiles (may be NULL) = the tiles of the batch,
 * supersample_out[d] (may be NULL) = the factor chosen for document d. */
DVD_API int dvd_unwarp_u8_sized_plan(const dvd_unwarp_sized_doc_t* docs_host, int n_docs, int C, int mh, int mw, float affine,
                                     void* table_host, size_t table_bytes, long long* total_tiles, int32_t* supersample_out);
/* one launch; a table planned for another C is ignored (nothing is written) */
DVD_API int dvd_unwarp_u8_sized(const void* table, int C, const float* map, void* stream);

/* ---- input preparation: the denoiser's y512 [docs,3,512,512] from the uint8 HWC RGB photo (the reference loader's
 * cv2.resize(photo, (512, 512), INTER_LINEAR) / 255, byte for byte: OpenCV's fixed-point bilinear resize, then an IEEE division
 * by 255).  Photos of any sizes (at least 1x1) in ONE launch, with the table design of the mixed-size unwarp: dvd_y512_u8_plan
 * fills the table in host memory (no CUDA call), the caller copies it to the device, dvd_y512_u8 launches; a CUDA graph captured
 * once serves every batch planned into the same device table. */
typedef struct dvd_y512_doc {
  const uint8_t* photo;                 /* [H,W,3] uint8, device */
  int32_t H, W;
} dvd_y512_doc_t;
/* bytes of a table for up to max_docs documents */
DVD_API size_t dvd_y512_table_bytes(int max_docs);
/* host only: validates (H, W >= 1, H*W*3 < 2^31, non-NULL photos, table_bytes large enough) and fills table_host */
DVD_API int dvd_y512_u8_plan(const dvd_y512_doc_t* docs_host, int n_docs, void* table_host, size_t table_bytes);
/* one launch; writes documents 0..n_docs-1 of y512 [>= n_docs,3,512,512] fp32 and nothing else */
DVD_API int dvd_y512_u8(const void* table, float* y512, void* stream);
/* WP:14-23,50-73 register_model2 / SpatialTransformer2: generic bilinear grid_sample,
 * align_corners=True, zeros padding.  img [B,C,H,W], grid [B,2,Ho,Wo] (ch0=x, ch1=y), out [B,C,Ho,Wo]. */
DVD_API int dvd_grid_sample_f32(const float* img, const float* grid, float* out, int B, int C, int H, int W,
                        int Ho, int Wo, void* stream);
/* EV:301-306 only: materialise the full-resolution sampling grid [B,2,H,W] (parity checks). */
DVD_API int dvd_fullres_grid_f32(const float* map, float* grid, int B, int H, int W, int mh, int mw,
                         float affine, void* stream);

/* ---- denoiser + sampler ------------------------------------------------------------------- */
DVD_API size_t dvd_workspace_bytes(int docs, int n_hyp, int precision);

/* CM:97-139 + CM:209-211 + CM:331: conditioning tables for `n_steps` scalar timesteps
 * (values AFTER the CM:575-579 remap).  tables [n_steps][DVD_TABLE_ROW]. */
DVD_API int dvd_tables_init(const dvd_weights_t* w, const float* t_values_host, int n_steps, float* tables,
                    void* stream);

/* Step-invariant, hypothesis-invariant work for `docs` documents (CM:585-594,605 and the K/V
 * projections of CM:237-257): pyramid, c/m/l patch embeds, static cross-attention K/V.
 * y512 [docs,3,512,512], mask_cat [docs,1,512,512], mask_y512 [docs,384,64,64], line_msk [docs,64,64,64]. */
DVD_API int dvd_static_forward(const dvd_weights_t* w, void* workspace, size_t workspace_bytes, int docs,
                       int n_hyp, int precision, const float* y512, const float* mask_cat,
                       const float* mask_y512, const float* line_msk, void* stream);

/* One denoiser forward + DDIM update for docs*n_hyp samples: CM:568-647 + GD:445-491,618-624.
 *   x_t       [docs*n_hyp,2,64,64]  current sample (document-major, hypothesis-minor)
 *   init_flow [docs*n_hyp,2,64,64]
 *   init_feat NULL  -> warp the pyramid feature with (init_flow+base64)*2-1 (GD:618-624) unless
 *             `feat_is_init` (CM:597-598, t>600) in which case the un-warped feature is used;
 *             non-NULL -> explicit [docs*n_hyp,256,64,64] NCHW tensor (drop-in model() calls).
 *   table_row one row of dvd_tables_init's output for this step
 *   pred_x0   [docs*n_hyp,2,64,64] out ; x_prev [docs*n_hyp,2,64,64] out (a*pred + b*x_t), may be NULL */
DVD_API int dvd_denoise_step(const dvd_weights_t* w, void* workspace, size_t workspace_bytes, int docs,
                     int n_hyp, int precision, const float* x_t, const float* init_flow,
                     const float* init_feat, int feat_is_init, const float* table_row,
                     float ddim_a, float ddim_b, float* pred_x0, float* x_prev, void* stream);

/* GD:639-640 + EV:137: mean over the hypotheses of each document, clamp to [-1,1]. */
DVD_API int dvd_hyp_mean_clamp(const float* pred_x0, float* out, int docs, int n_hyp, void* stream);

/* Whole S-step loop (GD:537-645) for `docs` documents after dvd_static_forward:
 *   x_T [docs*n_hyp,2,64,64]; init_flow0 [docs,2,64,64] (zeros in the default config);
 *   tables [S][DVD_TABLE_ROW] ordered by loop iteration (i = S-1 .. 0); t_scaled_host[S] the
 *   rescaled timesteps of RS:111-123 in the same order; ddim_a/b_host[S]; map_out [docs,2,64,64];
 *   init_feat0 [docs,256,64,64] or NULL (= zeros, EV:167): only read when the FIRST step has t <= 600. */
DVD_API int dvd_sample(const dvd_weights_t* w, void* workspace, size_t workspace_bytes, int docs, int n_hyp,
               int precision, const float* x_T, const float* init_flow0, const float* tables,
               const float* t_scaled_host, const float* ddim_a_host, const float* ddim_b_host,
               int S, const float* init_feat0, float* map_out, void* stream);

/* NHWC pyramid feature of the last dvd_static_forward: returns a pointer INSIDE the workspace,
 * [docs,64,64,256] fp32 (for the 'feat_dict' entry the reference sampler returns). */
DVD_API const float* dvd_workspace_feat(void* workspace, int docs, int n_hyp, int precision);

/* named fp32 intermediate inside the workspace (stage-level parity tests): "feat","cond","msk6","msk_line",
 * "kv_cond","xe","r","q","kv_r","xo","xs","qkv","X","qkv_d","att_d","f1","a_r","pe"; NULL if unknown. */
DVD_API const float* dvd_workspace_tensor(void* workspace, int docs, int n_hyp, int precision, const char* name,
                                          long long* numel);

/* test hook: make dvd_denoise_step (of the calling thread) return after a stage so that its output can be read with
 * dvd_workspace_tensor("X"): 0 = off, 1 = DiT block (X = x1|x2|x3|x4, CM:623), 2 = adaptive positional encoding (CA:143-157),
 * 3 + l = decoder layer l (CA:377-396). */
DVD_API int dvd_debug_stop_after(int stage);

/* ---- building blocks exported for parity tests (not needed by the reference-side binding) ---- */
DVD_API int dvd_test_gemm(const float* A, const float* W, const float* bias, float* C, int M, int N, int K,
                  int precision, void* scratch, size_t scratch_bytes, void* stream);
DVD_API int dvd_test_attention(const float* q, const float* k, const float* v, float* o, int batch, int heads,
                       int T, int d, float scale, int precision, void* scratch, size_t scratch_bytes,
                       void* stream);
/* Tensor-core attention on caller-prepared 16-bit operands, exactly the launch dvd_denoise_step makes:
 * q [nsamp*T, ldq]; context i: k[i] [nsamp/kv_div[i]*T, ldk], vt[i] = V^T [nsamp/kv_div[i], heads*d, T], o[i] (+ o_lo[i]) [nsamp*T, ldo].
 * nctx == 1: the kernel attention_tc selects (the CTA pair for d = 256 unless DVD_ATTN_V1=1); nctx 2..4: one multi-context launch.
 * f16: IEEE fp16 operands (DVD_PREC_BF16X3), else bf16.  k, vt, o, o_lo (may be NULL) and kv_div are HOST arrays of nctx entries.
 * Every argument is checked before any CUDA call. */
DVD_API int dvd_test_attention_tc(const void* q, int ldq, const void* const* k, int ldk, const void* const* vt, void* const* o,
                                  void* const* o_lo, int ldo, const int* kv_div, int nctx, int nsamp, int heads, int T, int d,
                                  float scale, int f16, void* stream);
/* Depthwise 3x3 (pad 1) over the 32x32 token grid + folded BN + ReLU as the decoder runs it in the tensor modes: in_hi / in_lo
 * [N,1024,C] bf16 (value = hi + lo; in_lo NULL: hi alone), w9 [9,C] fp32 (tap ky*3+kx), scale / shift [C] fp32, out_hi / out_lo
 * [N,1024,C] bf16 pair of the result (out_lo may be NULL).  C must be a multiple of 64, N > 0, every pointer 16-byte aligned. */
DVD_API int dvd_test_dwconv(const void* in_hi, const void* in_lo, const float* w9, const float* scale, const float* shift,
                            void* out_hi, void* out_lo, int N, int C, void* stream);
/* Plain tensor-core GEMM (tuning / micro-benchmarks): out = A[M,K] W[N,K]^T + bias; bf16 operands (A16_lo / W16_lo non-NULL:
 * split pairs, three passes; A16_lo NULL next to a weight pair: A16, W16 and W16_lo hold IEEE fp16, two passes), bf16 and/or fp32 output.
 * dvd_test_gemm accepts precision 3 for the same two-pass mode (fp16 activation x fp16 weight pair). */
DVD_API int dvd_gemm_bf16(const void* A16, const void* A16_lo, int lda, const void* W16, const void* W16_lo, int ldw,
                          const float* bias, void* out16, float* out32, int M, int N, int K, void* stream);
/* Same with the decoder's epilogue pieces: folded-BN scale / shift (NULL: none), ReLU, a split-pair 16-bit output (out16_lo) and an
 * fp32 residual (resid may alias out32). */
DVD_API int dvd_gemm_tune(const void* A16, const void* A16_lo, int lda, const void* W16, const void* W16_lo, int ldw,
                          const float* bias, const float* scale, const float* shift, int relu, void* out16, void* out16_lo,
                          float* out32, const float* resid, int M, int N, int K, void* stream);
/* Kernel-class profiler: between begin/end every dense contraction launched by this thread is bracketed by CUDA
 * events.  end() synchronises and returns, for the classes {0: GEMM, 1: attention, 2: pyramid conv}, the summed
 * device time (ms), algorithmic FLOPs (2 M N K), launch counts and the FLOPs the tensor pipe executed (the split-precision
 * mode runs three passes per k-step, two in the q|k|v GEMM of the decoder).  Any output pointer may be NULL. */
DVD_API int dvd_profile_begin(void);
DVD_API int dvd_profile_end(double* ms, double* flops, long long* launches, double* executed_flops);
/* number of kernel launches issued by this library on this thread since the last reset */
DVD_API long long dvd_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* DVD_B200_H */
