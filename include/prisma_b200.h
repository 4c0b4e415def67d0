/*
 * prisma_b200.h -- C ABI of libprisma_b200.so (sm_100a).
 *
 * The reference (Prisma-Multimodal/ViT-Prisma) has no FFI: its two hot paths are Python
 * methods that hand every flop to PyTorch ATen.  This header is the boundary a maintainer
 * binds instead (ctypes stub in INTEGRATION.md): plain pointers + sizes + a CUDA stream,
 * no torch types.  Every entry point names the reference code it stands in for
 * (paths relative to /root/reference/src/vit_prisma).
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - matrices are row-major; "ld*" are row strides in ELEMENTS;
 *   - weights enter GEMMs "K-major": B is [N][K] (one output column's weights contiguous);
 *   - return 0 on success, a negative PB_E* code otherwise; pb_last_error() gives the text.
 *     Nothing throws, nothing falls back to a CPU path.
 *   - launches go to the stream passed in; no internal host threads, no hidden syncs.
 */
#ifndef PRISMA_B200_H
#define PRISMA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* pb_stream_t; /* == cudaStream_t */

#if defined(__GNUC__)
#define PB_API __attribute__((visibility("default")))
#else
#define PB_API
#endif

enum { PB_OK = 0, PB_EINVAL = -1, PB_ECUDA = -2, PB_EUNSUPPORTED = -3, PB_ENODEVICE = -4 };
enum { PB_F32 = 0, PB_BF16 = 1 };
/* activation_name of HookedViTConfig (models/layers/mlp.py:41-62, models/activation_fns.py:19-58) */
enum { PB_ACT_NONE = 0, PB_ACT_RELU = 1, PB_ACT_GELU = 2, PB_ACT_SILU = 3, PB_ACT_GELU_NEW = 4,
       PB_ACT_GELU_FAST = 5, PB_ACT_QUICK_GELU = 6, PB_ACT_TANH_RELU = 7, PB_ACT_EXP = 8 };
enum { PB_GEMM_AUTO = 0, PB_GEMM_SIMT = 1, PB_GEMM_TC = 2 };

/* ---------------------------------------------------------------- library */
PB_API int pb_version(void);
PB_API const char* pb_last_error(void);
/* number of CUDA kernels this library has launched in this process (monotonic; bench.py's gpu_launches) */
PB_API unsigned long long pb_launch_count(void);
/* fills sm count / compute capability of the current device; PB_ENODEVICE without a GPU */
PB_API int pb_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* sizeof() of the ABI structs as compiled (0 PbGemm, 1 PbLayerNorm, 2 PbAttention, 3 PbVitLayerW,
 * 4 PbVitLayerSpill, 5 PbVitForward, ...; -1 for an unknown index): lets a binding verify its layout */
PB_API int pb_abi_sizeof(int which);

/* ------------------------------------------------------------------- GEMM
 * out = A[M,K] @ B[N,K]^T (+bias), fp32 accumulate.  Stands in for every
 * fancy_einsum/einops.einsum contraction on the two paths:
 *   models/layers/attention.py:158-244 (Q/K/V/O), mlp.py:69,78, head.py:31,
 *   patch_embedding.py:14-32 (stride==kernel conv as a GEMM), sae/sae.py:568,585.
 * Epilogue: out0 = acc + bias                       (the "pre" hook point; NULL = skip)
 *           out1 = act(out0)  or  residual + out0   (NULL = skip)
 * With n_split > 1 the N axis is cut into n_split blocks of split_n columns and block j
 * of out0 goes to out_split[j] (row stride ld0): one launch fills hook_q / hook_k / hook_v.
 * dtype PB_F32 : impl SIMT  -> exact fp32 FFMA;
 *                impl TC    -> tcgen05 kind::tf32 in 3 passes (A, A_lo, B, B_lo all required;
 *                              *_lo = x - tf32_trunc(x), see pb_split_tf32) ~fp32 accuracy.
 * dtype PB_BF16: impl TC    -> tcgen05 kind::f16 (bf16 in, fp32 accumulate in TMEM).
 * impl AUTO picks TC when the shape/alignment allows it, else SIMT.                         */
typedef struct {
  int32_t M, N, K;
  int32_t dtype, act, impl;
  const void* A;  int64_t lda;
  const void* B;  int64_t ldb;
  const void* A_lo; const void* B_lo;
  const void* bias;
  const void* residual; int64_t ldr;
  void* out0; int64_t ld0;
  void* out1; int64_t ld1;
  float* out1_lo;                    /* F32 only: tf32 residual of out1 (row stride ld1), or NULL */
  int32_t n_split, split_n;
  void* out_split[4];
} PbGemm;
PB_API int pb_gemm(const PbGemm* g, pb_stream_t stream);
/* lo[i] = x[i] - float(tf32_trunc(x[i]))  (the residual operand of the 3xTF32 scheme) */
PB_API int pb_split_tf32(const float* x, float* lo, int64_t n, pb_stream_t stream);

/* -------------------------------------------------------------- LayerNorm
 * models/layers/layer_norm.py:27-45 (LayerNormPre: w == b == NULL) and :75-93 (LayerNorm):
 *   xc = x - mean(x);  scale = sqrt(mean(xc^2) + eps);  y = xc/scale * w + b
 * x is read in dtype_in, arithmetic is fp32 (the reference upcasts non-fp32 inputs).
 *   scale     fp32 [rows]            -> hook_scale        (NULL = skip)
 *   norm_f32  fp32 [rows, cols]      -> hook_normalized when dtype_out != F32 (NULL = skip)
 *   out       dtype_out [rows, cols] -> the tensor downstream code consumes
 *   out_lo    fp32 [rows, cols]      -> tf32 residual of out for a following 3xTF32 GEMM
 *   scale_in  fp32 [rows] or NULL    -> when given, divide by THIS scale instead of the computed one
 *                                       (a user hook replaced / edited hook_scale's value)        */
typedef struct {
  int64_t rows; int32_t cols;
  int32_t dtype_in, dtype_out;
  float eps;
  const void* x; const void* w; const void* b;
  float* scale; float* norm_f32; void* out; float* out_lo;
  const float* scale_in;
} PbLayerNorm;
PB_API int pb_layernorm(const PbLayerNorm* p, pb_stream_t stream);

/* -------------------------------------------------------------- Attention
 * models/layers/attention.py:126-184, 246-281.  q,k,v,z: [B,T,H,dh]; scores,pattern: [B,H,T,T].
 *   scores  = q k^T / attn_scale          (hook_attn_scores; NULL = not materialised)
 *   pattern = softmax(scores), NaN -> 0   (hook_pattern;     NULL = not materialised)
 *   z       = pattern v                   (hook_z)
 * pb_attention runs all three in one kernel; the three split entry points exist for the
 * hooked path where user code may edit scores / pattern between the steps.               */
typedef struct {
  int32_t B, T, H, dh, dtype;
  float attn_scale;
  const void* q; const void* k; const void* v;
  void* scores; void* pattern; void* z;
} PbAttention;
PB_API int pb_attention(const PbAttention* p, pb_stream_t stream);
PB_API int pb_attn_scores(const PbAttention* p, pb_stream_t stream);              /* q,k -> scores   */
PB_API int pb_softmax_rows(const void* x, void* y, int64_t rows, int32_t cols, int32_t dtype,
                    pb_stream_t stream);                                   /* softmax, NaN->0 */
PB_API int pb_attn_pv(const PbAttention* p, pb_stream_t stream);                  /* pattern,v -> z  */

/* ------------------------------------------------------------ element-wise */
PB_API int pb_add(const void* a, const void* b, void* out, int64_t n, int32_t dtype, pb_stream_t s);
PB_API int pb_mul(const void* a, const void* b, void* out, int64_t n, int32_t dtype, pb_stream_t s);
PB_API int pb_activation(const void* x, void* y, int64_t n, int32_t act, int32_t dtype, pb_stream_t s);
/* out[r,:] = x[r,:] / max(||x[r,:]||_2, eps)     (F.normalize, models/base_vit.py:214-215) */
PB_API int pb_l2_normalize_rows(const void* x, void* out, int64_t rows, int32_t cols, float eps,
                         int32_t dtype, pb_stream_t s);
/* out[b,:] = mean_t x[b,t,:]                      (classification_type "gaap", base_vit.py:195-198) */
PB_API int pb_mean_tokens(const void* x, void* out, int32_t B, int32_t T, int32_t d, int32_t dtype,
                   pb_stream_t s);
/* images [B,C,S,S] -> patches [B*(S/P)^2, C*P*P] in conv-weight order (patch_embedding.py:26-32) */
PB_API int pb_im2col_patches(const void* images, void* patches, int32_t B, int32_t C, int32_t S,
                      int32_t P, int32_t dtype, pb_stream_t s);
/* full[b,0,:] = cls + pos[0];  full[b,1+i,:] = embed[b,i,:] + pos[1+i]  (base_vit.py:171-179)
 * with use_cls == 0: full[b,i,:] = embed[b,i,:] + pos[i]                                  */
PB_API int pb_embed_assemble(const void* embed, const void* cls, const void* pos, void* full,
                      int32_t B, int32_t n_patches, int32_t d, int32_t use_cls, int32_t dtype,
                      pb_stream_t s);
PB_API int pb_cast(const void* x, int32_t dtype_in, void* y, int32_t dtype_out, int64_t n, pb_stream_t s);

/* ------------------------------------------------ fused HookedViT forward
 * One call = HookedViT.forward (models/base_vit.py:152-217) with every requested HookPoint
 * activation spilled to its destination (prisma_tools/hooked_root_module.py:289-332 _save_hook).
 * Weight pointers are the K-major packs built by the host (vit_prisma/b200/vit_engine.py):
 *   wqkv [3*H*dh][d]  rows: q heads, k heads, v heads  <- W_Q/W_K/W_V [H,d,dh]
 *   wo   [d][H*dh]                                     <- W_O [H,dh,d]
 *   win  [d_mlp][d], wout [d][d_mlp]                   <- W_in [d,d_mlp], W_out [d_mlp,d]
 * A NULL spill pointer means "hook point not requested": the tensor is then never written to
 * HBM unless a later kernel needs it, in which case the host passes a scratch pointer.      */
typedef struct {
  const void *ln1_w, *ln1_b, *wqkv, *wqkv_lo, *bqkv, *wo, *wo_lo, *bo;
  const void *ln2_w, *ln2_b, *win, *win_lo, *bin, *wout, *wout_lo, *bout;
} PbVitLayerW;

typedef struct {
  float* ln1_scale;  float* ln1_norm_f32;  void* ln1_out;
  void *q, *k, *v;
  void *scores, *pattern;
  void* z;
  void* attn_out;    void* resid_mid;
  float* ln2_scale;  float* ln2_norm_f32;  void* ln2_out;
  void* pre;         void* post;
  void* mlp_out;     void* resid_post;
} PbVitLayerSpill;

typedef struct {
  /* geometry */
  int32_t batch, n_channels, image_size, patch_size, n_patches, n_tokens;
  int32_t d_model, n_heads, d_head, d_mlp, n_classes;
  int32_t n_layers_run;      /* blocks executed (stop_at_layer) */
  int32_t run_head;          /* 0: return residual after the last executed block */
  int32_t use_cls, layer_norm_pre, normalize_output, head_proj /* return_type != pre_logits */;
  int32_t pool_gaap;         /* classification_type: 0 = cls token (row 0), 1 = mean over tokens */
  int32_t act, dtype, gemm_impl;
  float eps, attn_scale;
  /* inputs + weights */
  const void* images;
  const void *patch_w, *patch_w_lo, *patch_b, *cls, *pos;
  const void *lnpre_w, *lnpre_b, *lnf_w, *lnf_b, *head_w, *head_w_lo, *head_b;
  const PbVitLayerW* layers_host;        /* HOST array [n_layers_run] */
  /* spill destinations / work buffers */
  void* patches;             /* [B*n_patches, C*P*P] im2col scratch                         */
  void* embed;               /* hook_embed [B,n_patches,d]                                  */
  void* full_embed;          /* hook_full_embed == residual before ln_pre [B,T,d]           */
  float* lnpre_scale; float* lnpre_norm_f32; void* lnpre_out;    /* residual fed to block 0 */
  const PbVitLayerSpill* spills_host;    /* HOST array [n_layers_run] */
  float* lnf_scale; float* lnf_norm_f32; void* lnf_out;
  void* pooled;              /* [B,d] cls/gaap-pooled ln_final output                       */
  void* pre_normalize;       /* hook_post_head_pre_normalize [B, n_classes or d]            */
  void* out;                 /* model output                                                */
  float* lo_scratch;         /* fp32 [max(B*T*(d + max(d_mlp, H*dh)), B*n_patches*C*P*P)]: tf32 residuals of the
                                GEMM A operands in 3xTF32 mode, or NULL (then fp32 GEMMs run on the exact FFMA path) */
} PbVitForward;
PB_API int pb_vit_forward(const PbVitForward* f, pb_stream_t stream);

/* ------------------------------------------------------- TopK SAE training step
 * Stands in for StandardSparseAutoencoder.forward + VisionSAETrainer.train_step
 * (sae/sae.py:557-645, 144-149, 275-297; sae/train_sae.py:278-411) with activation_fn_str == "topk".
 * All buffers fp32 unless noted; F = d_sae, d = d_in.  The encoder is stored feature-major:
 * W_encT [F][d] (the module's W_enc [d,F] parameter is a transposed view of the same memory).
 * One step = pb_sae_prep -> pb_gemm (hidden_pre = sae_in @ W_encT^T + b_enc) -> pb_sae_topk ->
 *            pb_sae_decode -> pb_sae_backward -> pb_sae_adam, all on one stream, no host sync.      */
typedef struct {
  int32_t rows, d, F, k;
  int32_t norm_mode;        /* cfg.normalize_activations: 0 none, 1 "layer_norm", 2 "constant_norm_rescale" */
  int32_t training;         /* 0: decode + loss only */
  int32_t step;             /* optimizer step count t >= 1 (Adam bias correction) */
  int32_t renorm_decoder;   /* 1: leave W_dec rows unit-norm after the update (= next step's set_decoder_norm_to_unit_norm) */
  float lr, beta1, beta2, adam_eps, max_grad_norm /* <= 0: no clipping */;
  /* inputs / parameters */
  const float* x;           /* [rows][d] raw activations */
  float* W_encT; float* W_encT_lo /* tf32 residual plane of the dense 3xTF32 encoder; may be NULL */; float* W_dec; float* b_enc; float* b_dec;
  /* per-step work buffers */
  float *sae_in, *mu, *sd, *xsum;            /* [rows][d], [rows], [rows], [d] (written by pb_sae_prep) */
  int32_t* idx; float* val;                  /* [rows][k] TopK support of hidden_pre (written by pb_sae_topk) */
  float* feat_count;                         /* [F] selections per feature this step (zero it before pb_sae_topk) */
  float *sae_out, *g, *dval;                 /* [rows][d] (optional), [rows][d], [rows][k] */
  int32_t *csc_off, *csc_cursor, *csc_entries;  /* [F+1], [F], [rows*k] */
  float *gW_dec, *gW_encT, *gb_enc, *gb_dec;  /* gradients [F][d], [F][d], [F], [d] */
  float *gcol, *gbdec2;                      /* [d] scratch */
  float* fired;                              /* [F] number of tokens with a positive activation of feature f */
  void* scalars;                             /* 8 floats: loss_sum, gnorm_sq, clip_coef, mse, l0, pos_count, grad_norm, - (zero before the step) */
  /* optimizer + bookkeeping state */
  float *m_dec, *v_dec, *m_enc, *v_enc, *m_be, *v_be, *m_bd, *v_bd;
  float* since_fired; float* act_freq;       /* [F] n_forward_passes_since_fired, act_freq_scores (train_sae.py:356-361); may be NULL */
  /* data parallel (p2p.cu): tokens of the GLOBAL batch (0 = rows) for the 1/(tokens*d) of the mean loss; dist = 1 makes
   * pb_sae_backward stop after the local gradients (norm / clip / Adam then run in pb_p2p_*), and xsum must already hold the
   * GLOBAL column sums of x when pb_sae_decode runs (pb_p2p_sum_xsum)                                                     */
  int32_t global_rows; int32_t dist;
  /* scratch of pb_sae_backward for features selected by more than 64 tokens (their lists are split across warps):
   * work_bytes >= 8 + 4*F + 8*(rows*k/32 + F + 1)                                                                        */
  void* work; int64_t work_bytes;
  /* [2] max_f ||W_encT[f,:]||_2 and max_f ||W_encT[f,:] - f16(.)||_2 AFTER this step's update, for the fused encoder's error bound
   * (pb_sae_encode_topk_fused); may be NULL                                                                               */
  float* enc_norm_max;
  /* 1: pb_sae_step_reset already zeroed gcol / gbdec2 / the work header for this step (pb_sae_backward then skips its memsets) */
  int32_t pre_zeroed;
  /* fp16 [F][(d + 7) & ~7] shadow of W_encT for the fused encoder's candidate GEMM, rewritten by pb_sae_adam; may be NULL.
   * f16(x): round to nearest, saturate to +-65504, results below 2^-14 in magnitude flushed to zero                         */
  void* W_encT_h;
} PbSaeStep;

/* sae_in = norm_in(x) - b_dec (+ tf32 residual, fp16 shadow [rows][(d + 7) & ~7] for the fused encoder, row mean / std, column
 * sums of x) -- sae.py:78-87, 557-566; sae_in_lo, sae_in_h, xsum may be NULL                                                */
PB_API int pb_sae_prep(const float* x, const float* b_dec, float* sae_in, float* sae_in_lo, void* sae_in_h, float* mu, float* sd,
                       float* xsum, int32_t rows, int32_t d, int32_t norm_mode, pb_stream_t stream);
/* torch.topk(hidden_pre, k, dim=-1) (sae.py:803-805): idx int32 / val fp32 [rows][k], sorted by value descending,
 * ties broken towards the lower index; feat_count[f] += 1 per selection (may be NULL);
 * scratch >= rows * ceil(F / 24576) * k * 8 bytes when F > 24576, else unused.                     */
PB_API int pb_sae_topk(const float* hidden_pre, int32_t rows, int32_t F, int32_t k, int32_t* idx, float* val,
                       float* feat_count, void* scratch, int64_t scratch_bytes, pb_stream_t stream);
/* dense feature_acts [rows][F] = zeros.scatter_(idx, relu(val)) (sae.py:806-808) -- only for callers that need the dense tensor */
PB_API int pb_sae_scatter_acts(const int32_t* idx, const float* val, float* dense, int32_t rows, int32_t k, int32_t F,
                               int32_t relu, pb_stream_t stream);
/* one launch that zeroes the step's accumulators: feat_count [F], scalars [8], gcol / gbdec2 [d], the header of `work`, and
 * fb_count [2] of the fused encoder (may be NULL)                                                                         */
PB_API int pb_sae_step_reset(const PbSaeStep* s, int32_t* fb_count, pb_stream_t stream);
/* sparse decode + normalised-MSE partials (+ g = dL/d(decoder output) and d(loss)/d(selected pre-activations) when training) */
PB_API int pb_sae_decode(const PbSaeStep* s, pb_stream_t stream);
/* per-feature gradients of W_dec / W_enc / b_enc / b_dec, global grad norm, clip coefficient */
PB_API int pb_sae_backward(const PbSaeStep* s, pb_stream_t stream);
/* clip -> remove decoder-parallel gradient -> Adam -> decoder row renorm -> dead-feature counters */
PB_API int pb_sae_adam(const PbSaeStep* s, pb_stream_t stream);
/* result[0] = mean( (out - x)^2 / ||x - mean_batch(x)||_2,row )  (_compute_mse_loss, sae.py:144-149); xsum_scratch: [d] */
PB_API int pb_sae_mse(const float* x, const float* out, float* xsum_scratch, float* result, int32_t rows, int32_t d,
                      pb_stream_t stream);
/* W[f,:] /= ||W[f,:]|| (set_decoder_norm_to_unit_norm, sae.py:275-277); optional tf32 residual */
PB_API int pb_unit_norm_rows(float* W, float* W_lo, int32_t F, int32_t d, pb_stream_t stream);

/* ------------------------------------------------ fused encoder -> TopK (no dense hidden_pre in HBM)
 * Replaces `hidden_pre = sae_in @ W_enc + b_enc` (sae/sae.py:568-574) + `torch.topk(hidden_pre, k)` (TopK.forward, :803-805) by
 *   phase 1  one-pass fp16 tcgen05 GEMM (kind::f16, fp32 accumulate) on the shadows sae_in_h / W_encT_h, whose epilogue keeps, per token and per 128-feature segment, the c_keep largest
 *            values as packed keys (cand: int32 [rows][d_sae / 128][c_keep]);
 *   phase 2  per token: the m_cand best keys (16 more per round, up to 128, while the proof below fails), EXACT fp32
 *            re-evaluation of those pre-activations, exact top-k of them, and a completeness proof with the per-row bound
 *            |fp16 product - exact| <= ||a - f16(a)|| max_f||w_f|| + ||a|| max_f||w_f - f16(w_f)|| + d 2^-22 ||a|| max_f||w_f||
 *            (operand rounding + fp32 accumulation); rows that fail are listed;
 *   phase 4  exact recomputation + selection for the listed rows (normally none).
 * Same outputs and ordering rules as pb_sae_topk.  phases = 0 runs all three.                                             */
typedef struct {
  int32_t rows, d, F, k;
  int32_t c_keep;               /* 4, 6 or 8 keys kept per (token, 128-feature segment)                                   */
  int32_t m_cand;               /* candidates re-evaluated exactly per token in the first round: k <= m_cand <= 128       */
  int32_t phases;               /* bit mask 1 | 2 | 4 (0 = all); + 8: fb_count was zeroed by the caller (pb_sae_step_reset) */
  float err_coef;               /* safety factor on the error bound; <= 0: default 1.05                                   */
  const float* sae_in;          /* [rows][d]                                                                              */
  const float* W_encT;          /* [F][d] feature-major encoder                                                           */
  const float* b_enc;           /* [F]                                                                                    */
  const float* enc_norm_max;    /* [2] max_f ||W_encT[f,:]||, max_f ||W_encT[f,:] - f16(.)|| (pb_rownorm_max / pb_sae_adam) */
  int32_t* cand; int64_t cand_bytes;
  int32_t* idx; float* val;     /* [rows][k]                                                                              */
  float* feat_count;            /* [F] += selections, may be NULL                                                         */
  int32_t* fb_count;            /* [2]: rows that took the exact path in this call; candidates re-scored over the other rows */
  int32_t* fb_rows;             /* [rows]                                                                                 */
  float* fb_scratch; int64_t fb_scratch_bytes;   /* >= F * 4 bytes; one d_sae row per resident CTA of the exact path      */
  const void* sae_in_h;         /* fp16 [rows][(d + 7) & ~7] = f16(sae_in)  (pb_sae_prep)                                  */
  const void* W_encT_h;         /* fp16 [F][(d + 7) & ~7]    = f16(W_encT)  (pb_rownorm_max / pb_sae_adam)                 */
} PbSaeEncode;
PB_API int pb_sae_fused_workspace(int32_t rows, int32_t F, int32_t c_keep, int64_t* cand_bytes, int64_t* fb_scratch_bytes);
PB_API int pb_sae_encode_topk_fused(const PbSaeEncode* e, pb_stream_t stream);
/* out[0] = max_f ||W[f,:]||_2, out[1] = max_f ||W[f,:] - f16(W[f,:])||_2 over the rows of a contiguous fp32 [F][d] matrix, and
 * (W_h != NULL) the fp16 shadow W_h [F][(d + 7) & ~7] = f16(W): one pass rebuilds everything the fused encoder derives from W */
PB_API int pb_rownorm_max(const float* W, int32_t F, int32_t d, float* out, void* W_h, pb_stream_t stream);

/* ------------------------------------------------ dense SAE step pieces (activation_fn_str = "relu" + L1) and ghost grads
 * StandardSparseAutoencoder.forward with a dense activation executes six [tokens x d_sae x d_in] products
 * (sae/sae.py:568, 585 and their autograd transposes); here they run on pb_gemm, these entry points are the glue between
 * them, and pb_sae_adam finishes the step exactly as in the TopK pipeline.  Ghost grads: sae/sae.py:151-179.          */
/* out[c][r] = in[r][c] (fp32 [rows][cols] -> [cols][rows]); out_lo (optional) = tf32 residual of the transposed values */
PB_API int pb_transpose(const float* in, float* out, float* out_lo, int32_t rows, int32_t cols, pb_stream_t stream);
/* out[c] (+)= sum_r x[r][c]                                    (gb_enc = colsum(d_hidden), sae.py autograd of :568)    */
PB_API int pb_colsum(const float* x, float* out, int32_t rows, int32_t cols, int32_t accumulate, pb_stream_t stream);
/* out[c] (+)= sum_f v[f] * W[f][c]                             (sum over tokens of d_hidden @ W_enc^T = gb_enc @ W_enc^T) */
PB_API int pb_gemv_rows(const float* W, const float* v, float* out, int32_t F, int32_t d, int32_t accumulate, pb_stream_t stream);
/* fired[f] += #{tokens: acts > 0}; *l1_sum += sum |acts|; scalars.pos_count += #{acts > 0}  (train_sae.py:356-365, sae.py:617) */
PB_API int pb_sae_dense_stats(const float* acts, int32_t rows, int32_t F, float* fired, float* l1_sum, void* scalars, pb_stream_t stream);
/* sae_out = norm_out(out_n); scalars.loss_sum += sum (sae_out-x)^2/||x - mean_batch x||; g = dL/d out_n; resid = x - sae_out
 * (sae.py:144-149, 584-595); sae_out / g / resid may be NULL; xsum = column sums of x over the GLOBAL batch of global_rows tokens */
PB_API int pb_sae_dense_loss(const float* x, const float* out_n, const float* mu, const float* sd, const float* xsum, float* sae_out,
                             float* g, float* resid, void* scalars, int32_t rows, int32_t global_rows, int32_t d, int32_t norm_mode,
                             pb_stream_t stream);
/* d_hidden = (d_acts + l1_grad) * [acts > 0] in place on d_acts (+ optional tf32 residual): ReLU backward with d(l1)/d(acts) */
PB_API int pb_sae_dense_dhid(float* d_acts, const float* acts, float* lo, float l1_grad, int64_t n, pb_stream_t stream);
/* scalars: gnorm_sq = ||all four gradients||^2, grad_norm, clip_coef (train_sae.py:394-397), mse, l0 -- then pb_sae_adam */
PB_API int pb_sae_grad_finish(const float* gW_dec, const float* gW_encT, const float* gb_enc, const float* gb_dec, int32_t F, int32_t d,
                              void* scalars, float max_grad_norm, int32_t rows, pb_stream_t stream);
/* E[r][j] = exp(hidden_pre[r][dead_idx[j]]), zero for nd <= j < ldE                                   (sae.py:164)  */
PB_API int pb_sae_ghost_gather(const float* hidden_pre, const int32_t* dead_idx, int32_t nd, int32_t rows, int32_t F, float* E, int32_t ldE,
                               pb_stream_t stream);
/* out[j] = W[idx[j]] (j < n), zero rows up to n_pad;   dst[idx[j]] += scale * src[j] (distinct indices)                */
PB_API int pb_gather_rows(const float* W, const int32_t* idx, int32_t n, int32_t n_pad, int32_t d, float* out, pb_stream_t stream);
PB_API int pb_scatter_add_rows(float* dst, const int32_t* idx, int32_t n, int32_t d, const float* src, float scale, pb_stream_t stream);
PB_API int pb_mul_inplace(float* y, const float* x, int64_t n, pb_stream_t stream);
/* per token row: rescale G0 = exp(h_dead) @ W_dec[dead] to half the residual norm, ghost_sum += sum c*(G-r)^2/rcn with
 * c = mse/((G-r)^2/rcn + 1e-6), and overwrite G0 with dL_ghost/dG0 (sae.py:157-178); rsum = column sums of resid            */
PB_API int pb_sae_ghost_rows(const float* resid, const float* rsum, float* G0, const void* scalars, float* ghost_sum, int32_t rows,
                             int32_t d, pb_stream_t stream);

/* ------------------------------------------------ Gated SAE step pieces (GatedSparseAutoencoder, sae/sae.py:648-792)
 * One encoder GEMM feeds both paths: pi = sae_in @ W_enc + b_gate, and the weight-shared magnitude pre-activation
 * sae_in @ (W_enc * exp(r_mag)) + b_mag equals (pi - b_gate) * exp(r_mag) + b_mag.                                       */
/* acts = [pi > 0] * relu(mag_pre) (:701-709), pi_act = relu(pi) (:769-774), optional tf32 residual planes;
 * fired[f] += #{acts > 0}, piact_colsum[f] += sum_b pi_act, scalars.pos_count += #{acts > 0}                              */
PB_API int pb_gated_fwd(const float* pi, const float* b_gate, const float* r_mag, const float* b_mag, float* acts, float* acts_lo,
                        float* pi_act, float* pi_act_lo, float* fired, float* piact_colsum, void* scalars, int32_t rows, int32_t F,
                        pb_stream_t stream);
/* ga = 2 (via - sae_in) / rows = d aux / d via;  *aux_sum += sum (via - sae_in)^2     (_compute_aux_reconstruction_loss, :783-788) */
PB_API int pb_gated_aux(const float* via, const float* sae_in, float* ga, float* aux_sum, int32_t rows, int32_t d, pb_stream_t stream);
/* in: d_acts = g @ W_dec^T, d_pia = ga @ W_dec^T.  d_acts is overwritten with D = dL/d(sae_in @ W_enc)
 * = [pi>0] (d_pia + l1_grad ||W_dec[f]||) + [pi>0][mag_pre>0] d_acts exp(r_mag); gb_gate, gb_mag, gr_mag, dsum = colsum(D) are zeroed and filled */
PB_API int pb_gated_bwd(float* d_acts, float* D_lo, const float* d_pia, const float* pi, const float* b_gate, const float* r_mag,
                        const float* b_mag, const float* wnorm, float l1_grad, float* gb_gate, float* gb_mag, float* gr_mag, float* dsum,
                        int32_t rows, int32_t F, pb_stream_t stream);
PB_API int pb_row_norms(const float* W, float* out, int32_t F, int32_t d, pb_stream_t stream);      /* out[f] = ||W[f,:]|| */
/* gW_dec[f,:] += l1_grad * piact_colsum[f] * W_dec[f,:] / wnorm[f];  *l1_sum += piact_colsum[f] * wnorm[f]   (_compute_l1_loss, :776-781) */
PB_API int pb_gated_l1_rows(float* gW_dec, const float* W_dec, const float* piact_colsum, const float* wnorm, float l1_grad, float* l1_sum,
                            int32_t F, int32_t d, pb_stream_t stream);
PB_API int pb_sumsq(const float* a, int64_t n, float* acc, pb_stream_t stream);                      /* *acc += sum a^2 */
/* scalars.gnorm_sq (accumulated by pb_sumsq) -> grad_norm, clip_coef (train_sae.py:394-397), mse, l0 */
PB_API int pb_sae_clip_finish(void* scalars, float max_grad_norm, int32_t rows, int32_t d, pb_stream_t stream);
/* torch.optim.Adam on one vector parameter with the step's clip coefficient read from scalars (r_mag, b_mag) */
PB_API int pb_adam_vec(float* p, const float* g, float* m, float* v, int32_t n, const void* scalars, float lr, float beta1, float beta2,
                       float eps, int32_t step, pb_stream_t stream);

/* ------------------------------------------------ data-parallel SAE step over NVLink peer memory
 * New functionality (the reference trains on one device, SURVEY 8e): gradients are reduce-scattered by direct peer loads,
 * the owner of a feature-row slice runs clip + projection + Adam + renorm and stores the new rows into every peer
 * (all-gather).  No NCCL on this path; torch.distributed is used once, to swap the IPC handles.
 * Pointer tables are indexed by rank; entry [rank] is the local buffer, the others come from pb_p2p_open.             */
#define PB_P2P_MAX_RANKS 8
typedef struct {
  int32_t rank, world, d, F, step, global_rows;
  float lr, beta1, beta2, adam_eps, max_grad_norm;
  float* gW_dec[PB_P2P_MAX_RANKS]; float* gW_encT[PB_P2P_MAX_RANKS]; float* gb_enc[PB_P2P_MAX_RANKS]; float* gb_dec[PB_P2P_MAX_RANKS];
  float* fired[PB_P2P_MAX_RANKS]; float* xsum[PB_P2P_MAX_RANKS];
  float* W_dec[PB_P2P_MAX_RANKS]; float* W_encT[PB_P2P_MAX_RANKS]; float* W_encT_lo[PB_P2P_MAX_RANKS]; float* b_enc[PB_P2P_MAX_RANKS];
  float* norm_parts[PB_P2P_MAX_RANKS]; uint32_t* flags[PB_P2P_MAX_RANKS];
  /* local only */
  float *gb_enc_red, *gb_dec_red, *fired_red, *part_accum;     /* [F], [d], [F], [4] */
  float* b_dec; void* scalars;
  float *m_dec, *v_dec, *m_enc, *v_enc, *m_be, *v_be, *m_bd, *v_bd;   /* only the owned row slice is touched */
  float* since_fired; float* act_freq;
  /* NVSwitch multicast views (pb_mc_*; all NULL = peer load / store path): the gradient matrices are then reduce-scattered with
   * multimem.ld_reduce (summed in the switch) and the updated parameter rows all-gathered with multimem.st; the table entries
   * [rank] above are this rank's own (unicast) mappings of the same memory, entries of other ranks are unused.             */
  const float *mc_gW_dec, *mc_gW_encT;
  float *mc_W_dec, *mc_W_encT, *mc_b_enc;
  /* 1: pb_p2p_adam_allgather updates the owned W_dec rows in the local copy only; pb_p2p_push_dec (any stream, followed by its own
   * barrier) sends them to the peers later -- the next step reads W_dec only at its decode                                */
  int32_t defer_dec;
} PbP2PStep;
PB_API int pb_p2p_alloc(int64_t bytes, void** dev_ptr, unsigned char* handle64);   /* cudaMalloc (zeroed) + 64-byte IPC handle */
PB_API int pb_p2p_open(const unsigned char* handle64, void** peer_ptr);
PB_API int pb_p2p_close(void* peer_ptr);
PB_API int pb_p2p_free(void* dev_ptr);
PB_API int pb_p2p_barrier(const PbP2PStep* s, uint32_t epoch, pb_stream_t stream);  /* epoch must increase by 1 per call on every rank */
PB_API int pb_p2p_sum_xsum(const PbP2PStep* s, float* xsum_global, pb_stream_t stream);
PB_API int pb_p2p_reduce_scatter(const PbP2PStep* s, pb_stream_t stream);
PB_API int pb_p2p_adam_allgather(const PbP2PStep* s, pb_stream_t stream);
PB_API int pb_p2p_push_dec(const PbP2PStep* s, pb_stream_t stream);        /* the deferred W_dec half of the all-gather (defer_dec = 1) */
/* NVSwitch multicast memory (csrc/mc.cu).  Collective protocol, driven from the host side (vit_prisma/b200/p2p.py):
 *   every rank pb_mc_supported -> rank 0 pb_mc_create (fd) -> fd to the other ranks (SCM_RIGHTS) -> pb_mc_import ->
 *   every rank pb_mc_add_device -> barrier -> every rank pb_mc_bind_alloc -> barrier.  PB_EUNSUPPORTED = fall back.      */
PB_API int pb_mc_supported(int32_t* supported);
PB_API int pb_mc_round_size(int32_t world, int64_t bytes, int64_t* rounded);
PB_API int pb_mc_create(int32_t world, int64_t bytes, uint64_t* mc_handle, int32_t* fd);
PB_API int pb_mc_import(int32_t fd, uint64_t* mc_handle);
PB_API int pb_mc_add_device(uint64_t mc_handle);
PB_API int pb_mc_bind_alloc(uint64_t mc_handle, int64_t bytes, void** uc_ptr, void** mc_ptr, uint64_t* mem_handle);

#ifdef __cplusplus
}
#endif
#endif /* PRISMA_B200_H */
