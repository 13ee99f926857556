/* m3l_b200 — C-ABI of the B200-native VTMAE hot path.
 *
 * Plain C: pointers, sizes and a CUDA stream handle (void* == cudaStream_t); no torch types.
 * All device pointers must be valid on the current CUDA device.  Every entry point returns 0 on
 * success or a non-zero status (1 invalid argument, 2 CUDA failure, 3 unsupported shape);
 * m3l_last_error() then holds a message for the calling thread.  Nothing here synchronises the
 * stream or allocates device memory, so every call can be captured in a CUDA graph.
 *
 * Each entry point names the reference interface it stands in for.  The reference is pure
 * PyTorch (no FFI of its own: SURVEY.md §2.1), so "replaces" means the eager ops that
 * /root/reference/models/pretrain_models.py dispatches at the cited lines; INTEGRATION.md shows
 * the ctypes binding a maintainer of the reference would add.
 */
#ifndef M3L_B200_H_
#define M3L_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Message of the last failing call on this thread ("" if none). */
const char* m3l_last_error(void);

/* ------------------------------------------------------------------------------------------
 * Dense contraction with fused epilogue (tcgen05 / TMEM / TMA):
 *     out[m, n] = epilogue(alpha * sum_k A[m, k] * B[n, k])
 * Replaces nn.Linear forward / dgrad / wgrad as dispatched by vit_pytorch's Attention and
 * FeedForward (pretrain_models.py:113,784), the patch-embedding Linear (:769-771,776-778) and
 * the to_pixels / to_tactiles heads (:115-116,328,333).
 * ---------------------------------------------------------------------------------------- */
typedef struct m3l_gemm_args {
  const void* a;      /* bf16. K-major: [m, k] row-major (lda). MN-major: [k, m] row-major (lda) */
  const void* b;      /* bf16. K-major: [n, k] row-major (ldb). MN-major: [k, n] row-major (ldb) */
  int32_t lda, ldb;   /* leading dimensions in elements, multiples of 8 */
  int32_t a_mn_major; /* 0: K-major, 1: MN-major (must equal b_mn_major) */
  int32_t b_mn_major;
  int32_t m, n, k;    /* n a multiple of 8 */
  int32_t splits;     /* split-K factor; > 1 requires out_mode 2 */
  int32_t bn;         /* N tile: 0 auto, 64, 128 or 256 */
  void* out;          /* [m, ldo] */
  int32_t ldo;
  int32_t out_mode;   /* 0: bf16 store, 1: fp32 store, 2: fp32 atomic accumulate (red.add) */
  const float* bias;  /* [n] fp32 or NULL */
  const void* residual; /* bf16 [m, ldr] or NULL; added after the activation (may alias out) */
  int32_t ldr;
  int32_t act;        /* 0 none; 1 exact-erf GELU (its derivative GELU'(pre-activation) stored to
                         aux_out if non-NULL); 2 multiply by aux_in[m, n] (backward of 1); 3 ReLU */
  void* aux_out;      /* bf16 [m, ld_aux] or NULL */
  const void* aux_in; /* bf16 [m, ld_aux] or NULL */
  int32_t ld_aux;
  float alpha;        /* must be 1 */
  float* colsum_out;  /* fp32 [n] or NULL: += column sums of the bf16 output (fused bias gradient) */
  void* out2;         /* bf16 [m, ldo] or NULL: a second copy of the output (act 0, residual given) */
  const void* dot_side; /* bf16 [m, ld_dot] or NULL (bf16 output, no residual / act; n % 64 == 0): */
  int32_t ld_dot;       /*   dot_out[row, c] = sum_{j<64} out[row, 64c+j] * dot_side[row, 64c+j]        */
  float* dot_out;       /* fp32 [m, n/64]: with out = dO and dot_side = O this is FlashAttention's delta */
  /* Fused LayerNorm backward (ln_x != NULL; n == 256 = the normalised dimension, bf16 output, no other epilogue
   * option): the product is the gradient w.r.t. LayerNorm(x)'s OUTPUT, dy = A B^T, and the kernel writes
   *     out = dLN(dy; x, stats, gamma) (+ ln_skip)           [m, 256] bf16
   * and accumulates ln_dgamma += sum_rows dy * xhat, ln_dbeta += sum_rows dy, ln_dxcol += sum_rows out (the bias
   * gradient of the Linear whose output gradient `out` is).  dy itself never reaches HBM.  This is the backward of
   * vit_pytorch's pre-norm blocks (`x = attn(norm(x)) + x`, `x = ff(norm(x)) + x`, pretrain_models.py:113,784):
   * the dgrad GEMM through to_qkv / FeedForward's first Linear, nn.LayerNorm's backward and the residual add. */
  const void* ln_x;       /* bf16 [m, 256]: the LayerNorm input */
  const float* ln_stats;  /* fp32 [m, 2]: (mean, rstd) per row, as m3l_layernorm_fwd / m3l_ln_mlp_fwd store them */
  const float* ln_gamma;  /* fp32 [256] */
  const void* ln_skip;    /* bf16 [m, 256] or NULL: gradient arriving through the residual connection */
  float* ln_dgamma;       /* fp32 [256], accumulated */
  float* ln_dbeta;        /* fp32 [256], accumulated */
  float* ln_dxcol;        /* fp32 [256] or NULL, accumulated */
  /* Dropout (drop_key != NULL; training mode of vit_pytorch's FeedForward / Attention.to_out Dropout layers).  The
   * mask Z is m3l_b200's counter-based one (see m3l_dropout_bwd), with row / column of the output, plane 0 and site
   * drop_site; Z is 0 or 65536 / (65536 - thr), thr = floor(drop_p * 65536 + 0.5).  Two epilogues take it:
   *   act 1 (GELU), no residual:   out = Z o GELU(acc + bias), aux_out = Z o GELU'(acc + bias)
   *   act 0 with a residual:       out = residual + Z o (acc + bias) (and out2 the same)
   * Any other combination, drop_p outside [0, 1), and drop_p > 0 with a NULL key return status 1. */
  const int64_t* drop_key;  /* device int64 [1]: the 64-bit Philox key, or NULL */
  int32_t drop_site;        /* (layer << 2) | site */
  float drop_p;
} m3l_gemm_args;

int m3l_gemm_bf16(const m3l_gemm_args* args, void* stream);


/* ------------------------------------------------------------------------------------------
 * Fused pre-norm feed-forward block, forward (dim == 256, hidden a multiple of 128 up to 1024):
 *     out = x + W2 GELU(W1 LayerNorm(x) + b1) + b2
 * One kernel for vit_pytorch's `x = ff(x) + x` (FeedForward.net = LayerNorm, Linear, GELU, Linear;
 * pretrain_models.py:113,784 through vit-pytorch 1.6.4): the [rows, hidden] activation stays in
 * tensor memory.  Optional training outputs (what the backward pass reads): stats (mean, rstd per
 * row), xn_out = LayerNorm(x), h_out = GELU(pre), gp_out = GELU'(pre) (h_out and gp_out together).
 * ---------------------------------------------------------------------------------------- */
typedef struct m3l_ln_mlp_args {
  const void* x;      /* bf16 [rows, dim] */
  int32_t rows, dim, hidden;
  const float* gamma; /* [dim] LayerNorm weight */
  const float* beta;  /* [dim] LayerNorm bias */
  float eps;
  const void* w1;     /* bf16 [hidden, dim] */
  const float* b1;    /* [hidden] */
  const void* w2;     /* bf16 [dim, hidden] */
  const float* b2;    /* [dim] */
  void* out;          /* bf16 [rows, dim]; out == x updates the residual stream in place */
  int32_t out_has_x;  /* non-zero: out (!= x) already holds a copy of x, e.g. written by the producing GEMM
                         (m3l_gemm_args.out2); then, as in the in-place case, the block output is added to out
                         with TMA reduce-adds and x is not fetched a second time */
  float* stats;       /* fp32 [rows, 2] or NULL */
  void* xn_out;       /* bf16 [rows, dim] or NULL */
  void* h_out;        /* bf16 [rows, hidden] or NULL */
  void* gp_out;       /* bf16 [rows, hidden] or NULL */
} m3l_ln_mlp_args;

int m3l_ln_mlp_fwd(const m3l_ln_mlp_args* args, void* stream);

/* ------------------------------------------------------------------------------------------
 * Mask sampling: per sample and per token segment (image, tactile1, tactile2, ...) the ascending
 * argsort of the supplied uniform noise; the first n_masked[s] positions of each segment's
 * permutation are "masked", the rest "unmasked"; lists are concatenated segment by segment.
 * Replaces torch.rand(...).argsort(-1) + slicing + cat, pretrain_models.py:223-248 (the noise is an
 * input so results can be compared bit-exactly with the reference).  Ties resolve stably.
 *   noise            fp32 [batch, n_total]
 *   masked           int64 [batch, sum n_masked]        (global token indices)
 *   unmasked         int64 [batch, n_total - sum n_masked]
 *   slot_of_token    int32 [batch, n_total] or NULL: >= 0 -> position in `unmasked`,
 *                    < 0 -> -(1 + position in `masked`)
 *   unmasked_i32     int32 copy of `unmasked` or NULL
 *   masked_row_of_token  int32 [batch, n_total] or NULL: row of the token in the two stacked
 *                    head-input matrices ([batch*n_masked_first rows of the first group (image) |
 *                    batch*(n_masked - n_masked_first) rows of the rest]), -1 for unmasked tokens
 * ---------------------------------------------------------------------------------------- */
#define M3L_MAX_SEGMENTS 8
typedef struct m3l_mask_segments {
  int32_t count;
  int32_t offset[M3L_MAX_SEGMENTS];   /* first token of the segment */
  int32_t length[M3L_MAX_SEGMENTS];   /* tokens in the segment */
  int32_t n_masked[M3L_MAX_SEGMENTS]; /* how many of them are masked */
} m3l_mask_segments;

int m3l_mask_indices(const float* noise, int batch, int n_total, const m3l_mask_segments* segs,
                     int64_t* masked, int64_t* unmasked, int32_t* slot_of_token,
                     int32_t* unmasked_i32, int32_t* masked_row_of_token, int n_masked_first,
                     void* stream);

/* ------------------------------------------------------------------------------------------
 * Patch sources: up to 4 fp32 NCHW maps of one modality (the image, or tactile1..tactile{nt}),
 * patchified on the fly as einops 'b c (h p1) (w p2) -> b (h w) (p1 p2 c)'
 * (pretrain_models.py:768,775); token_base = global index of the modality's first token.
 * ---------------------------------------------------------------------------------------- */
typedef struct m3l_patch_source {
  const void* src[4]; /* layout 0: fp32 [batch, channels, height, width] maps, one per sensor.
                         layout 1: base pointer of each sensor's first element in the RAW observation tensor */
  int32_t channels, height, width, patch_h, patch_w;
  int32_t token_base;
  /* layout 1 fuses utils/pretrain_utils.py:7-57 (vt_load: NHWC -> NCHW, per-sensor channel de-interleave,
   * (x - lo) / (hi - lo)) and the 5-D frame-stack reshape (models/pretrain_models.py:823-827, ppo_mae.py:236-242)
   * into the patch loads: map element (b, c, y, x) with c = f * chan_group + ch is read from
   *     src[s][b*stride_b + f*stride_f + ch*stride_ch + y*stride_y + x*stride_x]        (strides in elements)
   * and normalised as (raw - norm_lo) / norm_span in fp32; dtype 1 = uint8 frames, raw = value / 255 first.
   * E.g. images [B, F, H, W, 3]: chan_group 3, stride_f H*W*3, stride_ch 1, stride_y W*3, stride_x 3;
   * tactile [B, F, 3*sensors, h, w], sensor s: src[s] = base + 3*s*h*w, chan_group 3, stride_f 3*sensors*h*w,
   * stride_ch h*w, stride_y w, stride_x 1, norm_lo -1, norm_span 2. */
  int32_t layout;     /* 0 or 1 */
  int32_t dtype;      /* layout 1: 0 fp32, 1 uint8 */
  int64_t stride_b;
  int32_t chan_group;
  int32_t stride_f, stride_ch, stride_y, stride_x;
  float norm_lo, norm_span;
} m3l_patch_source;

/* Fused patchify + row gather + LayerNorm(patch_dim) -> bf16 rows [batch*ncols, P]
 * (pretrain_models.py:157,166 + the first LayerNorm of *_patch_to_emb, :769,776).
 * Row (b, jj) reads token tok_idx[b, col0 + jj] (tok_idx NULL: token_base + jj, i.e. all tokens).
 * xhat (optional) receives the normalised values before the affine, for the backward pass. */
int m3l_patch_layernorm(const m3l_patch_source* src, int batch, const int64_t* tok_idx, int idx_ld,
                        int col0, int ncols, const float* gamma, const float* beta, float eps,
                        void* out_bf16, void* xhat_bf16, void* stream);

/* LayerNorm forward over rows (nn.LayerNorm, eps 1e-5): y = LN(x) * gamma + beta
 *   (+ add0[add0_row[r]] + add1[add1_row[r]], fp32 rows: modality / position embeddings,
 *   pretrain_models.py:202-219).  x is bf16, or fp32 if x_fp32.  stats (optional) <- (mean, rstd)
 *   per row.  dst_row (optional): output row remap, negative = row not written. */
int m3l_layernorm_fwd(const void* x, int x_fp32, int rows, int dim, const float* gamma,
                      const float* beta, float eps, void* y_bf16, float* stats,
                      const int32_t* dst_row, const float* add0, const int32_t* add0_row,
                      const float* add1, const int32_t* add1_row, void* stream);

/* LayerNorm backward: dx = dLN(dy) (+ skip), dgamma/dbeta += column sums (block-reduced, then
 * fp32 atomics; grids are sized so each address sees at most a few hundred of them).
 * src_row (optional): dy row gather, negative = zero gradient row.
 * dx_colsum (optional): += column sums of dx, i.e. the bias gradient of the nn.Linear whose output
 * gradient dx is (saves a separate reduction pass over dx). */
int m3l_layernorm_bwd(const void* dy_bf16, const int32_t* src_row, const void* x, int x_fp32,
                      const float* stats, int rows, int dim, const float* gamma,
                      const void* skip_bf16, void* dx, int dx_fp32, float* dgamma, float* dbeta,
                      float* dx_colsum, void* stream);

/* Decoder input assembly (pretrain_models.py:270-307): z[b,t] = (visible ? d[b, slot] : mask_token)
 * + add0[tok_class[t]] + add1[t].  Backward scatters / reduces the gradient accordingly. */
int m3l_decoder_assemble_fwd(const void* d_bf16, int n_visible, const float* mask_token,
                             const int32_t* slot_of_token, int batch, int n_tokens, int dim,
                             const float* add0, const int32_t* tok_class, const float* add1,
                             void* z_bf16, void* stream);
int m3l_decoder_assemble_bwd(const void* dz_bf16, const int32_t* slot_of_token, int batch,
                             int n_tokens, int dim, int n_visible, void* dd_bf16,
                             float* dmask_token, float* dadd0, const int32_t* tok_class,
                             int n_classes, float* dadd1, void* stream);

/* Gradient of the broadcast embedding adds on the encoder side: dclass[slot_class[j]] += sum_b dx[b,j],
 * dpos[row_pos[b,j]] += dx[b,j] (either may be NULL). */
int m3l_rowclass_sum(const void* dx_bf16, int batch, int n_visible, int dim,
                     const int32_t* slot_class, float* dclass, const int32_t* row_pos, float* dpos,
                     void* stream);

/* Masked-patch MSE (pretrain_models.py:327-340): target rows are gathered from the raw maps;
 * *loss_acc += weight * sum((pred - target)^2); dpred = 2 * weight * (pred - target) (bf16);
 * dpred_colsum (optional, patch dim <= 1024): [P] fp32 += column sums of dpred, i.e. the bias
 * gradient of the head Linear (nn.Linear backward through to_pixels / to_tactiles).
 * workspace: device scratch (>= 256 + 4 * blocks bytes; 1 MiB is always enough) whose first 4 bytes
 * are zero on entry and zero again on exit; per-block partial losses are summed by the last block
 * to finish, which makes the loss bit-reproducible run to run. */
int m3l_mse_loss(const m3l_patch_source* src, int batch, const int64_t* tok_idx, int idx_ld, int col0,
                 int ncols, const float* pred, float weight, void* dpred_bf16, float* loss_acc,
                 float* dpred_colsum, void* workspace, size_t workspace_bytes, void* stream);

/* Plain patchify + row gather (no LayerNorm) -> bf16 rows [batch*ncols, ld], (p1, p2, c) order, columns [P, ld)
 * zero-filled: the input of a ViT patch embedding whose first layer is Conv2d(kernel = stride = patch), here the
 * frozen DINOv2 ViT-S/14 image branch of the DINO-tac-MAE variant (/root/reference/train_dino_tac_mae.py:29,
 * models/pretrain_models_dino_cat_mae.py:884-889). */
int m3l_patchify(const m3l_patch_source* src, int batch, const int64_t* tok_idx, int idx_ld, int col0, int ncols,
                 void* out_bf16, int ld, void* stream);

/* dst[b*n_total + tok_idx[b*idx_ld + j]] += src[b*ncols + j] over bf16 rows of `dim` elements (distinct tokens per
 * sample).  Joint MAE + policy-feature step (/root/reference/models/ppo_mae.py:260-263,280): the masked encoder's
 * input is a row gather of the full embedded token sequence the feature extractor also consumes; this adds the
 * gather's gradient into the full-sequence gradient so the patch embedding is back-propagated once. */
int m3l_row_scatter_add(const void* src_bf16, int batch, int ncols, const int32_t* tok_idx, int idx_ld, int n_total,
                        int dim, void* dst_bf16, void* stream);

/* vt_load as a kernel of its own (utils/pretrain_utils.py:7-57): raw observation (layout 1 source) of sensor
 * `sensor` -> fp32 [batch, channels, height, width] contiguous, for callers that need the maps materialised
 * (the EarlyCNN conv stem, reconstruct()); the masked-autoencoder step itself reads raw observations directly. */
int m3l_vt_load(const m3l_patch_source* src, int batch, int sensor, float* out_nchw, void* stream);

/* out[n] += sum_m x[m, n] (bias gradients). */
int m3l_colsum(const void* x_bf16, int rows, int cols, int ld, float* out, void* stream);

/* dgamma[p] += sum_r da[r,p] * xhat[r,p]; dbeta[p] += sum_r da[r,p] (patch LayerNorm parameters). */
int m3l_ln_param_grad(const void* da_bf16, const void* xhat_bf16, int rows, int dim, float* dgamma,
                      float* dbeta, void* stream);

/* ------------------------------------------------------------------------------------------
 * EarlyCNN conv stem (early_conv_masking=True; pretrain_models.py:37-56,180-191).  Convolutions are
 * im2col + m3l_gemm_bf16 (act 3 = ReLU); activations are NHWC bf16, i.e. [batch*H*W, C] matrices.
 *   im2col       col[(b,oy,ox), ci*k*k + ky*k + kx] = x[b, ci, oy*stride-pad+ky, ox*stride-pad+kx] (0 outside);
 *                x is fp32 NCHW (x_nhwc_bf16 = 0: the raw maps) or bf16 NHWC (= 1); the K order is that of
 *                nn.Conv2d.weight.flatten(1), so the weights are used as stored
 *   col2im_relu  dx[b,iy,ix,ci] = [relu_out[b,iy,ix,ci] > 0] * sum over taps of dcol (conv dgrad as a gather,
 *                fused with the ReLU backward of the layer below; relu_out may be NULL)
 *   token_finish out[dst_row[r]] = x[src(b, tok - tok_base)] + add0[tok_class[tok]] + add1[tok], r = b*ncols + jj,
 *                tok = tok_idx ? tok_idx[b*idx_ld + col0 + jj] : tok_base + jj   (modality / position adds +
 *                gather of the visible tokens, pretrain_models.py:202-216,256).  x stacks the modality's
 *                sources (sensors share one CNN) along the batch: src(b, tl) = ((tl/n_per)*batch + b)*n_per + tl%n_per.
 *                Its backward is the gather dtok[src(b,tl)] = slot >= 0 ? dx0[b*rows_per_sample + slot] : 0 with
 *                slot = slot_of_token[b, tok_base+tl] (slot_of_token NULL: slot = tok_base + tl)
 * ---------------------------------------------------------------------------------------- */
int m3l_im2col(const void* x, int x_nhwc_bf16, int batch, int channels, int height, int width, int k, int stride,
               int pad, void* col_bf16, void* stream);
int m3l_col2im_relu(const void* dcol_bf16, int batch, int channels, int height, int width, int k, int stride, int pad,
                    const void* relu_out_bf16, void* dx_bf16, void* stream);
int m3l_token_finish(const void* x_bf16, int batch, int n_per, const int32_t* tok_idx, int idx_ld, int col0, int ncols,
                     int tok_base, const float* add0, const int32_t* tok_class, const float* add1,
                     const int32_t* dst_row, void* out_bf16, int dim, void* stream);
int m3l_token_finish_bwd(const void* dx0_bf16, int batch, int rows_per_sample, int n_total,
                         const int32_t* slot_of_token, int tok_base, int n_mod, int n_per, int dim, void* dtok_bf16,
                         void* stream);

/* Token mean of the rollout feature extractor (MAEExtractor.forward: torch.mean(tokens, dim=1),
 * pretrain_models.py:837) and its backward.  x bf16 [batch, n_tokens, dim] -> out fp32 [batch, dim];
 * dout fp32 [batch, dim] -> dx bf16 [batch, n_tokens, dim] (= dout / n_tokens on every token). */
int m3l_token_mean_fwd(const void* x_bf16, int batch, int n_tokens, int dim, float* out, void* stream);
int m3l_token_mean_bwd(const float* dout, int batch, int n_tokens, int dim, void* dx_bf16, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused multi-head attention, sequence length n <= 256 (longer sequences: m3l_attention_long_* below),
 * dim_head == 64 (tcgen05 / TMEM / TMA).
 * Replaces vit_pytorch Attention's softmax(q k^T * scale) v and its backward
 * (pretrain_models.py:113,784 through vit-pytorch 1.6.4).
 *   qkv   bf16 [batch*n, 3*heads*64]: columns [q | k | v], head h at h*64 inside each third
 *   out   bf16 [batch*n, heads*64]   ('b h n d -> b n (h d)')
 *   lse   fp32 [batch, heads, n]     log-sum-exp of the scaled scores (saved for backward)
 *   dqkv  bf16 [batch*n, 3*heads*64]
 * ---------------------------------------------------------------------------------------- */
int m3l_attention_fwd(const void* qkv_bf16, int batch, int n, int heads, int dim_head, float scale,
                      void* out_bf16, float* lse, void* stream);
/* delta: fp32 [batch*n, heads] = rowsum(dO * O) per head, or NULL (computed in the kernel from out/dout);
 * m3l_gemm_bf16 produces it for free in the epilogue of the GEMM that computes dO (dot_side / dot_out). */
int m3l_attention_bwd(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16,
                      const float* lse, const float* delta, int batch, int n, int heads, int dim_head,
                      float scale, void* dqkv_bf16, void* stream);

/* ------------------------------------------------------------------------------------------
 * The same two operations for any sequence length n >= 1 (dim_head == 64, else status 3), with the
 * same arguments, layouts and LSE: FlashAttention-style kernels over 128-key tiles with an online
 * softmax (attention_long.cu).  m3l_attention_fwd/bwd cover n <= 256; longer sequences go through
 * these.  The backward is two kernels (dK / dV key-tile-stationary, dQ query-tile-stationary),
 * deterministic (no atomics), and allocates nothing.
 * ---------------------------------------------------------------------------------------- */
int m3l_attention_long_fwd(const void* qkv_bf16, int batch, int n, int heads, int dim_head, float scale,
                           void* out_bf16, float* lse, void* stream);
int m3l_attention_long_bwd(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16,
                           const float* lse, const float* delta, int batch, int n, int heads, int dim_head,
                           float scale, void* dqkv_bf16, void* stream);

/* ------------------------------------------------------------------------------------------
 * The same two operations for 32- and 128-wide heads (dim_head 32 or 128, else status 3; 64-wide
 * heads use the entry points above), any n >= 1, with the same arguments, layouts, LSE and
 * deterministic two-kernel backward as m3l_attention_long_*: the other instantiations of the same
 * kernels (attention_long.cuh, attention_dh.cu).  `delta` is optional as above.
 * ---------------------------------------------------------------------------------------- */
int m3l_attention_dh_fwd(const void* qkv_bf16, int batch, int n, int heads, int dim_head, float scale,
                         void* out_bf16, float* lse, void* stream);
int m3l_attention_dh_bwd(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16,
                         const float* lse, const float* delta, int batch, int n, int heads, int dim_head,
                         float scale, void* dqkv_bf16, void* stream);

/* ------------------------------------------------------------------------------------------
 * Dropout (training mode of vit_pytorch's Attention / FeedForward Dropout layers).
 *
 * The mask is a pure function of logical coordinates: Philox4x32-10 (Random123) under the 64-bit key *drop_key
 * (device memory), counter (col >> 3, row, plane, site); the four output words are eight 16-bit uniforms, low half
 * first, and element `col & 7` is kept iff its uniform u >= thr = floor(p * 65536 + 0.5).  Kept elements are
 * multiplied by 65536 / (65536 - thr) (fp32).  site = (layer << 2) | s with s = 0 attention probabilities,
 * 1 attention output (to_out), 2 after the feed-forward GELU, 3 feed-forward output.  Every entry point returns
 * status 1 for p outside [0, 1) or NaN and for a NULL key with p > 0.
 *
 * m3l_attention_dropout_fwd/bwd: m3l_attention_long_fwd/bwd with dropout on the attention probabilities
 * (row = query index, col = key index, plane = sample * heads + head), dim_head 32, 64 or 128 (else status 3), any
 * n.  The forward's lse is that of the undropped scores; out = (P o Z) V.  The backward takes the same optional
 * delta = rowsum(dout * out).  At p = 0 the results equal the kernels without dropout bit for bit.
 *
 * m3l_dropout_bwd: out = Z o dy for a contiguous bf16 [rows, cols] matrix (plane 0), and colsum[c] += sum_r out[r, c]
 * (fp32) when colsum is not NULL.  It is the backward of a dropout applied by m3l_gemm_bf16's dropout epilogues.
 * ---------------------------------------------------------------------------------------- */
int m3l_attention_dropout_fwd(const void* qkv_bf16, int batch, int n, int heads, int dim_head, float scale,
                              const int64_t* drop_key, int drop_site, float drop_p, void* out_bf16, float* lse,
                              void* stream);
int m3l_attention_dropout_bwd(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16,
                              const float* lse, const float* delta, int batch, int n, int heads, int dim_head,
                              float scale, const int64_t* drop_key, int drop_site, float drop_p, void* dqkv_bf16,
                              void* stream);
int m3l_dropout_bwd(const void* dy_bf16, int rows, int cols, const int64_t* drop_key, int drop_site, float drop_p,
                    void* out_bf16, float* colsum, void* stream);

/* ------------------------------------------------------------------------------------------
 * Optimizer over flat fp32 arenas: clip_grad_norm_(params, max_norm) + AdamW.step()
 * (pretrain_models.py:670-676,707-711; torch.optim.AdamW defaults).  `state` is 8 doubles on the
 * device: [0] step counter, [1] sum of squares of all gradients (zero it, then call
 * m3l_grad_sumsq once per live range), [2] total gradient norm, [3] 1 - beta1^step,
 * [4] sqrt(1 - beta2^step) ([2..4] written by step_begin, the bias corrections in double like the
 * Python scalars of torch.optim.AdamW).
 * Sequence per step: sumsq(ranges...) -> step_begin -> clip_adamw(ranges...).  Parameters whose
 * gradient is None in the reference are simply left out of the ranges.
 * hyper_dev (optional): device array of 6 floats [lr, beta1, beta2, eps, weight_decay, max_norm]
 * that overrides the scalar arguments at RUN time, so a captured CUDA graph follows
 * optimizer.param_groups (learning-rate schedules) without being re-captured.
 * ---------------------------------------------------------------------------------------- */
int m3l_grad_sumsq(const float* grads, size_t count, double* state, void* stream);
int m3l_optimizer_step_begin(double* state, float beta1, float beta2, const float* hyper_dev, void* stream);
int m3l_clip_adamw(float* params, float* grads, float* exp_avg, float* exp_avg_sq, size_t count,
                   const double* state, float lr, float beta1, float beta2, float eps,
                   float weight_decay, float max_norm, int write_clipped_grad, const float* hyper_dev,
                   void* stream);

/* bf16 shadow copies of the fp32 master weights consumed by the GEMMs: a flat cast, and transposed
 * copies (dst[c, r] = src[r, c]) of a table of matrices for the dgrad products. */
typedef struct m3l_matrix_desc {
  int64_t src_offset; /* elements from src_base */
  int64_t dst_offset; /* elements from dst_base */
  int32_t rows, cols; /* Momentum (EMA) teacher update over flat fp32 arenas: teacher = teacher * beta + one_minus_beta * student
 * (/root/reference/tactile_ssl/utils/ema.py:6-19, called from models/vtdino.py:159-173 after every train batch).
 * one_minus_beta is passed separately: the reference forms (1.0 - beta) in double precision before it meets the fp32
 * tensor, which is not the fp32 difference 1.0f - beta. */
int m3l_ema_update(float* teacher, const float* student, size_t count, float beta, float one_minus_beta, void* stream);

/* of the source, row-major */
} m3l_matrix_desc;
int m3l_cast_bf16(const float* src, void* dst_bf16, size_t count, void* stream);
int m3l_transpose_cast_bf16(const float* src_base, void* dst_base_bf16, const m3l_matrix_desc* descs_dev,
                            int count, void* stream);

/* LayerScale fold of DINOv2 fine-tuning (csrc/layerscale.cu).  fold: wf = bf16(gamma_r * w[r, c]) [rows, cols],
 * wf_t its transpose [cols, rows] (nullable), bf = gamma o b fp32 (nullable); gamma == NULL casts w unscaled.
 * The rounding is torch's (fp32 product, then round-to-nearest-even bf16).
 * unfold: from the fp32 gradients dwf / dbf of the folded Linear, dw = gamma o dwf, db = gamma o dbf,
 * dgamma[r] = sum_c w[r, c] dwf[r, c] + b[r] dbf[r] (all written, not accumulated). */
int m3l_layerscale_fold(const float* w, const float* b, const float* gamma, int rows, int cols, void* wf_bf16,
                        void* wf_t_bf16, float* bf, void* stream);
int m3l_layerscale_unfold(const float* dwf, const float* dbf, const float* w, const float* b, const float* gamma,
                          int rows, int cols, float* dw, float* db, float* dgamma, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* M3L_B200_H_ */
