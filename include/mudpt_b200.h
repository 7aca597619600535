/* mudpt_b200 -- C ABI of the B200-native MuDPT hot path (libmudpt_b200.so).
 *
 * The reference (YzM1a0/MuDPT) is pure Python/PyTorch and has no FFI of its own; the boundary
 * below is what a maintainer binds (ctypes stub: INTEGRATION.md) to replace, with no other
 * change, the bodies of
 *
 *   VisionTransformer_MuDPT.forward .......... clip/model.py:526-553
 *   Transformer / ResidualAttentionBlock_MuDPT  clip/model.py:254-301, 404-440
 *   TextEncoder.forward ...................... trainers/mudpt.py:142-156
 *   CustomCLIP.forward (normalise + logits) .. trainers/mudpt.py:170-184
 *   F.cross_entropy + loss.backward() ........ trainers/mudpt.py:249-251 (dgrad only: every
 *                                              CLIP weight is frozen, :205-212)
 *   d loss / d image ......................... the same backward continued through the stem to the
 *                                              pixels (mudpt_vision_backward_images)
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; fp32 unless noted;
 *   - the caller (PyTorch) owns every tensor it passes in or receives; the handle owns its
 *     converted frozen weights and its activation workspace;
 *   - calls are asynchronous on the `stream` argument (a cudaStream_t passed as void*), never
 *     synchronise the device, and are CUDA-graph capturable after the first (allocating) call;
 *   - return value 0 = ok, negative = error; mudpt_last_error() gives the message;
 *   - one handle per process/GPU; a handle is not thread-safe;
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 *
 * Row layout of token matrices: row = sequence * L + token ("NLD"); the reference's LND is a
 * permutation of the same data.
 */
#ifndef MUDPT_B200_H
#define MUDPT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MUDPT_ABI_VERSION 1

typedef struct mudpt_handle mudpt_handle;

/* Architecture + prompt geometry. Mirrors the CLIP(...) constructor arguments
 * (clip/model.py:667-681) and cfg.TRAINER.MUDPT.{N_CTX, DEEP_PROMPT_DEPTH} (train.py:114-119). */
typedef struct mudpt_config {
  int32_t embed_dim;
  int32_t image_resolution;
  int32_t vision_layers;
  int32_t vision_width;
  int32_t vision_patch_size;
  int32_t context_length;
  int32_t transformer_width;
  int32_t transformer_heads;
  int32_t transformer_layers;
  int32_t n_ctx;        /* prompt tokens per tower */
  int32_t prompt_depth; /* DEEP_PROMPT_DEPTH: layers 0..depth-1 see a fresh prompt */
  int32_t device;       /* CUDA device ordinal */
} mudpt_config;

enum { MUDPT_TOWER_VISION = 0, MUDPT_TOWER_TEXT = 1 };

int mudpt_abi_version(void);
/* message of the last failing call on this thread that had no handle (create, unit kernels) */
const char* mudpt_global_last_error(void);

int mudpt_create(const mudpt_config* cfg, mudpt_handle** out);
void mudpt_destroy(mudpt_handle* h);
/* Options (name, integer value):
 *   "ln_fused"  -1 (default) by tower size: LayerNorm folded into the forward GEMM epilogues for towers of >= 32768
 *               token rows, stand-alone LN kernels below (measured A/B); 1 always, 0 never (env MUDPT_LN_FUSED = 1 / 0).
 *               0 is also the setting for checkpoints whose residual rows have |mean| >> std: the fused form feeds
 *               bf16(x), not bf16(LN(x)), to the tensor cores
 *   "ln_bwd_fused" 0 (default; env MUDPT_LN_BWD_FUSED) 1 = LayerNorm dgrad in the dgrad GEMMs' epilogues (needs
 *               ln_fused; measured slower than the stand-alone kernel at the cfg-2 shapes, kept for narrow towers)
 *   "prune"     1 (default; env MUDPT_PRUNE) exact work skipping: the last block's out-proj / MLP (forward and
 *               dgrad) run on the CLS / EOT rows only (clip/model.py:548, trainers/mudpt.py:154), 0 = every row
 *   "grad_stream_bf16"  1 (default; env MUDPT_GRAD_BF16) the gradient of the residual stream travels between the
 *               LayerNorm backward kernels as bf16 -- the copy the dgrad GEMMs read as their A operand anyway; fp32 rows
 *               are kept for the deep-prompt window (what the splice backward sums); 0 = fp32 stream + bf16 copy.
 *               Ignored (fp32) when the dense input gradient d_x0 is requested or with ln_bwd_fused. */
int mudpt_set_option(mudpt_handle* h, const char* name, int32_t value);
const char* mudpt_last_error(mudpt_handle* h);

/* Frozen CLIP weights, one call per tensor, `name` = key of the reference CLIP.state_dict()
 * ("visual.conv1.weight", "visual.transformer.resblocks.3.attn.in_proj_weight",
 * "transformer.resblocks.0.mlp.c_fc.bias", "positional_embedding", "ln_final.weight",
 * "text_projection", "logit_scale", ...; clip/model.py:499-524, 667-779).  The data is converted
 * once (bf16, plus a transposed bf16 copy for the dgrad GEMMs) into handle-owned memory.
 * Returns 1 for names the hot path does not use (token_embedding.weight, prompt parameters). */
int mudpt_set_weight(mudpt_handle* h, const char* name, const float* data, int64_t numel, void* stream);
/* 0 when every weight the two towers need has been set. */
int mudpt_weights_complete(mudpt_handle* h);

/* ---- vision tower: VisionTransformer_MuDPT.forward (clip/model.py:526-553) -------------------
 * images   [B, 3, R, R]
 * prompts  [depth, n_ctx, vision_width]: prompts[0] = ln_pre(visual_ctx + shared_ctx) (the layer-0
 *          prompt rows after :541), prompts[i>=1] = t2v_visual_prompts[i-1] + visual_ctx_deep_prompts[i-1]
 * f_img    [B, embed_dim] = ln_post(x[:, 0]) @ proj */
int mudpt_vision_forward(mudpt_handle* h, const float* images, int32_t B, const float* prompts, float* f_img, void* stream);
/* d_f_img [B, embed_dim] -> d_prompts [depth, n_ctx, vision_width] (summed over the batch).
 * Must follow mudpt_vision_forward on the same handle (uses its saved activations). */
int mudpt_vision_backward(mudpt_handle* h, const float* d_f_img, float* d_prompts, void* stream);
/* Image gradients (adversarial evaluation / training, saliency): d_f_img [B, embed_dim] ->
 *   d_images  [B, 3, R, R], required: the gradient w.r.t. the images passed to the last mudpt_vision_forward (the
 *             tensor as given, i.e. after the caller's pixel normalisation);
 *   d_prompts [depth, n_ctx, vision_width] as mudpt_vision_backward, or NULL (not computed).
 * The tower backward runs densely down to its input (no work skipping below block 0, fp32 gradient stream), then the stem
 * backward: the patch rows before ln_pre are recomputed from the kept patches, ln_pre's dgrad, the patch dgrad GEMM against
 * conv1.weight and the inverse im2col.  With the options prune = 0 and grad_stream_bf16 = 0, d_prompts equals that of
 * mudpt_vision_backward bit for bit.  Must follow mudpt_vision_forward (not mudpt_vision_infer) with no mudpt_set_option
 * in between; may be repeated.  The first call may allocate (reported under mudpt_workspace_bytes kind 0; nothing for
 * callers that never ask for image gradients); CUDA-graph capturable after it.  For sequences over 128 tokens the
 * attention backward takes rowsum(dO O) from the bf16 O (DESIGN.md section 9): image gradients share that error with
 * the prompt gradients on rows dominated by an attention sink. */
int mudpt_vision_backward_images(mudpt_handle* h, const float* d_f_img, float* d_prompts, float* d_images, void* stream);
/* One l-inf PGD step (adversarial evaluation / training) on the images of the last mudpt_vision_forward, which were
 * x_norm = (x_adv - mean) / std.  d_f_img [B, embed_dim] -> the image gradient g = dL/dx_norm as in
 * mudpt_vision_backward_images (no prompt gradient), never written as an image, then per element, channel c:
 *   s      = sign(g / std[c])                                  (0 for a zero quotient)
 *   x'     = min(max(x_adv + alpha * s, x_clean - eps), x_clean + eps)
 *   x'     = min(max(x', 0), 1)
 *   x_adv  <- x'                                               (in place)
 *   x_norm <- (x' - mean[c]) / std[c]
 * x_adv, x_clean, x_norm [B, 3, R, R] (pixel space for the first two), 8-byte aligned.  Every operation is IEEE fp32
 * without flushing subnormals: bitwise the PyTorch loop x = (x + alpha * (g / std).sign()).clamp(x_clean - eps,
 * x_clean + eps).clamp(0, 1), whose g / std is the autograd of the normalisation.  x_norm may be the tensor the forward
 * read.  eps finite >= 0, alpha finite > 0, std finite > 0.  Memory and CUDA-graph capture as
 * mudpt_vision_backward_images; must follow mudpt_vision_forward; may be repeated (each call reads the same forward). */
int mudpt_vision_pgd_step(mudpt_handle* h, const float* d_f_img, float* x_adv, const float* x_clean, float* x_norm,
                          const float* mean_host, const float* std_host, float eps, float alpha, void* stream);

/* ---- text tower: TextEncoder.forward (trainers/mudpt.py:142-156) -------------------------------
 * Class set-up (once per class list): embeddings [C, src_len, width] are the token embeddings of the
 * tokenised class prompts (prefix | placeholder ctx rows | suffix, trainers/mudpt.py:83-90),
 * eot_host[C] = argmax of the token ids (:154).  seq_len <= src_len: tokens at positions >= seq_len
 * are dropped; with seq_len = max(eot)+1 this is exact under the causal mask (SURVEY.md 8c-i). */
int mudpt_text_set_classes(mudpt_handle* h, const float* embeddings, int32_t C, int32_t src_len, int32_t seq_len,
                           const int32_t* eot_host, void* stream);
/* The same class set-up with every class at its own length (ragged tower): class c keeps its first len_host[c] tokens,
 * 1 + n_ctx <= len_host[c] <= min(src_len, 128) and eot_host[c] < len_host[c]; len_c = max(eot_c + 1, 1 + n_ctx) is exact
 * under the causal mask.  The classes are packed (class c on rows [off_c, off_c + len_c), off_c = sum of the lengths before
 * it), so no row runs past its class's EOT.  A ragged tower always uses the stand-alone LayerNorm kernels (option
 * "ln_fused" does not apply) and the warp-MMA attention kernels.  The next mudpt_text_set_classes call makes the tower
 * padded again. */
int mudpt_text_set_classes_ragged(mudpt_handle* h, const float* embeddings, int32_t C, int32_t src_len, const int32_t* len_host,
                                  const int32_t* eot_host, void* stream);
/* prompts [depth, n_ctx, width]: prompts[0] = ctx + positional_embedding[1:1+n_ctx],
 *         prompts[i>=1] = deep_prompts[i-1] + v2t_text_prompts[i-1] (trainers/mudpt.py:175)
 * splice_layer0 = 0 keeps rows 1..n_ctx of the embeddings as given (per-class ctx, dense API).
 * f_txt [C, embed_dim] */
int mudpt_text_forward(mudpt_handle* h, const float* prompts, int32_t splice_layer0, float* f_txt, void* stream);
/* d_f_txt [C, embed_dim] -> d_prompts [depth, n_ctx, width]; d_x0 (optional, may be NULL)
 * [C, seq_len, width] = gradient of the tower input (dense module-level API).  Ragged tower: d_x0 is
 * [C, max(len_host), width] with zeros at positions >= len_c (exact: those tokens do not reach any output). */
int mudpt_text_backward(mudpt_handle* h, const float* d_f_txt, float* d_prompts, float* d_x0, void* stream);

/* ---- forward-only towers (evaluation, frozen towers) ---------------------------------------------
 * The same arguments and results as mudpt_vision_forward / mudpt_text_forward (the text tower runs over the registered
 * class set), for a result nothing will differentiate:
 *   - f_img / f_txt are bitwise equal to those of the training forward on the same inputs (same kernel sequence; the
 *     c_fc GEMMs write QuickGELU(h) only instead of h and QuickGELU(h));
 *   - the walk runs in an inference workspace of its own (a few buffers every layer shares, about 26 * width bytes per
 *     token row, DESIGN.md section 3), allocated at the first call; nothing a pending mudpt_*_backward reads is touched,
 *     so a training forward, an infer call (any batch size, any prompts) and the backward give the gradients of the
 *     forward alone;
 *   - stream ordering as for the other tower calls: the training and the inference workspaces are disjoint, so a
 *     training walk and an infer call may also run on two streams at once;
 *   - CUDA-graph capturable after the first (allocating) call with the largest shape. */
int mudpt_vision_infer(mudpt_handle* h, const float* images, int32_t B, const float* prompts, float* f_img, void* stream);
int mudpt_text_infer(mudpt_handle* h, const float* prompts, int32_t splice_layer0, float* f_txt, void* stream);
/* Device bytes the handle holds for `tower` (MUDPT_TOWER_*): kind 0 = training workspace (allocated at the first
 * mudpt_*_forward; vision: plus what the first mudpt_vision_backward_images adds), 1 = inference workspace (first
 * mudpt_*_infer), 2 = tower input (class set / vision stem output).
 * Requested sizes: each allocation carries 256 B of slack besides. */
int mudpt_workspace_bytes(mudpt_handle* h, int32_t tower, int32_t kind, int64_t* bytes);

/* ---- logits + loss head (trainers/mudpt.py:178-182, :250) ---------------------------------------
 * labels int64 [B] or NULL (logits only).  loss (1 float) = sum_b CE_b * inv_global_batch,
 * d_f_img [B,e] / d_f_txt [C,e] = gradients of that loss (NULL to skip). */
int mudpt_logits_head(mudpt_handle* h, const float* f_img, const float* f_txt, const int64_t* labels, int32_t B,
                      int32_t C, float inv_global_batch, float* logits, float* loss, float* d_f_img, float* d_f_txt,
                      void* stream);
/* backward of the logits for an external loss: dlogits [B, C] -> d_f_img, d_f_txt */
int mudpt_logits_backward(mudpt_handle* h, const float* f_img, const float* f_txt, const float* dlogits, int32_t B,
                          int32_t C, float* d_f_img, float* d_f_txt, void* stream);

/* ---- unit-testable pieces (no handle) -----------------------------------------------------------
 * bf16 buffers are passed as uint16_t*. */
int mudpt_layernorm_forward(const float* x, const float* gamma, const float* beta, void* out, int32_t out_bf16,
                            int32_t rows, int32_t width, void* stream);                     /* clip/model.py:164-170 */
int mudpt_layernorm_backward(const float* dy, const float* x, const float* gamma, const float* resid, float* dx,
                             uint16_t* dx_bf16, int32_t rows, int32_t width, void* stream);
/* The form the towers use when the gradient of the residual stream is kept in bf16 (option "grad_stream_bf16"):
 * dy bf16; x = fp32 rows (x_stats NULL) or their bf16 copy + per-64-column partial statistics (mudpt_rowstats);
 * resid = fp32 rows, or (resid_bf16 != 0) bf16 rows that may alias dx_bf16, or NULL; dx (fp32) / dx_bf16 may each be
 * NULL (not both); win_n >= 0: fp32 rows are written only where (row % win_L) is in [win_row0, win_row0 + win_n).
 * Every pointer must be 16-byte aligned (rows are moved with 16-byte vector accesses / bulk copies). */
int mudpt_layernorm_backward_stream(const uint16_t* dy, const void* x, const float* x_stats, const float* gamma,
                                    const void* resid, int32_t resid_bf16, float* dx, uint16_t* dx_bf16, int32_t rows,
                                    int32_t width, int32_t win_L, int32_t win_row0, int32_t win_n, void* stream);
int mudpt_splice_forward(float* x, const float* prompt, int32_t S, int32_t L, int32_t row0, int32_t n, int32_t width,
                         void* stream);                                                       /* clip/model.py:281-297 */
int mudpt_splice_backward(float* dx, uint16_t* dx_bf16, float* d_prompt, int32_t S, int32_t L, int32_t row0, int32_t n,
                          int32_t width, int32_t zero_rows, void* stream);
/* qkv [S*L, 3*width] bf16 -> o [S*L, width] bf16, lse2 [S, H, L] (log2 domain) */
int mudpt_attention_forward(const uint16_t* qkv, uint16_t* o, float* lse2, int32_t S, int32_t L, int32_t H,
                            int32_t causal, void* stream);                                    /* clip/model.py:271-273 */
int mudpt_attention_backward(const uint16_t* qkv, const uint16_t* o, const uint16_t* d_o, const float* lse2,
                             float* dsum_scratch, uint16_t* dqkv, int32_t S, int32_t L, int32_t H, int32_t causal,
                             void* stream);
/* Causal attention over packed variable-length sequences: sequence s occupies rows [seq_off[s], seq_off[s+1]) of
 * qkv [M, 3*width] / o / d_o [M, width] / dqkv (seq_off: device int32 [S+1], lengths 1..128, max_len = the longest);
 * lse2 [M * H] holds sequence s's [H, len_s] block at seq_off[s] * H. */
int mudpt_attention_varlen_forward(const uint16_t* qkv, uint16_t* o, float* lse2, const int32_t* seq_off, int32_t S,
                                   int32_t max_len, int32_t H, void* stream);
int mudpt_attention_varlen_backward(const uint16_t* qkv, const uint16_t* d_o, const float* lse2, uint16_t* dqkv,
                                    const int32_t* seq_off, int32_t S, int32_t max_len, int32_t H, void* stream);
/* C = A[M,K] x B[N,K]^T (bf16, fp32 accumulate on tcgen05) with epilogue `mode`:
 * 0 bf16 = acc+bias | 1 f32 = acc+bias | 2 f32 = acc+bias+resid | 3 out0 = h, out1 = QuickGELU(h)
 * 4 bf16 = acc * QuickGELU'(aux) | 5 patch-embedding scatter (+pos) */
int mudpt_gemm_bf16(const uint16_t* A, const uint16_t* B, int32_t M, int32_t N, int32_t K, int32_t mode, void* out0,
                    void* out1, const float* bias, const float* resid, const void* aux, int32_t ldc, int32_t patch_np,
                    int32_t patch_L, void* stream);
/* The same GEMM with every epilogue the towers use, incl. the LayerNorm-fused forms (clip/model.py:164-170 folded
 * into :273 / :299-300 and their dgrads).  Modes 0-5 as above, plus
 *   7  bf16 = rstd*(acc - mean*colsum) + bias            LN1 + in-proj   (A = bf16 LN input, B = gamma-folded weight)
 *   8  out0 = h = (same), out1 = QuickGELU(h)            LN2 + c_fc
 *   9  f32 = acc + bias + resid; out2 = bf16 copy; stats_out[row, col/64] = (sum, M2) of the new row; rows
 *      (r % splice_L) in [splice_row0, splice_row0 + splice_n) take splice_prompt (deep-prompt splice, :281-297)
 *   10 f32 = resid + rstd*(acc - c1 - xhat*c2) (+ bf16 copy): LayerNorm dgrad in the dgrad GEMM's epilogue,
 *      c1 = sum_p dots[row,p].x / ln_width, c2 = sum_p dots[row,p].y / ln_width, xhat from x2 and ln_stats
 *   11 mode 4 + dots_out[row, col/span] = (sum dh*colsum, sum dh*(h - bias')) with sb = interleaved (colsum, bias')
 *   12 out0 = QuickGELU(acc + bias): out1 of mode 3 alone (bitwise), one output stream   c_fc of a forward-only walk
 *   13 out0 = QuickGELU(rstd*(acc - mean*colsum) + bias): out1 of mode 8 alone (bitwise)
 * stream_k: 0 = whole tiles only, 1 = cut the tail wave into k-block ranges whenever possible, -1 = cost model. */
typedef struct mudpt_gemm_epilogue {
  int32_t mode, ldc;
  void* out0;
  void* out1;
  void* out2;
  const float* bias;
  const float* resid;
  const void* aux;
  const float* ln_stats;   /* [M, ln_parts, 2] */
  int32_t ln_parts, ln_width;
  float ln_eps;
  int32_t dot_parts;
  const float* colsum;
  float* stats_out;        /* [M, N/64, 2] */
  const float* splice_prompt;
  int32_t splice_row0, splice_n, splice_L, stream_k;
  const void* x2;          /* bf16 [M, ldc] */
  const float* dots;       /* [M, dot_parts, 2] */
  const float* sb;         /* [N, 2] */
  float* dots_out;         /* [M, N/mudpt_gemm_dots_span(N), 2] */
} mudpt_gemm_epilogue;
int mudpt_gemm_fused(const uint16_t* A, const uint16_t* B, int32_t M, int32_t N, int32_t K, const mudpt_gemm_epilogue* ep,
                     void* stream);
int32_t mudpt_gemm_dots_span(int32_t N);
/* xb = bf16(x), stats[row, p] = (sum, M2 about the partial mean) of columns [64p, 64p+64): the form in which the
 * fused-LayerNorm GEMMs take their LN input */
int mudpt_rowstats(const float* x, uint16_t* xb, float* stats, int32_t rows, int32_t width, void* stream);
/* W [N, K], gamma/beta [K], bias [N] -> W' = bf16(W gamma) [N, K] and its transpose [K, N], bias' = bias + W beta,
 * colsum[n] = sum_k W'[n,k], sb = interleaved (colsum, bias') */
int mudpt_fold_layernorm(const float* W, const float* gamma, const float* beta, const float* bias, uint16_t* Wl,
                         uint16_t* Wlt, float* bias_l, float* colsum, float* sb, int32_t N, int32_t K, void* stream);
/* attention backward that also emits the row dots of dqkv for the fused LayerNorm backward of the in-proj:
 * ln_sb [3*width, 2] = (colsum, bias'), ln_dots [S*L, 3*H, 2] */
int mudpt_attention_backward_dots(const uint16_t* qkv, const uint16_t* o, const uint16_t* d_o, const float* lse2,
                                  float* dsum_scratch, uint16_t* dqkv, int32_t S, int32_t L, int32_t H, int32_t causal,
                                  const float* ln_sb, float* ln_dots, void* stream);
/* which sequences take the tcgen05 / TMEM attention kernels: 0 = none (warp-MMA kernels), 1 = default (non-causal,
 * 129..256 tokens: the vision tower), 2 = every sequence of up to 256 tokens.  Process-wide (tests, A/B runs). */
int mudpt_set_attention_tc(int32_t mode);
int mudpt_im2col(const float* images, uint16_t* patches, int32_t B, int32_t R, int32_t patch, int32_t ld, void* stream);
/* inverse index map of mudpt_im2col, fp32: patches [B * (R/patch)^2, ld] -> images [B, 3, R, R]; every image element is
 * written exactly once (stride = kernel size: a permutation), columns >= 3 * patch^2 are not read */
int mudpt_col2im(const float* patches, float* images, int32_t B, int32_t R, int32_t patch, int32_t ld, void* stream);
/* the update of mudpt_vision_pgd_step alone: dpatch [B * (R/patch)^2, ld] in mudpt_col2im's layout (columns >= 3 * patch^2
 * not read) is g = dL/dx_norm; x_adv updated in place, x_norm written, both [B, 3, R, R] */
int mudpt_pgd_linf_update(const float* dpatch, int32_t ld, float* x_adv, const float* x_clean, float* x_norm, int32_t B,
                          int32_t R, int32_t patch, const float* mean_host, const float* std_host, float eps, float alpha,
                          void* stream);
int mudpt_cast_bf16(const float* in, uint16_t* out, int64_t numel, void* stream);

/* ---- own collectives over NVLink peer memory for the head's exchange (replaces the all_gather / reduce_scatter that
 * nn.DataParallel's gather / scatter of trainers/mudpt.py:230-233 become under class sharding).  peers_dev: DEVICE array of
 * `world` base pointers, one per rank of the node, to fp32 row matrices of `width` columns in memory every GPU maps
 * (symmetric allocation); row shards as in mudpt_b200/dist.py:shard_bounds.  The caller orders each call after a barrier
 * that makes the peers' writes visible, and before the next overwrite of the buffers.
 *   all_gather:      peers[r] = rank r's shard [rows(r), width];  out [n_total, width]
 *   reduce_scatter:  peers[r] = rank r's full matrix [n_total, width];  out [rows(rank), width] = sum over r, fixed order */
int mudpt_peer_all_gather_rows(const void* peers_dev, int32_t world, int32_t n_total, int32_t width, float* out, void* stream);
int mudpt_peer_reduce_scatter_rows(const void* peers_dev, int32_t world, int32_t rank, int32_t n_total, int32_t width, float* out,
                                   void* stream);

/* ---- trainable prompt algebra of MuDPT (trainers/mudpt.py:117-130, 143, 175; clip/model.py:534-541) --------------
 * The three trainable Linear layers, ln_pre on the shallow vision prompt and the stacking that turn the 10 trainable
 * tensors into the two prompt stacks the towers splice, and the backward into those tensors: 2 + 2 launches.
 * All pointers fp32, contiguous; n = n_ctx, depth = DEEP_PROMPT_DEPTH, dt / dv = text / vision width.
 *   forward : reads ctx [n,dt], deep [depth-1,n,dt], We [dv,dt], be [dv], Wd [dv,dt], bd [dv], vctx [n,dv],
 *             vdeep [depth-1,n,dv], Wv [dt,dv], bv [dt], ln_g / ln_b [dv] (ln_pre), pos [n,dt];
 *             writes P_v [depth,n,dv], P_t [depth,n,dt], ln_in [n,dv] (saved for the backward)
 *   backward: reads the above + dP_v, dP_t; u [n,dv] is scratch; writes the d_* gradients of the 10 tensors */
typedef struct mudpt_prompt_args {
  int32_t n, depth, dt, dv;
  float eps;
  const float *ctx, *deep, *We, *be, *Wd, *bd, *vctx, *vdeep, *Wv, *bv;
  const float *ln_g, *ln_b, *pos;
  float *P_v, *P_t, *ln_in;
  const float *dP_v, *dP_t;
  float* u;
  float *d_ctx, *d_deep, *d_We, *d_be, *d_Wd, *d_bd, *d_vctx, *d_vdeep, *d_Wv, *d_bv;
} mudpt_prompt_args;
int mudpt_prompt_forward(const mudpt_prompt_args* args, void* stream);
int mudpt_prompt_backward(const mudpt_prompt_args* args, void* stream);

/* ---- fused SGD step over the (small) trainable tensors -----------------------------------------
 * One launch for all tensors, torch.optim.SGD semantics (what Dassl's build_optimizer creates for
 * the yaml's OPTIM.NAME = "sgd", configs/trainers/MuDPT/*.yaml:15-22; called from
 * model_backward_and_update, trainers/mudpt.py:251):
 *   d = g + weight_decay * p;  buf = first_step ? d : momentum * buf + (1 - dampening) * d;
 *   d = nesterov ? d + momentum * buf : buf;  p -= lr * d          (momentum == 0: p -= lr * d, buf unused)
 * params / grads / bufs: host arrays of n device pointers (fp32, contiguous), numel: host array. n <= 32. */
int mudpt_sgd_step(void* const* params, const void* const* grads, void* const* bufs, const int64_t* numel, int32_t n,
                   float lr, float momentum, float dampening, float weight_decay, int32_t nesterov, int32_t first_step,
                   void* stream);

/* ---- input pipeline in front of the vision tower (SURVEY.md 8f N2) -------------------------------
 * Replaces, for the tensor MuDPT.parse_batch_train receives (trainers/mudpt.py:263-268), the CPU transform
 * the yaml names (configs/trainers/MuDPT/vit_b16_bz4_ep10_nctx2_depth9.yaml:8-13: random_resized_crop,
 * random_flip, normalize, bicubic) -- Dassl's builder maps it onto torchvision transforms on PIL images:
 * crop -> PIL.Image.resize(BICUBIC) -> window (CenterCrop at evaluation) -> hflip -> /255 -> (x - mean) / std.
 * Output is bit-identical to that pipeline.  Random parameters are drawn by the caller. */
typedef struct mudpt_image_desc {
  const uint8_t* src;                  /* DEVICE pointer: 8-bit RGB, HWC, rows `pitch` bytes apart */
  int32_t height, width, pitch;
  int32_t box_x, box_y, box_w, box_h;  /* crop box (PIL.Image.crop); resampling clamps at its edges */
  int32_t rs_w, rs_h;                  /* size the crop is resampled to (PIL.Image.resize) */
  int32_t win_x, win_y;                /* top-left of the out_h x out_w window of the resampled image */
  int32_t flip;                        /* != 0: mirror the window horizontally */
  int32_t reserved[2];
} mudpt_image_desc;                    /* 64 bytes */
/* device workspace (bytes) mudpt_augment_images needs for this batch; negative on a bad descriptor */
int64_t mudpt_augment_workspace_bytes(const mudpt_image_desc* descs_host, int32_t n, int32_t out_h, int32_t out_w);
/* descs: DEVICE copy of descs_host[n]; mean_host / std_host: 3 floats; out: fp32 [n, 3, out_h, out_w] */
int mudpt_augment_images(const mudpt_image_desc* descs, const mudpt_image_desc* descs_host, int32_t n, int32_t out_h,
                         int32_t out_w, const float* mean_host, const float* std_host, void* workspace,
                         int64_t workspace_bytes, float* out, void* stream);

/* ---- introspection for tests / profiling --------------------------------------------------------
 * name in {"x_in","x_mid","qkv","o","h","lse","dx"}; layer ignored for "dx". */
int mudpt_debug_buffer(mudpt_handle* h, int32_t tower, const char* name, int32_t layer, void** ptr, int64_t* numel);
/* Per-kernel-class timing with CUDA events on the launch stream (bench.py's roofline leg).  Between
 * begin and end every tower launch is bracketed by an event pair.  end() blocks until the recorded
 * work has finished and fills out_host[cat*4 + {0,1,2,3}] = {total ms, launches, algorithmic FLOPs,
 * algorithmic bytes} for cat = gemm (other), attn_fwd, attn_bwd, ln_fwd, ln_bwd, splice, head, stem, then the eight
 * GEMMs of a block: gemm_qkv, gemm_out, gemm_fc, gemm_proj, gemm_dproj, gemm_dfc, gemm_dout, gemm_dqkv (16 x 4 doubles). */
int mudpt_profile_begin(mudpt_handle* h);
int mudpt_profile_end(mudpt_handle* h, double* out_host, int32_t n_out);
/* The same with a fifth value per class: sum over its launches of max(FLOPs / peak_tflops, bytes / hbm_gbs) in ms -- the
 * time the class would take if every launch ran at the bound that applies to it (n_out >= 5 * classes). */
int mudpt_profile_end_bound(mudpt_handle* h, double* out_host, int32_t n_out, double peak_tflops, double hbm_gbs);
/* number of kernel launches issued by the library on this handle since creation */
int64_t mudpt_launch_count(mudpt_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* MUDPT_B200_H */
