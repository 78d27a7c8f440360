/*
 * d2s.h -- C ABI of libd2s_b200.so: the B200 (sm_100a) token-sparsification hot path of
 * Dense2Sparse-ViT / DynamicViT.
 *
 * The reference (marc345/Dense2Sparse-ViT) has no FFI or operator registry: its boundary is the Python
 * surface of vit_models/{dynamic_vit,default_dynamic_vit,peturbed_topk}.py (SURVEY.md section 8b).  This
 * header is the boundary introduced underneath it; each entry point names the reference call site it
 * replaces (file:line under the reference tree).  INTEGRATION.md shows the ctypes stub a maintainer
 * would add on the reference side.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller; nothing is allocated, no host sync is
 *     performed, no stream is created.  Work is enqueued on `stream` (a cudaStream_t passed as void*).
 *   - tensors are dense row-major ("contiguous"); shapes are given in the comments.
 *   - indices are int64 (torch.long), matching the reference.
 *   - return value 0 = ok; non-zero = error, message via d2s_last_error() (thread-local).  Shape and
 *     alignment errors are reported before any launch.  There is no CPU fallback and no other arch.
 */
#ifndef D2S_H
#define D2S_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* d2s_stream_t; /* cudaStream_t */

enum { D2S_F32 = 0, D2S_BF16 = 1 };
enum { D2S_ORDER_INDEX_ASC = 0, D2S_ORDER_SCORE_DESC = 1 };
enum { D2S_PROB_SOFTMAX = 0, D2S_PROB_SIGMOID = 1 };
enum { D2S_ACT_NONE = 0, D2S_ACT_GELU = 1, D2S_ACT_RELU = 2 };

enum {
  D2S_OK = 0,
  D2S_ERR_ARG = 1,      /* bad shape / null pointer / unsupported size */
  D2S_ERR_ALIGN = 2,    /* pointer or row pitch not 16-byte aligned   */
  D2S_ERR_CUDA = 3,     /* launch failed (message holds cudaGetErrorString) */
  D2S_ERR_ARCH = 4      /* device is not sm_100 */
};

const char* d2s_last_error(void);
int d2s_version(void);
/* number of kernels this library has launched in the calling process (for bench.py's gpu_launches) */
uint64_t d2s_launch_count(void);

/* ---- (1a) selection --------------------------------------------------------------------------
 * Replaces torch.argsort(descending)+slice(+2x torch.sort) at vit_models/dynamic_vit.py:858-862
 * (order = INDEX_ASC, writes kept and dropped) and vit_models/default_dynamic_vit.py:463
 * (order = SCORE_DESC, dropped may be NULL).  Stable: equal scores keep the lower index first;
 * NaN sorts largest.  score (B,N) f32; kept (B,K) i64; dropped (B,N-K) i64 or NULL.  1 <= N <= 1024. */
int d2s_select_topk_f32(const float* score, int B, int N, int K, int order,
                        int64_t* kept, int64_t* dropped, d2s_stream_t stream);

/* Dynamic keep-ratio selection (the prefix-sum form of the select): replaces sort / cumsum / compare / scatter at
 * vit_models/dynamic_vit.py:880-890 (training) and :935-945 (inference).  score (B,N) f32 keep probabilities; a token is
 * kept iff the cumulative sum of the ascending-sorted scores (stable: equal scores in index order; double accumulator rounded
 * to f32 per prefix, as torch's CPU cumsum) at its rank exceeds `threshold`.  mask (B,N) uint8 0/1, count (B) int32 kept
 * tokens per image, kept (B,N) int64 kept indices ascending then -1 padding (what a variable-length gather consumes); any of
 * the three may be NULL. */
int d2s_threshold_select_f32(const float* score, int B, int N, float threshold, uint8_t* mask, int* count, int64_t* kept,
                             d2s_stream_t stream);

/* ---- variable-length (padded) form of the dynamic keep-ratio inference ----------------------------------------------------
 * The inference branch of the threshold mode (dynamic_vit.py:935-960: threshold select, then x.flatten()[mask].reshape(B, -1, D))
 * keeps a different number of tokens per image.  Batched, a stage's tokens are PADDED: x (B,Tmax,D) plus a device length per
 * image (len (B) int32, CLS included); rows len[b]..Tmax-1 are pad rows, written as zeros by the varlen gather and finite (but
 * otherwise unspecified) after it; no valid output depends on them.  Lengths are read on the device (one value per image, clamped
 * to [0, Tmax]); the kernels are the dense ones compiled with the per-image length.
 *
 * d2s_threshold_select_varlen_f32: d2s_threshold_select_f32 on each image's prefix score[b, :n[b]] (score (B,Nmax) f32, n (B)
 * int32); entries past n[b] are never read, their mask is 0 and their kept entry -1.  Replaces dynamic_vit.py:935-945. */
int d2s_threshold_select_varlen_f32(const float* score, const int* n, int B, int Nmax, float threshold, uint8_t* mask, int* count,
                                    int64_t* kept, d2s_stream_t stream);
/* d2s_score_tail_b_varlen: the Variant B tail of d2s_score_tail_b without selection (dynamic_vit.py:547-554) over the first n[b]
 * rows of hidden (B,Nmax,C); the softmax runs over those rows only; pad rows are never read, their scores are -inf and their
 * probabilities 0. */
int d2s_score_tail_b_varlen(const void* hidden, const int* n, int dtype, int B, int Nmax, int C, const float* ln_w, const float* ln_b,
                            float ln_eps, const float* W, const float* bias, int prob_mode, float* scores, float* probs,
                            d2s_stream_t stream);
/* d2s_pool_concat_varlen_inplace: d2s_pool_concat_inplace with the mean over each image's first n[b] rows (dynamic_vit.py:539-545
 * with padding), written into those rows; pad rows are neither read nor written. */
int d2s_pool_concat_varlen_inplace(void* z, const int* n, int dtype, int B, int Nmax, int C, d2s_stream_t stream);
/* d2s_attn_varlen_fwd: Attention.forward's core (dynamic_vit.py:218-234) over the first len[b] tokens of every image, no policy:
 * qkv (B,Tmax,3,H,hd), out (B,Tmax,H*hd), cls_row (B,H,Tmax) f32 or NULL; out rows and cls_row columns >= len[b] are zeros.
 * BF16: the tcgen05 kernel of d2s_attn_policy_fwd (hd == 64), F32: its SIMT parity kernel (hd in {32,64}).  Tmax <= 256; the kernel
 * template is chosen from Tmax.  Valid rows are bit-identical to d2s_attn_policy_fwd run on the image alone when len[b] and Tmax
 * are on the same side of 128. */
int d2s_attn_varlen_fwd(const void* qkv, const int* len, int dtype, int B, int Tmax, int H, int hd, float scale, void* out,
                        float* cls_row, d2s_stream_t stream);
/* d2s_gather_layernorm_varlen / d2s_gather_layernorm_stats_varlen: d2s_gather_layernorm / _stats (dynamic_vit.py:954-960 + the next
 * block's norm1) with idx (B,Kmax) holding image b's count[b] kept spatial indices, then padding that is never read (-1 from the
 * select); output rows 1 + count[b] .. Kmax are zeros (out_sum and out_norm), their stats the (mean, rstd) of a zero row. */
int d2s_gather_layernorm_varlen(const void* x, const int64_t* idx, const int* count, const void* gamma, const void* beta, int dtype,
                                int B, int T_in, int D, int Kmax, float eps, void* out_sum, void* out_norm, d2s_stream_t stream);
int d2s_gather_layernorm_stats_varlen(const void* x, const int64_t* idx, const int* count, int B, int T_in, int D, int Kmax, float eps,
                                      void* out_sum, float* stats, d2s_stream_t stream);

/* ---- (1b) fused predictor tails -----------------------------------------------------------------
 * Variant A tail: Linear(C,2)+LogSoftmax (default_dynamic_vit.py:319-320), then either
 *   eval : top-K of logp[:,:,0] in descending-score order (default_dynamic_vit.py:461-463)  -> kept
 *   train: Gumbel keep decision with injected noise (default_dynamic_vit.py:454; torch
 *          F.gumbel_softmax(hard=True)) times prev_decision                    -> decision, ysoft
 * hidden (B,N,C) f32|bf16 post-GELU activations; W (2,C) f32; bias (2) f32; logp (B,N,2) f32 out.
 * eval:  gumbel=NULL, kept (B,K) i64 (NULL: log-probs only); prev_kept (B,K) f32 or NULL receives
 *        batch_index_select(prev_decision, kept) (default_dynamic_vit.py:467; prev NULL => ones).
 * train: gumbel (B,N,2) f32, prev (B,N) f32, decision (B,N) f32, ysoft (B,N) f32 (soft keep probability).
 * act_input = D2S_ACT_GELU applies the GELU that precedes the last Linear (:318) on load, so `hidden` may be the
 * previous Linear's raw output.  C <= 1024, C % 8 == 0. */
int d2s_score_tail_a(const void* hidden, int dtype, int B, int N, int C,
                     const float* W, const float* bias,
                     int K, const float* gumbel, const float* prev,
                     float* logp, int64_t* kept, float* decision, float* ysoft,
                     int act_input, float* prev_kept, d2s_stream_t stream);

/* Variant B tail: [LayerNorm(C)] + Linear(C,1) + flatten + softmax over N | sigmoid
 * (dynamic_vit.py:424-426, :547-554), then top-K with kept/dropped sorted ascending (:858-862).
 * ln_w/ln_b NULL => no LayerNorm (BatchNorm variants normalise upstream).  W (C) f32, bias (1) f32 device pointer or NULL.
 * scores (B,N) f32 raw logits, probs (B,N) f32, kept (B,K), dropped (B,N-K) (kept may be NULL to skip). */
int d2s_score_tail_b(const void* hidden, int dtype, int B, int N, int C,
                     const float* ln_w, const float* ln_b, float ln_eps,
                     const float* W, const float* bias, int prob_mode, int K,
                     float* scores, float* probs, int64_t* kept, int64_t* dropped, d2s_stream_t stream);

/* Stand-alone Gumbel keep decision and its straight-through backward (default_dynamic_vit.py:454-459).
 * logp, gumbel (n,2); prev, decision, ysoft (n); n = B*N.  decision = hard0 * prev, hard0 = [y0 >= y1].
 * Backward recomputes hard0 / y0 from (logp, gumbel): glogp (n,2) = gout*prev*y0*(1-y0) * (+1,-1);
 * gprev (n) = gout*hard0 (prev is the previous stage's decision and carries gradient at :459), NULL to skip. */
int d2s_gumbel_decision_f32(const float* logp, const float* gumbel, const float* prev, int64_t n,
                            float* decision, float* ysoft, d2s_stream_t stream);
int d2s_gumbel_decision_bwd_f32(const float* gout, const float* logp, const float* gumbel, const float* prev,
                                int64_t n, float* glogp, float* gprev, d2s_stream_t stream);

/* ---- (3) gather / scatter of kept tokens ------------------------------------------------------------
 * prepend_cls=1 replaces cat(0, kept+1) + torch.gather / batch_index_select of the token matrix
 * (dynamic_vit.py:907-912, :954-960; default_dynamic_vit.py:464-466): x (B,T,D), idx (B,K) spatial
 * indices in [0,T-1) -> out (B,K+1,D) with row 0 = CLS.  prepend_cls=0 is plain batch_index_select
 * (default_dynamic_vit.py:37-53, e.g. prev_decision at :467): idx in [0,T) -> out (B,K,D).
 * D*elem_size must be a multiple of 16 for the vector path; other sizes (e.g. D=1) use a scalar path. */
int d2s_gather_tokens(const void* x, int dtype, int B, int T, int D,
                      const int64_t* idx, int K, int prepend_cls, void* out, d2s_stream_t stream);
/* Backward of the gather (autograd of torch.gather at dynamic_vit.py:912): gout (B,K[+1],D) ->
 * gx (B,T,D), rows not selected are zero-filled here.  Indices must be unique per image. */
int d2s_scatter_tokens_bwd(const void* gout, int dtype, int B, int T, int D,
                           const int64_t* idx, int K, int prepend_cls, void* gx, d2s_stream_t stream);

/* ---- (2) PerturbedTopK -----------------------------------------------------------------------------
 * Replaces PerturbedTopKFunction.forward/backward (vit_models/peturbed_topk.py:16-80) without the
 * (b,nS,k,d) one-hot tensor.  x (B,N) f32; noise (B,S,N) f32 standard normal (injected, as the
 * reference draws it on the host at :29); indicators (B,K,N) f32; egrad (B,K,N) f32 = the backward's
 * expected-gradient tensor (:77-78), NULL to skip.  N <= 224, 1 <= K <= N, S >= 1. */
int d2s_ptopk_fwd(const float* x, const float* noise, int B, int N, int K, int S, float sigma,
                  float* indicators, float* egrad, d2s_stream_t stream);
/* Same, drawing the noise in-kernel (Philox4x32-10 + Box-Muller keyed by (seed, b, s, token)); a
 * different, faster contract than the reference's host RNG: statistically equivalent, not bit-equal. */
int d2s_ptopk_fwd_rng(const float* x, uint64_t seed, int B, int N, int K, int S, float sigma,
                      float* indicators, float* egrad, d2s_stream_t stream);
/* grad_x (B,N) = sum_k gout (B,K,N) * egrad (B,K,N)   (peturbed_topk.py:79) */
int d2s_ptopk_bwd(const float* gout, const float* egrad, int B, int N, int K, float* gx,
                  d2s_stream_t stream);

/* ---- (4) policy-masked attention --------------------------------------------------------------------
 * softmax_with_policy as a single pass (dynamic_vit.py:195-214 == default_dynamic_vit.py:185-199):
 *   P_ij = (exp(s_ij - max_j s_ij) * m_ij + eps/T) / (sum_j exp(.)*m_ij + eps),  m_ij = p_j + (1-p_j)[i==j]
 * attn (B,H,T,T) f32|bf16; policy (B,T) f32 or NULL (=> plain softmax, eps ignored); out same dtype;
 * stats (B,H,T,2) f32 = (row max, denominator) saved for backward, may be NULL. */
int d2s_softmax_policy_fwd(const void* attn, const float* policy, int dtype, int B, int H, int T,
                           float eps, void* out, float* stats, d2s_stream_t stream);
/* Backward in both arguments.  gout (B,H,T,T) same dtype as attn; gattn out; gpolicy (B,T) f32 is
 * ACCUMULATED into (caller zero-fills), may be NULL.  Includes the gradient through the subtracted max. */
int d2s_softmax_policy_bwd(const void* attn, const float* policy, const void* gout, const float* stats,
                           int dtype, int B, int H, int T, float eps,
                           void* gattn, float* gpolicy, d2s_stream_t stream);

/* Padded-row variants used by the training attention (ops.attention_train): bf16 only, tensors are (B,H,T,ld) with
 * ld % 8 == 0, T <= ld <= 256, so every row is 16-byte aligned and moved with 16-byte accesses; padding columns of `out`
 * / `gattn` are written as zeros.  gattn may alias gout.  `rows` >= T is the row count of the buffers (rows T..rows-1 of
 * `out` are zero-filled by the forward so the padded tensor can be a GEMM operand; the backward leaves them untouched).
 * The backward omits the gradient through the subtracted row max (sum_j dS_ij = O(eps) * g ~ 1e-6 relative, below bf16
 * resolution; d2s_softmax_policy_bwd keeps it for the fp32 parity runs). */
int d2s_softmax_policy_fwd_ld(const void* attn, const float* policy, int B, int H, int T, int rows, int ld, float eps,
                              void* out, float* stats, d2s_stream_t stream);
int d2s_softmax_policy_bwd_ld(const void* attn, const float* policy, const void* gout, const float* stats, int B, int H,
                              int T, int rows, int ld, float eps, void* gattn, float* gpolicy, d2s_stream_t stream);

/* Head-major relayout for the training attention (dynamic_vit.py:218-221), bf16: token-major packed (B,T,G,H,hd)
 * (G = 3: qkv Linear output; G = 1: attention output / its gradient) <-> head-major (G,B,H,Tp,hd), Tp >= T; split writes
 * the padding rows T..Tp-1 as zeros, merge drops them.  hd % 8 == 0. */
int d2s_split_heads_bf16(const void* src, int B, int T, int Tp, int G, int H, int hd, void* dst, d2s_stream_t stream);
int d2s_merge_heads_bf16(const void* src, int B, int T, int Tp, int G, int H, int hd, void* dst, d2s_stream_t stream);

/* Column sums of a bf16 matrix in fp32: out[n] = sum_m dy[m, n] (out is overwritten): the bias gradient of an nn.Linear
 * under autograd (dynamic_vit.py:159-236).  N % 8 == 0, N <= 8192. */
int d2s_colsum_bf16(const void* dy, long long M, int N, float* out, d2s_stream_t stream);
/* Same, ACCUMULATING: out[n] += sum_m dy[m, n] -- lands the bias gradient straight in the parameter's gradient slot (what
 * autograd's AccumulateGrad node does with a second pass, torch/csrc/autograd/functions/accumulate_grad.h). */
int d2s_colsum_acc_bf16(const void* dy, long long M, int N, float* out, d2s_stream_t stream);

/* GELU backward fused with the bias gradient of the Linear in front of it (Mlp.forward, dynamic_vit.py:170-172), bf16:
 * du (M,N) = ga * gelu'(u) (exact-erf GELU), db (N) f32 = column sums of du (NULL: not wanted; overwritten otherwise). */
int d2s_gelu_bwd_colsum_bf16(const void* u, const void* ga, long long M, int N, void* du, float* db, d2s_stream_t stream);
/* Same with db ACCUMULATED into (db += column sums of du). */
int d2s_gelu_bwd_colsum_acc_bf16(const void* u, const void* ga, long long M, int N, void* du, float* db, d2s_stream_t stream);

/* Token distillation rows: kl_rows[b*N+n] = KL(softmax(t[b,n,:]) || softmax(s[b,n,:])) over the C channels -- the
 * F.kl_div(F.log_softmax(token_s), F.log_softmax(token_t), log_target=True) of BackboneLoss (losses.py:220-225) before its
 * batchmean -- and diff (B*N, C) f32 = softmax(s) - softmax(t), the gradient of kl_rows in s (the backward is a row scaling).
 * s, t: (B,N,C) f32 | bf16 with element strides (batch_stride, C, 1), so x[:, 1:] views are read in place.
 * C % 8 == 0, C <= 1024. */
int d2s_token_kl_fwd(const void* s, int s_dtype, long long s_batch_stride, const void* t, int t_dtype, long long t_batch_stride,
                     int B, int N, int C, float* kl_rows, float* diff, d2s_stream_t stream);

/* AdamW over the slice [begin, end) of flat fp32 buffers p (parameters), g (gradients), m, v (moments), all of one layout:
 * the optimizer.step() of the training loop (train.py:63-66; the reference builds torch/timm AdamW in mask_predictor.py and
 * ddp_training.py), decoupled weight decay, bias correction from the step count:
 *   g' = g * grad_scale;  p *= 1 - lr*wd;  m += (g'-m)(1-beta1);  v = v*beta2 + (1-beta2) g'^2;
 *   p -= lr/(1-beta1^t) * m / (sqrt(v)/sqrt(1-beta2^t) + eps)
 * lr and t (the 1-based step count, as a float) are read from DEVICE memory so a captured CUDA graph serves every step.
 * shadow_bf16 (same layout, NULL: none) receives the updated parameters rounded to bf16 -- the copy the next forward's GEMMs
 * read.  One launch per parameter group (its own lr pointer / weight decay). */
int d2s_adamw_flat_f32(float* p, const float* g, float* m, float* v, void* shadow_bf16, long long begin, long long end,
                       const float* lr, const float* step, float beta1, float beta2, float eps, float weight_decay,
                       float grad_scale, d2s_stream_t stream);

/* Fused attention core of Attention.forward (dynamic_vit.py:218-234; default_dynamic_vit.py:203-213):
 * qkv (B,T,3,H,hd) packed as produced by the qkv Linear; out (B,T,H*hd) ready for the proj Linear;
 * cls_row (B,H,T) f32 = probabilities of query row 0 (dynamic_vit.py:233-234) or NULL.
 * dtype BF16: tcgen05/TMEM tensor-core kernel (hd == 64, T <= 256).
 * dtype F32 : fp32 SIMT kernel used for 1e-4 parity runs (hd in {32,64}, T <= 256).
 * stats (B,H,T,4) f32 or NULL (BF16 only): per query row (m', 1/den, c/den, unused) with e_ij = 2^(k2 s_ij - m') m_ij,
 * den = sum_j e_ij + eps', c = eps'/T (eps' = eps 2^(k2 max_j s_ij - m')): what d2s_attn_policy_bwd recomputes P from.
 * scale > 0.  The exponent reference m' is raised (exactly, by whole binades) whenever a logit exceeds it by more than
 * 100 binades, so the result does not depend on where a row's maximum sits. */
int d2s_attn_policy_fwd(const void* qkv, const float* policy, int dtype, int B, int T, int H, int hd,
                        float scale, float eps, void* out, float* cls_row, float* stats, d2s_stream_t stream);
/* d2s_attn_long_fwd: the same attention core (dynamic_vit.py:195-214 softmax_with_policy, :218-234 Attention.forward) for
 * sequences beyond 256 tokens (384 / 512-pixel inputs): bf16 only, hd == 64, 1 <= T <= 2048, key-blocked tcgen05/TMEM kernel
 * (128-row query tiles x 128-column key blocks, K / V streamed, no (B,H,T,T) tensor, no global scratch).
 * qkv (B,T,3,H,64), out (B,T,H*64), cls_row (B,H,T) f32 or NULL, as d2s_attn_policy_fwd; no row statistics.
 * policy (B,T) f32 or NULL: the policy softmax of d2s_attn_policy_fwd (mask p_j off the diagonal, eps/T on every entry).
 * len (B) int32 or NULL: the variable-length form of d2s_attn_varlen_fwd (image b = its first len[b] tokens, out rows and
 * cls_row columns >= len[b] written as zeros); policy and len are never both given.  scale > 0; B == 0 is a no-op. */
int d2s_attn_long_fwd(const void* qkv, const float* policy, const int* len, int B, int T, int H, int hd, float scale, float eps,
                      void* out, float* cls_row, d2s_stream_t stream);

/* Backward of d2s_attn_policy_fwd (bf16, hd == 64, T <= 208): Attention.forward's core under autograd, differentiable in qkv AND
 * in the keep policy (dynamic_vit.py:195-214, :218-231; default_dynamic_vit.py:185-199, :203-213), flash style -- scores and
 * probabilities are recomputed on chip from qkv and the forward's row statistics, no (B,H,T,T) tensor is read or written.
 *   qkv (B,T,3,H,64), out (B,T,H*64) = the forward's output, gout (B,T,H*64) = d loss / d out,
 *   cls_row / g_cls (B,H,T) f32 or NULL: the forward's CLS-row output and its gradient (g_cls NULL: none),
 *   stats (B,H,T,4) f32 as written by the forward (slot 3 is scratch: delta_i = gout_i . out_i is stored there),
 *   dqkv (B,T,3,H,64) bf16 = d loss / d qkv (every element written), gpolicy (B,T) f32 ACCUMULATED into (caller zero-fills;
 *   NULL iff policy is NULL).  The O(eps) gradient through the subtracted row maximum is not propagated. */
int d2s_attn_policy_bwd(const void* qkv, const float* policy, const void* out, const void* gout, const float* cls_row,
                        const float* g_cls, float* stats, int B, int T, int H, int hd, float scale, void* dqkv,
                        float* gpolicy, d2s_stream_t stream);

/* ---- predictor body (inference path of PredictorLG.forward, default_dynamic_vit.py:324-330; dynamic_vit.py:538-546)
 * d2s_pool_act: z (B,N,C) = in_conv's Linear output; local (B,N,C/2) = act(z[:,:,:C/2]);
 *   pooled (B,C/2) = sum_n act(z[b,n,C/2:]) * policy[b,n] / sum_n policy[b,n]   (policy (B,N) f32; NULL => mean).
 *   local NULL: only pooled is produced (z already activated, its local half consumed in place by the next kernel).
 * d2s_bias_act: u (rows,C) = act(u + bias[row / N]) in place; bias (rows/N, C) (N == 0: one shared row; NULL: none)
 *   -- the per-image term pooled @ W_global^T + b of the split Linear that replaces cat + Linear (:329,
 *   out_conv[0]); with bias NULL it is the in-place activation of Mlp.forward (dynamic_vit.py:170-171).
 *   GELU is the erf form; for bf16 tensors erf is evaluated to ~1e-6 absolute (far below bf16 resolution). */
int d2s_pool_act(const void* z, const float* policy, int dtype, int B, int N, int C, int act, void* local, void* pooled,
                 d2s_stream_t stream);
int d2s_bias_act(void* u, const void* bias, int dtype, long long rows, int N, int C, int act, d2s_stream_t stream);
/* pooled only, over a row slice of a wider bf16 tensor: z points at the first pooled row of image 0, images are z_batch_stride
 * elements apart (x[:, 1:] of a (B,N+1,C) tensor: z = x + C, z_batch_stride = (N+1)*C). */
int d2s_pool_strided_bf16(const void* z, const float* policy, int B, int N, int C, long long z_batch_stride, int act, void* pooled,
                          d2s_stream_t stream);
/* The second half of the Variant-A predictor of one pruning stage as ONE tcgen05 kernel (bf16, D == 384; PredictorLG.forward,
 * default_dynamic_vit.py:329-330 = out_conv on cat(local, pooled.expand), fused with the stage's selection, :461-467):
 * Linear(D,D/2) + GELU (split as local @ W2[:, :D/2]^T + per_image, per_image = pooled @ W2[:, D/2:]^T + b2), Linear(D/2,D/4) +
 * GELU, Linear(D/4,2), LogSoftmax and the stable descending top-K -- replaces two library GEMMs, d2s_bias_act and d2s_score_tail_a.
 *   local (B,N,H) bf16 (H = D/2 = 192) with a row stride of ld elements (ld = H: dense, as written by d2s_pool_act; ld = 2H: the
 *   first half of every row of the (B,N,D) Linear + GELU output, read in place) and a batch stride of lb elements (N * ld when
 *   dense; (N + 1) * ld for the rows 1.. of a (B,N+1,D) tensor), per_image (B,H) bf16; w2 (H,2H) (only its first H columns
 *   are read), w3 (H/2,H) bf16 row-major as nn.Linear stores them, b3 bf16; w4 (2,H/2), b4 (2) f32; prev (B,N) f32 keep
 *   decisions or NULL (all ones);
 *   logp (B,N,2) f32, kept (B,K) int64 in descending-score order (ties: lower index first), prev_kept (B,K) f32 =
 *   prev gathered at kept (NULL to skip).  N <= 256.  The hidden activations never touch HBM. */
int d2s_predictor_a_tail_bf16(const void* local, int ld, long long lb, const void* per_image, const void* w2, const void* w3, const void* b3,
                              const float* w4, const float* b4, const float* prev, int B, int N, int H, int K,
                              float* logp, int64_t* kept, float* prev_kept, d2s_stream_t stream);
/* Variant B's concat (dynamic_vit.py:539-545) in place: z (B,N,C) <- cat(z[:,:,:C/2], mean_n(z[:,:,C/2:]).expand). */
int d2s_pool_concat_inplace(void* z, int dtype, int B, int N, int C, d2s_stream_t stream);

/* Training form of the same local / global split, with autograd in h and in the keep policy (PredictorLG.forward,
 * default_dynamic_vit.py:326-329: policy-weighted mean; dynamic_vit.py:541-545: plain mean, policy NULL), f32 | bf16:
 *   out[b,n,:C/2] = h[b,n,:C/2];  pooled[b,c] = sum_n w[b,n] h[b,n,C/2+c] / sum_n w[b,n];  out[b,n,C/2+c] = pooled[b,c]
 * pooled (B,C/2) f32 and wsum (B) f32 are saved for the backward, which returns dh (B,N,C) and, when dpolicy is not NULL,
 * dpolicy (B,N) f32 = sum_c (h[b,n,C/2+c] - pooled[b,c]) G[b,c] / wsum[b] with G = column sums of dout's global half.
 * policy (B,N) f32.  C/2 a multiple of the 16-byte vector, C/2 <= 768 (bf16) | 384 (f32). */
int d2s_pool_concat_fwd(const void* h, const float* policy, int dtype, int B, int N, int C, void* out, float* pooled,
                        float* wsum, d2s_stream_t stream);
int d2s_pool_concat_bwd(const void* dout, const void* h, const float* policy, const float* pooled, const float* wsum,
                        int dtype, int B, int N, int C, void* dh, float* dpolicy, d2s_stream_t stream);

/* ---- token assembly (dynamic_vit.py:816-824; default_dynamic_vit.py:437-442) -----------------------------------
 * out (B,N+1,D) = cat(cls (D) broadcast, patches (B,N,D)) + pos (N+1,D), one pass instead of concat + add. */
int d2s_assemble_tokens(const void* patches, const void* cls, const void* pos, int dtype, int B, int N, int D,
                        void* out, d2s_stream_t stream);

/* im2col of non-overlapping patches for PatchEmbed.proj as a GEMM (dynamic_vit.py:286-303):
 * img (B,C,H,W) -> out (B, (H/ph)*(W/pw), C*ph*pw) with k = (c, py, px); pw must be a multiple of 8 (bf16) / 4 (f32). */
int d2s_patchify(const void* img, int dtype, int B, int C, int H, int W, int ph, int pw, void* out, d2s_stream_t stream);

/* The same im2col from RAW uint8 images (the host side of the end-to-end path: half the PCIe bytes of bf16): ToTensor + Normalize
 * -- x / 255, then (x - mean[c]) / std[c] in fp32, rounded to out_dtype -- applied on the fly, bit-identical to the torch
 * pipeline (per-channel 256-entry table built with the same IEEE operations).  mean, std (C) f32; C <= 4, W % 16 == 0. */
int d2s_patchify_u8(const void* img, const float* mean, const float* std, int out_dtype, int B, int C, int H, int W, int ph, int pw,
                    void* out, d2s_stream_t stream);

/* ---- residual add + LayerNorm ("next" row of the scope table: Block.forward) -----------------------------
 * Inference path of x = x + branch; h = norm(x) (dynamic_vit.py:263-283; default_dynamic_vit.py:234-237) and of the
 * predictors' leading LayerNorm over x[:, 1:] (dynamic_vit.py:409, :491; default_dynamic_vit.py:308) in one pass:
 *   s = x + y (rounded to dtype; y NULL => s = x), out_sum (B,T,D) = s (NULL to skip),
 *   out_norm (B,T-norm_row0,D) = LayerNorm(s[:, norm_row0:]) * gamma + beta, statistics in fp32.
 * x is (B,T,D) with element strides (x_stride_b, x_stride_t) and contiguous rows; y, outputs contiguous;
 * gamma, beta (D) in the same dtype as x.  D % 8 == 0 (bf16) / D % 4 == 0 (f32), D <= 1536 (bf16) / 768 (f32). */
int d2s_add_layernorm(const void* x, const void* y, const void* gamma, const void* beta, int dtype, int B, int T, int D,
                      long long x_stride_b, long long x_stride_t, float eps, int norm_row0,
                      void* out_sum, void* out_norm, d2s_stream_t stream);

/* Kept-token gather fused with the LayerNorm that follows it (default_dynamic_vit.py:464-468 / dynamic_vit.py:907-912, then
 * Block.forward's norm1): out_sum (B,K+1,D) = [CLS, x[:, idx+1]] (x (B,T_in,D) contiguous, idx (B,K) int64 spatial indices),
 * out_norm (B,K+1,D) = LayerNorm(out_sum) * gamma + beta.  Same dtype / D constraints as d2s_add_layernorm. */
int d2s_gather_layernorm(const void* x, const int64_t* idx, const void* gamma, const void* beta, int dtype, int B, int T_in,
                         int D, int K, float eps, void* out_sum, void* out_norm, d2s_stream_t stream);

/* Token assembly fused with the first block's norm1 (dynamic_vit.py:820-823 + Block.forward :263; default_dynamic_vit.py:440-443):
 * out_sum (B,N+1,D) = cat(cls, patches) + pos, out_norm = LayerNorm(out_sum) * gamma + beta.
 * patches (B,N,D), cls (D), pos (N+1,D), all of `dtype`. */
int d2s_assemble_layernorm(const void* patches, const void* cls, const void* pos, const void* gamma, const void* beta, int dtype,
                           int B, int N, int D, float eps, void* out_sum, void* out_norm, d2s_stream_t stream);
/* The same two with per-row (mean, rstd) of out_sum instead of the normalised output (bf16): the consumer -- the qkv projection,
 * d2s_linear_lnin_act_pair_bf16 -- applies norm1 to its resident input rows itself, so LayerNorm(out_sum) is never written or read.
 * stats (B*(K+1), 2) / (B*(N+1), 2) f32. */
int d2s_gather_layernorm_stats(const void* x, const int64_t* idx, int B, int T_in, int D, int K, float eps, void* out_sum,
                               float* stats, d2s_stream_t stream);
int d2s_assemble_layernorm_stats(const void* patches, const void* cls, const void* pos, int B, int N, int D, float eps, void* out_sum,
                                 float* stats, d2s_stream_t stream);
/* out (rows, D) bf16 = LayerNorm of rows of x taken from GIVEN statistics (row r of x at x + r * x_row_stride elements, its (mean,
 * rstd) at stats + 2 * r * stat_row_stride floats), with the arithmetic of the GEMM kernels' on-the-fly normalisation: for the few
 * rows another consumer needs materialised (the CLS rows in front of the CLS-only last MLP). */
int d2s_apply_layernorm_stats_bf16(const void* x, const float* stats, const void* gamma, const void* beta, int rows, int D,
                                   long long x_row_stride, long long stat_row_stride, void* out, d2s_stream_t stream);

/* Linear + activation in one tcgen05 GEMM (fc1 + GELU of Mlp.forward, dynamic_vit.py:159-175), bf16 only:
 * out (M,N) = act(a (M,K) @ w (N,K)^T + bias (N)); fp32 accumulation; bias may be NULL.
 * N % 256 == 0 or N % 192 == 0 (256- or 192-column tiles; N <= 4096), K % 64 == 0.  CTA pair (tcgen05 cta_group::2, 256-row tiles, half of the weight tile per CTA).
 * pre (M,N) or NULL: also write the pre-activation a @ w^T + bias (training: GELU' needs it; saves torch's separate GELU pass). */
int d2s_linear_act_pair_bf16(const void* a, const void* w, const void* bias, int M, int N, int K, int act, void* out,
                             void* pre, d2s_stream_t stream);
/* The same with the LayerNorm of the INPUT rows applied on the fly (Block.forward's norm1 in front of attn.qkv, dynamic_vit.py:277;
 * N % 192 == 0, N % 256 != 0, K <= 384): x (M,K) is the residual stream, in_stats (M,2) f32 its per-row (mean, rstd) as written by
 * d2s_mlp_lnin_residual_ln_bf16 (out_stats), in_gamma / in_beta (K) bf16; the row tile is normalised in shared memory (bit-identical
 * to the normalised copy) before the MMAs read it. */
int d2s_linear_lnin_act_pair_bf16(const void* x, const float* in_stats, const void* in_gamma, const void* in_beta, const void* w,
                                  const void* bias, int M, int N, int K, int act, void* out, d2s_stream_t stream);

/* Linear + residual add + LayerNorm in one tcgen05 GEMM: attn.proj / mlp.fc2 of Block.forward together with the
 * residual add and the NEXT LayerNorm (dynamic_vit.py:263-283: x = x + attn(norm1(x)); x = x + mlp(norm2(x))), bf16 only:
 *   y = bf16(a (M,K) @ w (N,K)^T + bias (N));  out_sum (M,N) = bf16(x (M,N) + y);
 *   out_norm (M,N) = LayerNorm(out_sum) * gamma + beta (statistics in fp32), or skipped when out_norm is NULL.
 * Roundings are the reference's (Linear output, residual sum, LayerNorm output each rounded to bf16).
 * N in {192, 384} (a CTA keeps whole rows in TMEM) or 768 (DeiT-B: two 384-column halves accumulated one after the other, the
 * row statistics carried across), K % 64 == 0; x may alias out_sum. */
int d2s_linear_residual_ln_bf16(const void* a, const void* w, const void* bias, const void* x, const void* gamma,
                                const void* beta, float eps, int M, int N, int K, void* out_sum, void* out_norm,
                                d2s_stream_t stream);
/* The same without the normalised output: out_sum = x + bf16(a @ w^T + bias) and stats (M,2) f32 = per-row (mean, rstd) of out_sum
 * (rstd = rsqrt(var + eps)); the consumer (d2s_mlp_lnin_residual_ln_bf16) applies the LayerNorm itself, which saves writing and
 * re-reading the (M,N) normalised copy. */
int d2s_linear_residual_stats_bf16(const void* a, const void* w, const void* bias, const void* x, float eps, int M, int N, int K,
                                   void* out_sum, float* stats, d2s_stream_t stream);

/* The whole MLP branch of Block.forward in one kernel (dynamic_vit.py:159-175, :263-283), bf16, D == 384:
 *   u = GELU(h (M,D) @ w1 (HID,D)^T + b1);  out_sum (M,D) = bf16(x + bf16(u @ w2 (D,HID)^T + b2));
 *   out_norm (M,D) = LayerNorm(out_sum) * gamma + beta, or skipped when out_norm is NULL.
 * The (M,HID) hidden activations never leave the SM (128-column chunks through TMEM and shared memory); roundings are the
 * reference's (fc1 output after GELU, fc2 output, residual sum, LayerNorm output each rounded to bf16).
 * The M rows are B images of T tokens; out_norm skips the first norm_row0 tokens of every image and is (B, T-norm_row0, D)
 * (the predictors' LayerNorm over x[:, 1:], dynamic_vit.py:409, default_dynamic_vit.py:308); T = 1, norm_row0 = 0 for plain rows.
 * HID % 128 == 0, 128 <= HID <= 2048; x may alias out_sum. */
int d2s_mlp_residual_ln_bf16(const void* h, const void* w1, const void* b1, const void* w2, const void* b2, const void* x,
                             const void* gamma, const void* beta, float eps, int M, int D, int HID, int T, int norm_row0,
                             void* out_sum, void* out_norm, d2s_stream_t stream);
/* The same with the LayerNorm of the MLP's INPUT applied on the fly (Block.forward's norm2, dynamic_vit.py:281): x (M,D) is the
 * residual stream itself, in_stats (M,2) f32 its per-row (mean, rstd) as written by d2s_linear_residual_stats_bf16, in_gamma /
 * in_beta (D) bf16 that LayerNorm's affine; h = bf16((x - mean) * rstd * gamma + beta) is formed in shared memory (the arithmetic of
 * d2s_linear_residual_ln_bf16's own LayerNorm pass: bit-identical A operand) and never written to HBM.  x is also the residual input.
 * out_stats (M,2) f32 or NULL: per-row (mean, rstd) of out_sum for `eps`, for a consumer that applies the NEXT LayerNorm itself
 * (d2s_linear_lnin_act_pair_bf16: the next block's qkv projection); out_norm may then be NULL. */
int d2s_mlp_lnin_residual_ln_bf16(const void* x, const float* in_stats, const void* in_gamma, const void* in_beta, const void* w1,
                                  const void* b1, const void* w2, const void* b2, const void* gamma, const void* beta, float eps,
                                  int M, int D, int HID, int T, int norm_row0, void* out_sum, void* out_norm, float* out_stats,
                                  d2s_stream_t stream);

/* LayerNorm forward / backward for the training path (norm1 / norm2 / predictor norms of Block.forward,
 * dynamic_vit.py:263-283) with mixed dtypes for bf16 autocast: x (rows,D) f32|bf16 -> h (rows,D) f32|bf16,
 * gamma/beta f32 (D), stats (rows,2) f32 = (mean, rstd) saved for backward.  Backward: dx (dtype of x),
 * dgamma/dbeta (D) f32 are ACCUMULATED into (caller zero-fills).  D % 8 == 0, D <= 768. */
int d2s_layernorm_fwd(const void* x, int x_dtype, const float* gamma, const float* beta, long long rows, int D,
                      float eps, void* h, int h_dtype, float* stats, d2s_stream_t stream);
int d2s_layernorm_bwd(const void* dh, int h_dtype, const void* x, int x_dtype, const float* stats, const float* gamma,
                      long long rows, int D, void* dx, float* dgamma, float* dbeta, d2s_stream_t stream);

/* The same over the rows `skip`.. of every (seg + skip)-row segment of x -- LayerNorm(x[:, 1:]) as the predictors apply it
 * (default_dynamic_vit.py:461 -> :313, dynamic_vit.py:846 -> :386) without the slice copy: x holds rows/seg segments of
 * seg + skip rows, h and stats are dense over the `rows` normalised rows (rows % seg == 0).  Backward writes dx in x's layout,
 * zeros in the skipped rows. */
int d2s_layernorm_seg_fwd(const void* x, int x_dtype, const float* gamma, const float* beta, long long rows, int D, int seg,
                          int skip, float eps, void* h, int h_dtype, float* stats, d2s_stream_t stream);
int d2s_layernorm_seg_bwd(const void* dh, int h_dtype, const void* x, int x_dtype, const float* stats, const float* gamma,
                          long long rows, int D, int seg, int skip, void* dx, float* dgamma, float* dbeta, d2s_stream_t stream);

/* The residual add folded into the LayerNorm that follows it, training path (Block.forward, dynamic_vit.py:276-283:
 * x = x + branch; norm(x)): forward writes out_sum = x + res (dtype of x) and h = LayerNorm(out_sum) (+ stats); backward
 * returns dx = LayerNorm input gradient + gsum, gsum = the gradient that reaches out_sum directly (NULL: none). */
int d2s_add_layernorm_fwd(const void* x, const void* res, int x_dtype, const float* gamma, const float* beta, long long rows,
                          int D, float eps, void* out_sum, void* h, int h_dtype, float* stats, d2s_stream_t stream);
int d2s_add_layernorm_bwd(const void* dh, int h_dtype, const void* xsum, int x_dtype, const float* stats, const float* gamma,
                          const void* gsum, long long rows, int D, void* dx, float* dgamma, float* dbeta, d2s_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* D2S_H */
