/*
 * merv_fusion.h — C ABI of libmerv_fusion.so: MERV's multi-encoder feature-fusion hot path on B200 (sm_100a).
 *
 * The reference (princetonvisualai/merv) is pure Python/PyTorch and has no FFI; the boundary it exposes for
 * this path is the nn.Module surface of merv/util/nn_utils.py.  Each entry point below replaces the body of
 * one reference method (cited as file:line, relative to the reference root) and is what a ctypes binding in
 * that file would call (see INTEGRATION.md).  Conventions:
 *
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer owned by the caller (PyTorch's caching
 *     allocator in practice); the library allocates no device memory and keeps no reference after return;
 *   - every call is asynchronous and ordered on `stream` (a cudaStream_t passed as void*), does no host
 *     synchronisation and is CUDA-graph capturable;
 *   - return value: 0 on success, a negative MERV_E_* code otherwise; merv_last_error() gives the message of
 *     the calling thread's last failure.  There is NO CPU fallback: a non-sm_100 device is MERV_E_ARCH;
 *   - tensors are row-major with the channel/feature dimension contiguous; `dtype` selects the element type of
 *     activations AND weights (MERV_BF16: bf16 storage, fp32 accumulation, tcgen05 tensor cores for the
 *     projector GEMMs; MERV_F32: fp32 storage and SIMT fp32 arithmetic, the 1e-5 parity path).
 */
#ifndef MERV_FUSION_H_
#define MERV_FUSION_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MERV_ABI_VERSION 5

enum { MERV_F32 = 0, MERV_BF16 = 1 };
enum { MERV_ACT_NONE = 0, MERV_ACT_GELU_ERF = 1 };
enum {
  MERV_OK = 0,
  MERV_E_SHAPE = -1,   /* a dimension is non-positive / inconsistent / unsupported */
  MERV_E_ALIGN = -2,   /* a pointer or leading dimension violates the 16-byte alignment the kernels need */
  MERV_E_DTYPE = -3,   /* unknown dtype / activation code, or combination not implemented */
  MERV_E_ARCH = -4,    /* current device is not compute capability 10.x */
  MERV_E_CUDA = -5,    /* a CUDA runtime / driver call failed (message has the CUDA error string) */
  MERV_E_ARG = -6      /* null pointer where one is required, too many encoders, ... */
};

#define MERV_MAX_ENCODERS 8
#define MERV_MAX_SEGMENTS 4
#define MERV_ROWDOT_BLOCK 64 /* column-block width of the row-dot partials emitted by the GEMM epilogue */

int merv_abi_version(void);
const char* merv_last_error(void);
/* 0 if the CURRENT device can run the library (sm_100), MERV_E_ARCH otherwise. */
int merv_device_check(void);
int merv_num_sms(void);

/* ---------------------------------------------------------------------------------------------------------
 * Adaptive spatio-temporal average pooling, channel-last in and out.
 * Replaces AveragePooling3DProjector.forward's rearrange -> AdaptiveAvgPool3d -> rearrange
 * (merv/util/nn_utils.py:320-329) for up to MERV_MAX_ENCODERS encoders in ONE launch.
 *
 *   x : [B, F, H*W, C]  (element strides x_batch_stride / x_frame_stride / x_token_stride, channel stride 1)
 *   y : [B, T*S*S, C]   token index t*S*S + i*S + j (j fastest); row stride y_row_stride elements
 *   window k of an axis n_in -> n_out is [floor(k*n_in/n_out), ceil((k+1)*n_in/n_out))
 *   score_vec / score_partial (optional, fp32): score_partial[b, i] = partial sums (one per internal work
 *     item i of video b, deterministic order) of sum_{tokens, channels} score_vec[c] * Y[b, token, c] with Y as
 *     rounded to the storage dtype; the number of partials per video is shape-dependent only and is given by
 *     merv_pool3d_score_parts().  Feeds the encoder scores of the affine fast path (see merv_affine_score_vec).
 * Accumulation is fp32 for both dtypes (as ATen's kernel does).  C % 8 == 0 (bf16) or C % 4 == 0 (fp32).
 * The main kernel streams the input through shared memory with 5-D TMA; unusual shapes (more than 2048 patch
 * tokens per frame) take a plain vectorised-load kernel.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct {
  const void* x;
  void* y;
  const float* score_vec; /* [C] or NULL */
  float* score_partial;   /* [B, parts] or NULL (both or neither) */
  const int32_t* batch_index; /* [B] or NULL: output video b reads input video batch_index[b] (the gather by
                                 `multimodal_indices` at merv/models/vidlms/merv.py:572 fused into the load) */
  int32_t src_batch;          /* videos in x when batch_index is given (0 = B) */
  int32_t F, H, W, C, T, S;
  int64_t x_batch_stride, x_frame_stride, x_token_stride;
  int64_t y_batch_stride, y_row_stride;
  /* ABI v5: the pooling windows read x displaced by (shift_f, shift_h, shift_w) frames / patch rows / patch columns, positions that
   * fall outside the [F, H, W] grid contributing ZERO while the divisor stays the full window size — i.e. the adaptive average pool of
   * one tap of a zero-padded "same" convolution.  pool(conv3d(x)) = sum_taps W_tap pool(shift_tap(x)) + b, so the 27 shifted poolings
   * written side by side ([B, T*S*S, 27*C], y_row_stride = 27*C) are the A operand of ONE GEMM that evaluates
   * Convolutional3DProjector.convolution_pooling (merv/util/nn_utils.py:349-352,364) on the pooled grid.  All zero: plain pooling. */
  int32_t shift_f, shift_h, shift_w, reserved_;
} merv_pool_desc;

/* parts[e] = number of score partials per video the pool kernel emits for encoder e (independent of B). */
int merv_pool3d_score_parts(const merv_pool_desc* enc, int num_encoders, int dtype, int32_t* parts);
/* max_ctas: 0 = one persistent CTA per SM; k > 0 caps the grid at k CTAs so the kernel can share the GPU with a
 * concurrently running kernel on another stream (see merv_fused_linear_mix). */
int merv_pool3d(const merv_pool_desc* enc, int num_encoders, int B, int dtype, int max_ctas, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Projector layer: Y = act(A W^T + bias).  Replaces nn.Linear (+ nn.GELU) inside LinearProjector.forward /
 * MLPProjector.forward / FusedMLPProjector.forward (merv/util/nn_utils.py:31-32,46-55,97-108).
 *
 *   A [M, K] (lda), W [N, K] (ldw, PyTorch nn.Linear layout), bias [N] (dtype of W; may be NULL), Y [M, N] (ldy)
 *   act: MERV_ACT_NONE | MERV_ACT_GELU_ERF (exact erf GELU, nn.GELU() default)
 *   rowdot_vec / rowdot_out (optional, bf16 path only): rowdot_out[m, j] = sum over columns n of block j
 *     (MERV_ROWDOT_BLOCK wide) of rowdot_vec[n] * Y[m, n] (Y as rounded to the output dtype); shape
 *     [M, ceil(N / MERV_ROWDOT_BLOCK)] fp32.  Feeds the encoder scores without re-reading Y.
 * MERV_BF16 runs on tcgen05 (TMA-fed, TMEM accumulators); needs K % 8 == 0, N % 8 == 0, 16-byte aligned bases.
 * ------------------------------------------------------------------------------------------------------- */
int merv_linear_bias_act(const void* A, int64_t lda, const void* W, int64_t ldw, const void* bias, void* Y,
                         int64_t ldy, int M, int N, int K, int act, int dtype, const float* rowdot_vec,
                         float* rowdot_out, void* stream);

/* The same GEMM with either operand given TRANSPOSED in memory (bf16, tensor cores only): a_mn != 0: A is stored as [K, M] row-major
 * (lda = its row stride), w_mn != 0: W is stored as [K, N] row-major.  tcgen05 reads MN-major operands straight from shared memory
 * (TMA boxes of 64 M / N elements x 64 k-rows, 128-byte swizzle), so the backward of a Linear needs no transposed copies:
 *   dW [N_out, K_in] = dY^T X : A = dY [M, N_out] with a_mn, W-operand = X [M, K_in] with w_mn, contraction over the M tokens
 *   dX [M, K_in]     = dY W   : A = dY (K-major),           W-operand = W [N_out, K_in] with w_mn, contraction over N_out
 * (autograd of merv/util/nn_utils.py:31-32,46-55 inside the training step, base_strategy.py:240-241).  With both operands MN-major K
 * may be any positive number (the k tail is zero-filled); otherwise K % 8 == 0. */
int merv_gemm_ex(const void* A, int64_t lda, int a_mn, const void* W, int64_t ldw, int w_mn, const void* bias, void* Y, int64_t ldy,
                 int M, int N, int K, int act, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * The learnable-query "cross attention" collapses to a dot product with an input-independent vector
 * (SURVEY.md §3.3): weights[b,:] = softmax_e(u . mean_t V[b,e,t,:]),
 *   u = Wk^T (Wq Q^T + b_q) / sqrt(embed).
 * Replaces the q/k projections inside nn.MultiheadAttention as called at merv/util/nn_utils.py:499-512.
 *   Q [1, embed], Wq [embed, embed], Wk [embed, llm_dim], in_proj_bias [3*embed] (dtype); u [llm_dim] fp32;
 *   workspace: at least embed floats; with round_up(embed, 4) + merv_gemv_t_workspace(embed, llm_dim) floats the transposed
 *   GEMV Wk^T q runs in its two-stage form (row blocks in parallel; matters when llm_dim / 32 CTAs cannot fill the GPU).
 *   Both run once per weight version in inference but once per optimizer step in training.
 * ------------------------------------------------------------------------------------------------------- */
size_t merv_gemv_t_workspace(int D, int K); /* floats; 0 = the single-stage kernel is used for a [D, K] matrix */
int merv_fusion_query_vec(const void* Q, const void* Wq, const void* Wk, const void* in_proj_bias, float* u,
                          float* workspace, size_t workspace_floats, int embed, int llm_dim, int dtype, void* stream);

/* For an affine last projector layer y = W x + b:  u . y = (W^T u) . x + u . b.
 *   W [N, K] (ldw), bias [N] or NULL, u [N] fp32  ->  v [K] fp32, c [1] fp32.
 *   workspace (optional, merv_gemv_t_workspace(N, K) floats): two-stage W^T u. */
int merv_affine_score_vec(const void* W, int64_t ldw, const void* bias, const float* u, float* v, float* c, float* workspace,
                          size_t workspace_floats, int N, int K, int dtype, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Scores -> softmax over encoders -> mixing weights.  Two sources for the raw scores [B, E] (fp32):
 *   merv_scores_from_tokens   : s[b,e] = mean_t(u . V_e[b,t,:]) read from the projected tokens themselves
 *                               (general path; V_e [B, T_e, K] with T_e in {T, 1}, nn_utils.py:494-509)
 *   merv_scores_from_partials : s[b,e] = (1/T) * sum_{i < count[e]} partial_e[b, i] + c_e, from partial dot
 *                               products emitted by the pool kernel (score_partial) or by the GEMM epilogue
 *                               (rowdot_out, count = T * ceil(N / MERV_ROWDOT_BLOCK)) — no re-read of V.
 * Both use a fixed reduction order (no atomics): results are bit-reproducible per video.
 * ------------------------------------------------------------------------------------------------------- */
int merv_scores_from_tokens(const void* const* V, const int32_t* tokens, const float* u, float* scores,
                            float* workspace, size_t workspace_floats, int B, int E, int T, int K, int dtype,
                            void* stream);
size_t merv_scores_from_tokens_workspace(int B, int E, int T, int K);
/* General form of merv_scores_from_tokens, covering the other two branches of CrossAttentionAdapterLearnableQuery.forward:
 *   u_token_stride == K (averagetoken=False, merv/util/nn_utils.py:514-518): the key is the flattened [T*K] token block, so u
 *       (merv_fusion_query_vec with llm_dim = T*K) has one row per token; s[b,e] = sum_t u[t,:] . V_e[b,t,:] with a single-token
 *       encoder read T times (its repeat at nn_utils.py:502).  u_token_stride == 0 is the averagetoken=True form.
 *   c (fp32 [E] or NULL): additive per-encoder constants, s[b,e] += c[e] — positional_embedding=True adds pe[e] to the mean
 *       token (nn_utils.py:510-511), i.e. c[e] = u . pe[e] (merv_score_consts).
 *   mean != 0 divides the sum by the number of tokens (the token mean of nn_utils.py:508). */
int merv_scores_from_tokens_ex(const void* const* V, const int32_t* tokens, const float* u, int64_t u_token_stride,
                               const float* c, int mean, float* scores, float* workspace, size_t workspace_floats, int B,
                               int E, int T, int K, int dtype, void* stream);
/* c_out[e] = u . pe[e,:] + (c_in && c_in[e] ? *c_in[e] : 0);  pe [E, K] (ldpe) in `dtype`, u fp32 [K], c_out fp32 [E]. */
int merv_score_consts(const void* pe, int64_t ldpe, const float* u, const float* const* c_in, float* c_out, int E, int K,
                      int dtype, void* stream);
int merv_scores_from_partials(const float* const* partial, const int32_t* count,
                              const float* const* c /* per-encoder additive constants, entries or array may be NULL */,
                              float* scores, int B, int E, int T, void* stream);

/* weights[b,:] = softmax(scores[b,:]) (fp32);  optionally bias_mix[b,n] = sum_e weights[b,e] * bias_e[n]
 * (the per-video bias of the fused affine path; bias_e in `dtype`, may contain NULL entries).
 * merv_softmax_weights_ex additionally writes a bf16 copy of the weights (what the modules return in bf16 mode). */
int merv_softmax_weights(const float* scores, float* weights, const void* const* bias, float* bias_mix, int B,
                         int E, int N, int dtype, void* stream);
int merv_softmax_weights_ex(const float* scores, float* weights, void* weights_bf16, const void* const* bias,
                            float* bias_mix, int B, int E, int N, int dtype, void* stream);

/* merv_scores_from_partials + merv_softmax_weights_ex in one launch (bf16 biases), bit-identical to the pair. */
int merv_scores_softmax_weights(const float* const* partial, const int32_t* count, const float* const* c,
                                const void* const* bias, float* scores, float* weights, void* weights_bf16,
                                float* bias_mix, int B, int E, int T, int N, void* stream);

/* out[b,t,:] = sum_e weights[b,e] * V_e[b,t,:]   — replaces torch.stack + torch.bmm at nn_utils.py:503,521.
 * Reads every V_e element once, writes every fused token once.  T_e in {T, 1} (broadcast, nn_utils.py:502).
 * If `scores` is non-NULL the softmax is done in-kernel (warp shuffles over the E lanes) and `weights` is an
 * output; otherwise `weights` is an input. */
int merv_softmax_mix(const void* const* V, const int32_t* tokens, const float* scores, float* weights, void* out,
                     int B, int E, int T, int K, int dtype, void* stream);
/* merv_softmax_mix writing video b's fused tokens at out + b * out_batch_stride, rows ldo apart: the prefix slot of the
 * [B, bos + T + L_text, K] multimodal embedding buffer that MERV.forward otherwise builds with torch.cat (merv.py:633-640).  Writes
 * nothing outside the [B, T, K] block.  ldo and out_batch_stride whole 16-byte vectors (MERV_E_ALIGN), ldo >= K and
 * out_batch_stride >= T * ldo (MERV_E_SHAPE).  merv_softmax_mix is this call with ldo = K, out_batch_stride = T * K (bit-identical). */
int merv_softmax_mix_ex(const void* const* V, const int32_t* tokens, const float* scores, float* weights, void* out, int64_t ldo,
                        int64_t out_batch_stride, int B, int E, int T, int K, int dtype, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Fused affine path (the shipped "3davg+linear" + "cross_attention_avg_lq" configuration):
 *   out[m,:] = sum_s scale[video(m), s] * (A_s[m,:] W_s^T) + bias_mix[video(m), :]
 * One persistent tcgen05 kernel; per-encoder projected tokens are never written to HBM; each fused token is
 * written exactly once.  A_s [M, K_s] (lda[s]) are the pooled features, W_s [N, K_s] (ldw[s]);
 * scale [M / rows_per_video, nseg] fp32 (the mixing weights), bias_mix [M / rows_per_video, N] fp32.
 * out_batch_stride (elements): 0 or rows_per_video * ldo = one contiguous [M, N] output; larger = video b's rows start at
 * out + b * out_batch_stride, i.e. the prefix is written straight into its slot of the [B, bos + T + L_text, N] multimodal
 * embedding buffer that MERV.forward otherwise builds with torch.cat (merv.py:633-640); needs rows_per_video % 128 == 0.
 * Replaces LinearProjector.forward x E + CrossAttentionAdapterLearnableQuery.forward's stack/bmm
 * (nn_utils.py:31-32,503,521).  bf16 only.  max_ctas: 0 = one CTA per SM; k > 0 caps the persistent grid at k CTAs, leaving
 * the remaining SMs to a concurrently running HBM-bound kernel (the pool of the next chunk of videos): the GEMM is
 * tensor-bound and the pool HBM-bound, so running them side by side hides the pool.
 * ------------------------------------------------------------------------------------------------------- */
int merv_fused_linear_mix(const void* const* A, const int64_t* lda, const void* const* W, const int64_t* ldw,
                          const int32_t* K, int nseg, const float* scale, const float* bias_mix, void* out,
                          int64_t ldo, int64_t out_batch_stride, int M, int N, int rows_per_video, int max_ctas,
                          void* stream);

/* Channel-concat fusion (feature_fusion == "concat_channel"): out = concat_s(A_s, dim=-1) W^T + bias as ONE K-segmented
 * tcgen05 GEMM, out[m,:] = sum_s A_s[m,:] W[:, k_s : k_s + K_s]^T + bias — the [M, sum K_s] concatenation the reference
 * builds with torch.concat (merv.py:603-605) before its LinearProjector(E * llm_dim, llm_dim) (merv.py:217-218,606) is
 * never materialised.  A_s [M, K_s] (lda[s]) are the per-encoder projected tokens, W [N, sum K_s] (ldw) row-major
 * (nn.Linear layout), bias [N] bf16 or NULL.  bf16 only, nseg <= MERV_MAX_SEGMENTS. */
int merv_concat_linear(const void* const* A, const int64_t* lda, const void* W, int64_t ldw, const int32_t* K, int nseg,
                       const void* bias, void* out, int64_t ldo, int M, int N, void* stream);

/* Fused GEMM + all-gather over NVLink peer memory: as merv_fused_linear_mix, and every finished output tile is ALSO stored
 * (TMA stores to peer-mapped addresses) to the same rows of `peer_out[0..num_peers)` — the other ranks' symmetric prefix
 * buffers, already offset to this rank's block of videos.  The transfer overlaps the tensor-core work tile by tile; the
 * caller synchronises the ranks afterwards (e.g. the symmetric-memory barrier).  Replaces "compute, then ncclAllGather"
 * for consumers that want the whole batch's prefixes on every rank (SURVEY.md §8e).  num_peers <= 7. */
int merv_fused_linear_mix_gather(const void* const* A, const int64_t* lda, const void* const* W, const int64_t* ldw,
                                 const int32_t* K, int nseg, const float* scale, const float* bias_mix, void* out,
                                 int64_t ldo, int64_t out_batch_stride, int M, int N, int rows_per_video, int max_ctas,
                                 void* const* peer_out, int num_peers, void* stream);

/* The same all-gather through the NVSwitch MULTICAST mapping of the symmetric buffers: `mc_out` is the multicast address of this
 * rank's block (one virtual address that the switch replicates into the buffer of EVERY rank, the caller's included), and every
 * finished output box is written exactly once with multimem.st (16 bytes per thread, 128-byte rows) instead of once per peer.
 * NVLink egress per GPU drops from (ranks - 1) x block to 1 x block; what remains is each GPU's ingress of the other ranks'
 * blocks.  `out` receives nothing separately (the multicast covers the local buffer) but must be the local address of the
 * same block: it only provides the shape checks.  Flat [M, N] output with leading dimension ldo; bf16. */
int merv_fused_linear_mix_multicast(const void* const* A, const int64_t* lda, const void* const* W, const int64_t* ldw,
                                    const int32_t* K, int nseg, const float* scale, const float* bias_mix, void* out,
                                    int64_t ldo, int M, int N, int rows_per_video, int max_ctas, void* mc_out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Whole fused path in ONE call (affine "linear" projectors, bf16): pool -> scores -> softmax -> fused GEMM, i.e.
 * merv/models/vidlms/merv.py:587-589 + 607-609 for the shipped "3davg+linear" + "cross_attention_avg_lq" configs.
 * Exists for the small-batch serving case (generate runs the path once per video at B = 1), where host overhead per
 * launch dominates: 3 kernels are enqueued from one FFI crossing.  All workspaces are caller-provided.
 *   pool[e]        : as for merv_pool3d; .y is the pooled workspace [B, T*S*S, C_e], .score_vec = v_e (fp32 [C_e]),
 *                    .score_partial = workspace [B, parts_e] (parts_e from merv_pool3d_score_parts)
 *   W, ldw, bias, c: last-layer weights [N, C_e], biases [N] (bf16) and score constants c_e (fp32 [1]) per encoder
 *   scores, weights: workspaces fp32 [B, E]; bias_mix fp32 [B, N]; weights_bf16 (optional) bf16 [B, E] copy of weights
 *   out            : bf16 [B, rows_per_video, N] with row stride ldo and batch stride out_batch_stride (0 = contiguous)
 * ------------------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t num_encoders, B, N, rows_per_video;
  merv_pool_desc pool[MERV_MAX_SEGMENTS];
  int32_t parts[MERV_MAX_SEGMENTS];
  const void* W[MERV_MAX_SEGMENTS];
  int64_t ldw[MERV_MAX_SEGMENTS];
  const void* bias[MERV_MAX_SEGMENTS];
  const float* c[MERV_MAX_SEGMENTS];
  float* scores;
  float* weights;
  float* bias_mix;
  void* weights_bf16; /* may be NULL */
  void* out;
  int64_t ldo, out_batch_stride;
  /* reserved: ignored by the library; they keep the ABI v5 layout, so any value a v5 caller stores here is harmless */
  int32_t* reserved_ptr_;
  int32_t reserved_[2];
} merv_fused_desc;

int merv_fused_forward(const merv_fused_desc* d, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Backward of the module-by-module path (training drop-in; projectors and adapter are trainable in every stage,
 * merv/models/vidlms/merv.py:318-320,342-343,363-365; backbones are frozen so nothing flows into the features).
 *   merv_transpose : y[c, r] = x[r, c]           (operands of dW = dY^T P for the K-major tcgen05 GEMM)
 *   merv_colsum    : out[n] = sum_m x[m, n]      (bias gradient), workspace merv_colsum_workspace(M, N) floats
 *   merv_gelu      : elementwise erf-GELU forward / backward (the training path keeps the pre-activations)
 *   merv_mix_backward : gradients of CrossAttentionAdapterLearnableQuery.forward (nn_utils.py:487-521) w.r.t. every
 *       V_e and Q / q_proj_weight / k_proj_weight / in_proj_bias; v_proj_weight and out_proj get none (the attention
 *       output is discarded in the reference as well).  weights = forward output (fp32), u = merv_fusion_query_vec.
 * ------------------------------------------------------------------------------------------------------- */
int merv_transpose(const void* x, void* y, int R, int C, int64_t ldx, int64_t ldy, int dtype, void* stream);
/* out = gelu(z) when dy == NULL, else out = dy * gelu'(z)  (exact erf GELU; MLP projectors in the training step) */
int merv_gelu(const void* z, const void* dy, void* out, int64_t n, int dtype, void* stream);
size_t merv_colsum_workspace(int M, int N);
int merv_colsum(const void* x, void* out, float* workspace, int M, int N, int64_t ld, int dtype, void* stream);
size_t merv_mix_backward_workspace(int B, int E, int T, int K, int embed);
int merv_mix_backward(const void* const* V, const void* dOut, const float* weights, const float* dweights_out,
                      const float* u, const void* Q, const void* Wq, const void* Wk, const void* in_proj_bias,
                      void* const* dV, void* dQ, void* dWq, void* dWk, void* dbias, float* workspace,
                      size_t workspace_floats, int B, int E, int T, int K, int embed, int dtype, void* stream);
/* merv_mix_backward for every configuration the forward (merv_scores_from_tokens_ex + merv_softmax_mix) supports; with
 * ds = softmax backward of (dw + dweights_out) as above:
 *   tokens[e] in {T, 1}: a single-token encoder (repeated to T tokens, nn_utils.py:502) gets dV_e [B, 1, K] = the sum over t of
 *       the T-token gradient rows, i.e. w_e sum_t dOut[b,t] + ds_e ubar, and dw_e = <sum_t dOut[b,t], V_e[b,0]>;
 *   u_token_stride == 0 (averagetoken=True, u [K]):   dV_e = w_e dOut + (ds_e / T) u,  du = sum_{b,e} ds_e (mean_t V_e + pe[e]), ubar = u;
 *       pe [E, K] (ldpe, `dtype`) or NULL: positional_embedding=True (nn_utils.py:510-511); then dpe[e] = (sum_b ds_e[b]) u, dpe [E, K];
 *   u_token_stride == K (averagetoken=False, nn_utils.py:514-518, u [T*K]): dV_e = w_e dOut[b,t] + ds_e u[t],
 *       du[t] = sum_{b,e} ds_e V_e[b,t] (length T*K, Wk / dWk are [embed, T*K]), ubar = sum_t u[t]; pe must be NULL.
 * Then dq, dWk, dWq, db_q, dQ from du as in merv_mix_backward.  Fixed-order reductions (bit-reproducible).  With every tokens[e] == T,
 * u_token_stride == 0 and pe == NULL it is merv_mix_backward (same kernels, bit-identical).  workspace: merv_mix_backward_ex_workspace
 * floats (B * K fewer suffice when every encoder has T tokens). */
size_t merv_mix_backward_ex_workspace(int B, int E, int T, int K, int embed, int64_t u_token_stride);
int merv_mix_backward_ex(const void* const* V, const int32_t* tokens, const void* dOut, const float* weights,
                         const float* dweights_out, const float* u, int64_t u_token_stride, const void* pe, int64_t ldpe,
                         const void* Q, const void* Wq, const void* Wk, const void* in_proj_bias, void* const* dV, void* dQ,
                         void* dWq, void* dWk, void* dbias, void* dpe, float* workspace, size_t workspace_floats, int B, int E,
                         int T, int K, int embed, int dtype, void* stream);
/* merv_mix_backward_ex reading dOut in place from a batch-strided slot: video b's rows start at dOut + b * dout_batch_stride, rows lddo
 * apart (the gradient of the prefix slot of the multimodal embedding buffer), in every pass that reads it; dV stays contiguous.  dOut
 * 16-byte aligned, lddo and dout_batch_stride whole 16-byte vectors (MERV_E_ALIGN), lddo >= K and dout_batch_stride >= T * lddo
 * (MERV_E_SHAPE).  merv_mix_backward_ex is this call with lddo = K, dout_batch_stride = T * K (the same kernels, bit-identical). */
int merv_mix_backward_strided(const void* const* V, const int32_t* tokens, const void* dOut, int64_t lddo, int64_t dout_batch_stride,
                              const float* weights, const float* dweights_out, const float* u, int64_t u_token_stride, const void* pe, int64_t ldpe,
                              const void* Q, const void* Wq, const void* Wk, const void* in_proj_bias, void* const* dV, void* dQ, void* dWq,
                              void* dWk, void* dbias, void* dpe, float* workspace, size_t workspace_floats, int B, int E, int T, int K, int embed,
                              int dtype, void* stream);
/* Gradients of ScalarAdapter.forward (feature_fusion == "scalar", nn_utils.py:524-537): w = softmax(scalar) [E] for every video,
 * out = sum_e w_e V_e, returned weights w[None].  With dweights_out [E] the gradient of the returned weights:
 *     dV_e = w_e dOut,   g_e = sum_b <dOut[b], V_e[b]> + dweights_out[e],   dscalar = w (.) (g - <w, g>)
 * V_e, dOut, dV_e [B, T, K] contiguous in `dtype` (the reference stacks the encoders, so all share one shape), weights fp32 [E],
 * dweights_out fp32 [E] or NULL, dscalar fp32 [E] out.  One pass reads dOut and every V_e once and writes every dV_e once; the dots
 * are reduced in a fixed order (bit-reproducible).  B == 0 reads no tensor: dscalar from dweights_out alone.
 * workspace: merv_scalar_mix_backward_workspace(B, E, K) floats. */
size_t merv_scalar_mix_backward_workspace(int B, int E, int K);
int merv_scalar_mix_backward(const void* const* V, const void* dOut, const float* weights, const float* dweights_out, void* const* dV,
                             float* dscalar, float* workspace, size_t workspace_floats, int B, int E, int T, int K, int dtype, void* stream);
/* merv_scalar_mix_backward with dOut read in place from a batch-strided slot (rows lddo apart, videos dout_batch_stride apart; checks as for
 * merv_mix_backward_strided); V_e and dV_e stay contiguous.  merv_scalar_mix_backward is this call with lddo = K, dout_batch_stride = T * K. */
int merv_scalar_mix_backward_strided(const void* const* V, const void* dOut, int64_t lddo, int64_t dout_batch_stride, const float* weights,
                                     const float* dweights_out, void* const* dV, float* dscalar, float* workspace, size_t workspace_floats, int B,
                                     int E, int T, int K, int dtype, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Backward of the FUSED path (linear projectors linked to the adapter, forward = merv_fused_linear_mix): the training step of
 * the shipped configs (merv/models/vidlms/merv.py:587-589,608 under base_strategy.py:210-241) without ever materialising the
 * per-encoder projections Y_e or their gradients dV_e.  With P_e the pooled tokens (kept from the forward), Z_e = dOut W_e:
 *     dw_e = <Z_e, P_e> + b_e . colsum_t(dOut)        ds = softmax backward of (dw + dweights_out)
 *     dW_e = dOut^T (w_e (.) P_e) + u (x) g_e          g_e = sum_b ds_e[b] mean_t P_e[b]
 *     db_e = sum_b w_e[b] colsum_t(dOut[b]) + u sum_b ds_e[b]          du = sum_e (W_e g_e + b_e sum_b ds_e[b])  ->  dQ, dWq, dWk, db_q
 * The two GEMMs per encoder (Z_e and dOut^T (w_e (.) P_e)) are merv_linear_bias_act calls; the entry points below are the rest:
 *   merv_video_colsum       out[b, k] = scale * sum_t x[b, t, k]  (fp32 [B, K]); x rows `ld` apart, videos `batch_stride` apart
 *   merv_pair_dot           partial[b, c] = chunk c of sum_i x[b, i] y[b, i], c < merv_pair_dot_chunks(); x, y [B, n] contiguous
 *   merv_transpose_rowscale y[c, r] = scale[(r / rows_per_scale) * scale_stride] * x[r, c] (scale NULL: 1); columns R..R_pad-1 of y are
 *                           zero-filled (K-major GEMM operands need R_pad % 8 == 0 in bf16)
 *   merv_fused_backward     everything after the GEMMs: ds, g_e, db_e, the rank-1 update of dW_e (in place), du and the adapter's
 *                           parameter gradients.  workspace: merv_fused_backward_workspace(desc) floats.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t B, E, K, embed;                 /* videos, encoders, llm_dim, text embedding dim */
  int32_t C[MERV_MAX_ENCODERS];           /* channels per encoder */
  const float* weights;                   /* [B, E] mixing weights of the forward (fp32) */
  const float* dweights_out;              /* [B, E] gradient w.r.t. the returned weights, or NULL */
  const float* u;                         /* [K] merv_fusion_query_vec */
  const float* gsum;                      /* [B, K] merv_video_colsum(dOut) */
  const float* dw_partial[MERV_MAX_ENCODERS]; /* [B, merv_pair_dot_chunks()] merv_pair_dot(Z_e, P_e) */
  const float* pbar[MERV_MAX_ENCODERS];   /* [B, C_e] merv_video_colsum(P_e, scale = 1 / T) */
  const void* W[MERV_MAX_ENCODERS];       /* [K, C_e] projector weights (`dtype`), row stride ldw */
  int64_t ldw[MERV_MAX_ENCODERS];
  const void* bias[MERV_MAX_ENCODERS];    /* [K] or NULL */
  const void *Q, *Wq, *Wk, *in_proj_bias; /* adapter parameters (`dtype`); in_proj_bias may be NULL */
  float* ds;                              /* out [B, E] */
  void* dW[MERV_MAX_ENCODERS];            /* in/out [K, C_e]: dOut^T (w_e (.) P_e) on entry, + u (x) g_e on exit */
  int64_t lddw[MERV_MAX_ENCODERS];
  void* db[MERV_MAX_ENCODERS];            /* out [K] or NULL */
  void *dQ, *dWq, *dWk, *dbias;           /* out [embed], [embed, embed], [embed, K], [3 * embed] */
  float* workspace;
  size_t workspace_floats;
} merv_fused_bwd_desc;
int merv_video_colsum(const void* x, float* out, int B, int T, int K, int64_t ld, int64_t batch_stride, float scale, int dtype,
                      void* stream);
int merv_pair_dot_chunks(void);
int merv_pair_dot(const void* x, const void* y, float* partial, int B, int64_t n, int dtype, void* stream);
/* merv_pair_dot that also writes y_scaled[b, i] = scale[b * scale_stride] * y[b, i] in the same pass: w_e (.) P_e, the MN-major
 * W-operand of dW_e = dOut^T (w_e (.) P_e) for merv_gemm_ex (no transposed copy of P_e, and P_e is read once for both). */
int merv_pair_dot_scale(const void* x, const void* y, float* partial, const float* scale, int64_t scale_stride, void* y_scaled,
                        int B, int64_t n, int dtype, void* stream);
int merv_transpose_rowscale(const void* x, void* y, int R, int R_pad, int C, int64_t ldx, int64_t ldy, const float* scale,
                            int64_t scale_stride, int rows_per_scale, int dtype, void* stream);
/* The weight gradient AND the mixing-weight gradient of one encoder from ONE pass over dOut and the pooled tokens (bf16, tcgen05):
 *     dW [N_out, C]  = sum_b scale[b * scale_stride] * dY[b]^T X[b]        (dW_e = dOut^T (w_e (.) P_e) without materialising w_e (.) P_e)
 *     dot_partial[b] = merv_pair_dot_chunks() partial sums of <W, dY[b]^T X[b]>   (= <dOut[b] W_e, P_e[b]>: the Z_e = dOut W_e GEMM and the
 *                      pair-dot pass of the formulation above are not needed at all — half of the backward's tensor work)
 * dY [videos * tokens_per_video, N_out] (lddy), X [videos * tokens_per_video, C] (ldx), W / dW [N_out, C] (ldw / lddw), all read in place
 * (MN-major operands); the contraction runs over the tokens, the accumulator is drained once per video: scaled into the running sum in
 * fp32 registers and dotted with the W tile.  tokens_per_video % 64 == 0.  When the tile count leaves SMs idle (96 - 128 tiles on 148 SMs
 * at the merv-full shapes) the videos are split into contiguous ranges handled as separate work items whose fp32 partial tiles are folded
 * in fixed order afterwards (deterministic).  workspace: merv_wgrad_video_workspace(videos, N_out, C) floats, 16-byte aligned. */
int merv_wgrad_video_parts(int N_out, int C);
size_t merv_wgrad_video_workspace(int videos, int N_out, int C);
int merv_wgrad_video(const void* dY, int64_t lddy, const void* X, int64_t ldx, const float* scale, int64_t scale_stride, const void* W,
                     int64_t ldw, void* dW, int64_t lddw, float* dot_partial, float* workspace, int videos, int tokens_per_video, int N_out,
                     int C, void* stream);
/* merv_wgrad_video with dY video b's rows at dY + b * dy_batch_stride (rows lddy apart): the gradient of the prefix slot of the multimodal
 * embedding buffer read in place by a 3-D TMA map (N_out columns, token in video, video).  dY 16-byte aligned, lddy and dy_batch_stride
 * multiples of 8 (MERV_E_ALIGN), dy_batch_stride >= tokens_per_video * lddy (MERV_E_SHAPE).  With dy_batch_stride = tokens_per_video * lddy
 * it is merv_wgrad_video (the same kernel, bit-identical); other strides run a separate instantiation doing the same reductions. */
int merv_wgrad_video_ex(const void* dY, int64_t lddy, int64_t dy_batch_stride, const void* X, int64_t ldx, const float* scale, int64_t scale_stride,
                        const void* W, int64_t ldw, void* dW, int64_t lddw, float* dot_partial, float* workspace, int videos, int tokens_per_video,
                        int N_out, int C, void* stream);
size_t merv_fused_backward_workspace(const merv_fused_bwd_desc* desc);
int merv_fused_backward(const merv_fused_bwd_desc* desc, int dtype, void* stream);
/* The same fused training step in front of the ScalarAdapter (one w [E] for every video, no query vector).  Per encoder,
 * merv_wgrad_video(dOut, P_e, scale = &w[e], scale_stride = 0, W_e) gives dW_e = w_e dOut^T P_e and dw_partial[e] = the partials of
 * <W_e, dOut[b]^T P_e[b]>; merv_video_colsum(dOut) gives gsum [B, K].  This finishes the step, all sums in a fixed order:
 *     gs = sum_b gsum[b],   db_e = w_e gs,   g_e = sum(dw_partial[e]) + b_e . gs + dweights_out[e],   dscalar = w (.) (g - <w, g>)
 * weights fp32 [E], dweights_out fp32 [E] or NULL, dw_partial[e] fp32 [B, merv_pair_dot_chunks()], bias[e] / db[e] [K] (`dtype`) or
 * NULL entries, dscalar fp32 [E] out.  workspace: merv_scalar_fused_backward_workspace(E, K) floats. */
size_t merv_scalar_fused_backward_workspace(int E, int K);
int merv_scalar_fused_backward(const float* weights, const float* dweights_out, const float* gsum, const float* const* dw_partial,
                               const void* const* bias, void* const* db, float* dscalar, float* workspace, size_t workspace_floats, int B,
                               int E, int K, int dtype, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Attentive pooler ("attntv" resampler: AttentivePooler.forward, merv/util/nn_utils.py:229-238; constructed at
 * merv/models/vidlms/merv.py:124-130).  Its LayerNorms, Linears and GELU are merv_layernorm / merv_linear_bias_act; these are the rest:
 *   merv_cross_attention  CrossAttention.forward (nn_utils.py:393-412) after the q / kv Linears:
 *         out[b, i, h*hd + d] = sum_k softmax_k(scale * q[b, i, h, :] . K[b, k, h, :]) V[b, k, h, d]
 *         q [n_q, heads * hd] rows `ldq` apart, batch entries `q_batch_stride` apart (0: the same learned queries for every entry);
 *         kv [batches * n_kv, 2 * heads * hd] rows `ldkv` apart: K in the first heads * hd columns, V in the last (nn_utils.py:398-399);
 *         out [batches * n_q, heads * hd] rows `ldo` apart.  fp32 softmax; head_dim <= 128, a multiple of 8 (bf16) / 4 (fp32).
 *   merv_add_rows         out[m, :] = a[m, :] + b[m % period, :]  — the residual adds of CrossAttentionBlock.forward (nn_utils.py:449-450);
 *         period = n_q adds the learned query tokens to every frame's attention output.
 * ------------------------------------------------------------------------------------------------------- */
int merv_cross_attention(const void* q, int64_t ldq, int64_t q_batch_stride, const void* kv, int64_t ldkv, void* out, int64_t ldo,
                         int batches, int n_q, int n_kv, int heads, int head_dim, float scale, int dtype, void* stream);
/* Backward of merv_cross_attention on the tensor cores (bf16; n_q <= 64, n_kv <= 256, head_dim % 32 == 0 and <= 128): S and P are
 * recomputed, dP = dO V^T, dS = scale P (.) (dP - rowsum(P (.) dP)), dV = P^T dO, dK = dS^T Q, dQ = dS K — five tcgen05 contractions per
 * (frame, head).  dout [batches, n_q, C] (lddo), dq [batches, n_q, C] (lddq): dQ of EVERY frame (with shared queries, q_batch_stride == 0,
 * the caller sums the frames), dkv [batches * n_kv, 2C] (lddkv) = [dK | dV] in the layout of kv.  Rows 16-byte aligned.
 * Same as merv_cross_attention_backward_ex(..., MERV_BF16, NULL, 0, stream): other shapes are rejected. */
int merv_cross_attention_backward(const void* q, int64_t ldq, int64_t q_batch_stride, const void* kv, int64_t ldkv, const void* dout,
                                  int64_t lddo, void* dq, int64_t lddq, void* dkv, int64_t lddkv, int batches, int n_q, int n_kv,
                                  int heads, int head_dim, float scale, void* stream);
/* The backward of merv_cross_attention on its whole domain: fp32 or bf16 (`dtype`), any n_q and n_kv, head_dim <= 128 and a multiple of
 * 8 (bf16) / 4 (fp32), shared or per-entry queries, rows 16-byte aligned; same operands and outputs as above.  bf16 inside the tcgen05
 * tile (n_q <= 64, n_kv <= 256, head_dim % 32 == 0) runs the tensor-core kernel, bit-identical to merv_cross_attention_backward;
 * everything else (and every shape under MERV_ATTN_IMPL=simt) runs a CUDA-core kernel: softmax statistics and D = rowsum(P (.) dP)
 * recomputed in a first sweep over the keys, then a keys-outer sweep; P and every sum in fp32, outputs rounded once; fixed-order
 * reductions, no atomics, so results are bit-reproducible and a frame's gradients do not depend on the other frames of the call.
 * workspace: merv_cross_attention_backward_ex_workspace(...) floats (0 when the tcgen05 kernel runs; workspace may then be NULL). */
size_t merv_cross_attention_backward_ex_workspace(int batches, int n_q, int n_kv, int heads, int head_dim, int dtype);
int merv_cross_attention_backward_ex(const void* q, int64_t ldq, int64_t q_batch_stride, const void* kv, int64_t ldkv, const void* dout,
                                     int64_t lddo, void* dq, int64_t lddq, void* dkv, int64_t lddkv, int batches, int n_q, int n_kv,
                                     int heads, int head_dim, float scale, int dtype, float* workspace, size_t workspace_floats,
                                     void* stream);
int merv_add_rows(const void* a, int64_t lda, const void* b, int64_t ldb, void* out, int64_t ldo, int64_t M, int C, int period, int dtype,
                  void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * LayerNorm over the channel dimension of (possibly segmented) rows: Y[m, :] = LN(concat_s X_s[m, :]) * gamma + beta.
 *   nseg == 1 : nn.LayerNorm(vision_dim) in front of a projector — `pre_proj_layernorm=True`
 *               (merv/util/nn_utils.py:26-29,41-44,67-70,91-94; merv/models/vidlms/merv.py:165-171)
 *   nseg == E : nn.LayerNorm(E * llm_dim) of feature_fusion == "concat_channel_ln" (merv.py:219-223) applied to the channel
 *               concatenation of merv.py:603-605, which is never materialised un-normalised.
 * X_s [M, K_s] (ldx[s]), gamma / beta [sum K_s] in `dtype` (either may be NULL), Y [M, sum K_s] (ldy).  Statistics in fp32,
 * biased variance, two passes over register-resident values.  sum K_s <= 32768 (bf16) / 16384 (fp32).
 * merv_layernorm_backward: dX = d/dX of the above (optional, [M, sum K_s]) and GX = dY * xhat (optional); the parameter
 * gradients are the column sums dgamma = merv_colsum(GX), dbeta = merv_colsum(dY).
 * ------------------------------------------------------------------------------------------------------- */
int merv_layernorm(const void* const* X, const int64_t* ldx, const int32_t* K, int nseg, const void* gamma, const void* beta,
                   float eps, void* Y, int64_t ldy, int M, int dtype, void* stream);
int merv_layernorm_backward(const void* const* X, const int64_t* ldx, const int32_t* K, int nseg, const void* dY, int64_t lddy,
                            const void* gamma, float eps, void* dX, int64_t lddx, void* GX, int64_t ldgx, int M, int dtype,
                            void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MERV_FUSION_H_ */
