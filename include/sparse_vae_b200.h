/*
 * sparse_vae_b200 -- C ABI of the B200-native hot path of norabelrose/sparse-vae.
 *
 * libsvae_b200.so exports exactly the entry points declared here: plain pointers, sizes and POD
 * descriptors, no torch / C++ types.  All device pointers are borrowed for the duration of the
 * stream-ordered launch; the caller (PyTorch on the host side) owns every buffer, output and scratch.
 * Every launch goes to the `stream` argument (a cudaStream_t passed as void*); no entry point
 * synchronises the device.  Functions return 0 on success and a negative SVAE_ERR_* otherwise;
 * svae_last_error() returns a thread-local, human-readable description of the last failure.
 *
 * Reference interfaces replaced (paths relative to the reference repository root):
 *   svae_layout_*      SparseAttention.get_master_layout            sparse_vae/core/sparse_attention.py:38-59
 *                      + LUT builders of the Triton ops             sparse_vae/core/sparse_matmul.py:133-144,251-326
 *   svae_attn_fwd      SparseAttention.__call__ = sdd->softmax->dsd sparse_vae/core/sparse_attention.py:75-92
 *                      (triton.ops.blocksparse.matmul / softmax, triton==1.1.0, requirements.txt:11)
 *   svae_attn_bwd      autograd of the above                        sparse_vae/core/sparse_matmul.py:463-488
 *   svae_bottleneck_*  ConditionalGaussian.forward                  sparse_vae/core/conditional_gaussian.py:18-30
 *                      + ContinuousVAE.sample_z                     sparse_vae/core/continuous_autoencoder.py:42-52
 *                      + torch.distributions.Normal.rsample (Philox stream of at::native normal_)
 *   svae_radam_step    RAdam.step                                   sparse_vae/core/rectified_adam.py:15-88
 *   svae_clip_grad_norm  LanguageModel.on_after_backward            sparse_vae/core/language_model.py:120-122
 * There is no CPU implementation behind this ABI: host pointers are rejected by the host-side wrappers
 * and the library needs an sm_100a device.
 */
#ifndef SPARSE_VAE_B200_H_
#define SPARSE_VAE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVAE_ABI_VERSION 1

#if defined(__GNUC__)
#define SVAE_API __attribute__((visibility("default")))
#else
#define SVAE_API
#endif

/* element types of q/k/v/out and of the bottleneck's mu|logvar input */
#define SVAE_DTYPE_F32  0   /* exact CUDA-core path (fp32 FFMA); parity mode, 1e-4 */
#define SVAE_DTYPE_BF16 1   /* tcgen05 / TMEM / TMA path */
#define SVAE_DTYPE_F16  2   /* tcgen05 / TMEM / TMA path */

#define SVAE_OK                0
#define SVAE_ERR_INVALID      -1   /* bad argument (shape, stride, dtype, alignment) */
#define SVAE_ERR_UNSUPPORTED  -2   /* valid request outside what the kernels implement */
#define SVAE_ERR_CUDA         -3   /* CUDA runtime / driver error, see svae_last_error() */
#define SVAE_ERR_DEVICE       -4   /* not an sm_100 device */

/* svae_attn_desc.flags */
#define SVAE_ATTN_FORCE_EXACT  1   /* run 16-bit inputs through the exact CUDA-core path (cross-check / debugging) */
#define SVAE_ATTN_BWD_TWO_PASS 4   /* backward: use the two-pass kernels even where the one-pass kernel applies (cross-check) */
#define SVAE_ATTN_PERSISTENT   2   /* forward: persistent warp-specialised kernel (what the host wrapper selects for <= 8 key slots;
                                      without the flag: one CTA per tile, also used for wider windows and score dumps) */

/* Block-sparse attention problem.  Tensors are [batch, heads, seq_len, head_dim] with arbitrary
 * batch/head/row strides (in ELEMENTS) and unit inner stride -- the reference hands the op strided
 * views of [B, L, H*Dh] (core/attention.py:76). */
typedef struct svae_attn_desc {
  int32_t batch, heads, seq_len, head_dim;
  int32_t dtype;          /* SVAE_DTYPE_* of q, k, v, out and the gradients */
  int32_t block_size;     /* must be 32 (SparseAttention.block_size) */
  int32_t window_size;    /* SparseAttention.window_size */
  int32_t causal;         /* SparseAttention.causal */
  int32_t include_cls;    /* SparseAttention.include_cls */
  int32_t flags;          /* SVAE_ATTN_* */
  float   scale;          /* softmax scale, reference: head_dim ** -0.5 */
  int32_t reserved;
  int64_t q_stride[3], k_stride[3], v_stride[3], o_stride[3];       /* {batch, head, row} */
  int64_t do_stride[3], dq_stride[3], dk_stride[3], dv_stride[3];   /* backward only */
} svae_attn_desc;

SVAE_API int svae_abi_version(void);
SVAE_API const char* svae_last_error(void);
/* 0 if the current CUDA device can run the kernels (compute capability 10.x), else SVAE_ERR_DEVICE */
SVAE_API int svae_device_check(void);

/* ---- measurement: per-kernel device time of every launch the library makes between begin and end, taken
 * with CUDA events on the launching stream.  svae_profile_end synchronises on the recorded events and writes a
 * JSON object {"<kernel>": {"launches": n, "ms": total}, ...} into buf. */
SVAE_API void svae_profile_begin(void);
SVAE_API int svae_profile_end(char* buf, size_t buf_bytes);

/* ---- layout (host only; bit-exact with get_master_layout()[..., :nb, :nb]) ------------------- */
/* non-zero blocks per head */
SVAE_API int64_t svae_layout_nnz(int32_t num_blocks, int32_t window_size, int32_t causal, int32_t include_cls);
/* Any output pointer may be NULL.  layout: [num_heads, nb, nb] int64 0/1.  row_ptr[nb+1] / col_idx[nnz]
 * enumerate each block-row's key blocks in `layout.nonzero()` order; colT_ptr[nb+1] / rowT_idx[nnz]
 * enumerate each key block's query block-rows (used by the dK/dV pass). */
SVAE_API int svae_layout_build(int32_t num_blocks, int32_t window_size, int32_t causal, int32_t include_cls,
                      int32_t num_heads, int64_t* layout, int32_t* row_ptr, int32_t* col_idx,
                      int32_t* colT_ptr, int32_t* rowT_idx);

/* ---- attention ------------------------------------------------------------------------------ */
/* out = softmax(scale * q k^T + key_padding_mask[b, key]; layout, causal) v, fused, S/P never reach HBM.
 * key_padding_mask: additive fp32 [batch, seq_len] (0 / -inf / -1e7 ...) or NULL.
 * lse: fp32 [batch, heads, seq_len] natural-log-sum-exp of every row (saved for backward). */
SVAE_API int svae_attn_fwd(const svae_attn_desc* desc, const void* q, const void* k, const void* v,
                  const float* key_padding_mask, void* out, float* lse, void* stream);

/* Which kernels svae_attn_bwd will run for this problem: the tcgen05 kernels need 16-bit tensors, head_dim 64 and
 * a band of <= 13 key blocks; everything else takes the exact CUDA-core kernels (20-40x slower; the host wrapper
 * warns when 16-bit tensors end up there).  < 0: invalid descriptor. */
#define SVAE_BWD_PATH_TCGEN05 0            /* one pass over the sequence (causal, window <= 4: the reference's default) */
#define SVAE_BWD_PATH_EXACT   1
#define SVAE_BWD_PATH_TCGEN05_TWO_PASS 2   /* dQ pass + dK/dV pass (non-causal layouts, windows 5..10) */
SVAE_API int svae_attn_bwd_path(const svae_attn_desc* desc);

SVAE_API size_t svae_attn_bwd_workspace_bytes(const svae_attn_desc* desc);
/* dq, dk, dv (same dtype as q) from dout; workspace: device scratch of at least
 * svae_attn_bwd_workspace_bytes(desc) bytes, 256-byte aligned, contents ignored on entry. */
SVAE_API int svae_attn_bwd(const svae_attn_desc* desc, const void* q, const void* k, const void* v,
                  const void* out, const void* dout, const float* lse, const float* key_padding_mask,
                  void* dq, void* dk, void* dv, void* workspace, size_t workspace_bytes, void* stream);

/* Test hook (no global state): variant of svae_attn_fwd for the tcgen05 path.  s_dump (may be NULL): raw scores S = q k^T (before
 * scale/masks) of every query row against its tile's key slots, [batch, heads, seq_len, slots*32] fp32
 * (slots = svae_attn_fwd_slots(desc)).  timeline must be NULL: the argument is kept for ABI compatibility, and a
 * non-NULL timeline returns SVAE_ERR_UNSUPPORTED. */
SVAE_API int svae_attn_fwd_slots(const svae_attn_desc* desc);
SVAE_API int svae_attn_fwd_debug(const svae_attn_desc* desc, const void* q, const void* k, const void* v,
                        const float* key_padding_mask, void* out, float* lse, float* s_dump,
                        long long* timeline, void* stream);


/* ---- latent bottleneck ---------------------------------------------------------------------- */
#define SVAE_BOTTLENECK_WORKSPACE_BYTES 8448
/* mulogvar: [rows, 2*latent] (dtype), mu = [:, :latent], logvar = [:, latent:], row stride `ld` elements.
 * token_counts: int64 [rows].  eps for element (row, d) is the value torch's CUDA `normal_` would write
 * to element row*latent + d of a [rows*latent] tensor of `dtype` with Philox (seed, offset) on a device
 * with `sm_count` SMs / `max_threads_per_sm` -- i.e. bit-identical to Normal(mu, sigma).rsample().
 * Outputs (fp32, contiguous): z[rows, latent], sigma[rows, latent], kl_elem[rows, latent] (may be NULL),
 * raw_kl[rows], kl[1] = mean(raw_kl / token_counts).  `workspace`: device scratch of
 * SVAE_BOTTLENECK_WORKSPACE_BYTES bytes, zero-filled ONCE by the caller before its first use; the kernel
 * leaves it zeroed again (deterministic two-level reduction of kl; no atomics on floating point). */
SVAE_API int svae_bottleneck_fwd(const void* mulogvar, int64_t ld, int32_t dtype, const int64_t* token_counts,
                        int64_t rows, int32_t latent, uint64_t philox_seed, uint64_t philox_offset,
                        int32_t sm_count, int32_t max_threads_per_sm,
                        float* z, float* sigma, float* kl_elem, float* raw_kl, float* kl,
                        void* workspace, void* stream);
/* Number the Philox offset must be advanced by after the call (ATen calc_execution_policy). */
SVAE_API uint64_t svae_bottleneck_philox_increment(int64_t rows, int32_t latent, int32_t sm_count,
                                          int32_t max_threads_per_sm);
/* d_mulogvar[rows, 2*latent] (dtype, row stride ld_out) from upstream gradients (any may be NULL = zero):
 * dz[rows, latent], dsigma[rows, latent], dkl_elem[rows, latent], draw_kl[rows] (fp32), dkl[1] (fp32, device).
 *   d mu     = dz + g mu                                 g = dkl_elem + draw_kl[row] + dkl / (rows * token_counts[row])
 *   d logvar = (dz eps + dsigma) sigma / 2 + g (exp(logvar) - 1) / 2
 * eps is regenerated from (seed, offset); nothing but mu|logvar is re-read. */
SVAE_API int svae_bottleneck_bwd(const void* mulogvar, int64_t ld, int32_t dtype, const int64_t* token_counts,
                        int64_t rows, int32_t latent, uint64_t philox_seed, uint64_t philox_offset,
                        int32_t sm_count, int32_t max_threads_per_sm,
                        const float* dz, const float* dsigma, const float* dkl_elem, const float* draw_kl,
                        const float* dkl, void* d_mulogvar, int64_t ld_out, void* stream);

/* ---- optimizer step of the data-parallel trainer (SURVEY 8f row 4) ------------------------------ */
/* Tensor lists are HOST arrays of n device pointers (fp32 tensors, contiguous) with numel[n] element counts. */
/* number of 65536-element chunks the list splits into = floats of `partials` svae_clip_grad_norm needs */
SVAE_API int64_t svae_multi_tensor_chunks(int32_t n, const int64_t* numel);
/* dst[i][:] = src[i][:] * scale for every tensor of the list: packs per-parameter gradients into the flat fp32
 * all-reduce buckets of the data-parallel trainer (and folds the 1/world_size averaging in). */
SVAE_API int svae_multi_tensor_scale_copy(int32_t n, void* const* dst, void* const* src, const int64_t* numel, float scale,
                                 void* stream);
/* dst[i] = (dst_dtype) src[i] over two equally shaped lists (src fp32): the autocast-dtype copies of the projection
 * weights for one training step, in a handful of launches.  dst_dtype: SVAE_DTYPE_BF16 or SVAE_DTYPE_F16. */
SVAE_API int svae_multi_tensor_cast(int32_t n, void* const* dst, void* const* src, const int64_t* numel, int32_t dst_dtype,
                           void* stream);
/* torch.nn.utils.clip_grad_norm_(params, max_norm) as called by LanguageModel.on_after_backward
 * (sparse_vae/core/language_model.py:120-122): norm_coef[0] = || all grads ||_2, norm_coef[1] =
 * min(1, max_norm / (norm + 1e-6)), every gradient multiplied in place by norm_coef[1].  Deterministic
 * (two-level fixed-order reduction through `partials`, device scratch of partials_len floats). */
SVAE_API int svae_clip_grad_norm(int32_t n, void* const* grads, const int64_t* numel, float max_norm, float* partials,
                        int64_t partials_len, float* norm_coef, void* stream);
/* One RAdam step (lamb=False) over all tensors, sparse_vae/core/rectified_adam.py:15-88: `step` is the
 * group's 1-indexed step counter, lr the group's current learning rate (before rectification).  Scalars are
 * doubles: the schedule is evaluated in double precision like the reference's Python arithmetic. */
SVAE_API int svae_radam_step(int32_t n, void* const* params, void* const* grads, void* const* exp_avg,
                    void* const* exp_avg_sq, const int64_t* numel, double lr, double beta1, double beta2, double eps,
                    double weight_decay, int64_t step, void* stream);

/* ---- dense attention of a few queries over a long key sequence (the Perceiver encoder's learned-query layers:
 * reference core/perceiver.py:16-50 -> core/attention.py:83-100; non-causal, additive key padding) ---- */
typedef struct svae_xattn_desc {
  int32_t batch, heads, num_queries, num_keys, head_dim;
  int32_t dtype;          /* SVAE_DTYPE_BF16 / SVAE_DTYPE_F16 */
  float   scale;          /* head_dim ** -0.5 */
  int32_t reserved;
  int64_t q_stride[3], k_stride[3], v_stride[3], o_stride[3];       /* {batch, head, row}, elements; unit inner stride */
  int64_t do_stride[3], dq_stride[3], dk_stride[3], dv_stride[3];   /* backward only */
} svae_xattn_desc;
/* 1 if the tcgen05 kernels apply: 16-bit tensors, head_dim 64, 1..128 queries (backward: <= 64) */
SVAE_API int svae_xattn_supported(const svae_xattn_desc* desc);
/* out[b,h,q,:] = softmax_k(scale * q k^T + key_padding_mask[b, k]) v ; lse: fp32 [batch, heads, num_queries] */
SVAE_API int svae_xattn_fwd(const svae_xattn_desc* desc, const void* q, const void* k, const void* v,
                   const float* key_padding_mask, void* out, float* lse, void* stream);
SVAE_API int svae_xattn_bwd(const svae_xattn_desc* desc, const void* q, const void* k, const void* v, const void* out,
                   const void* dout, const float* lse, const float* key_padding_mask, void* dq, void* dk, void* dv,
                   void* stream);

/* ---- CUDA-graph variants (core/graph_step.py): a captured training step is replayed with NEW random numbers and NEW
 * optimizer scalars each time, so these read them from device memory the host refreshes before every replay.
 * philox_dev -> {seed, base offset} (uint64[2]); the `offset` argument is then the launch's fixed increment over the base
 * (the position of this draw inside the step), exactly torch's own offset_intragraph scheme.  NULL = the plain call. */
SVAE_API int svae_bottleneck_fwd_g(const void* mulogvar, int64_t ld, int32_t dtype, const int64_t* token_counts, int64_t rows,
                          int32_t latent, uint64_t seed, uint64_t offset, const uint64_t* philox_dev, int32_t sm_count,
                          int32_t max_threads_per_sm, float* z, float* sigma, float* kl_elem, float* raw_kl, float* kl,
                          void* workspace, void* stream);
SVAE_API int svae_bottleneck_bwd_g(const void* mulogvar, int64_t ld, int32_t dtype, const int64_t* token_counts, int64_t rows,
                          int32_t latent, uint64_t seed, uint64_t offset, const uint64_t* philox_dev, int32_t sm_count,
                          int32_t max_threads_per_sm, const float* dz, const float* dsigma, const float* dkl_elem,
                          const float* draw_kl, const float* dkl, void* d_mulogvar, int64_t ld_out, void* stream);
SVAE_API int svae_residual_dropout_add_g(const float* x, const void* h, int32_t h_dtype, float* out, int64_t numel, float p,
                                uint64_t seed, uint64_t offset, const uint64_t* philox_dev, void* stream);
SVAE_API int svae_dropout_branch_grad_g(const float* g, void* dh, int32_t h_dtype, int64_t numel, float p, uint64_t seed,
                               uint64_t offset, const uint64_t* philox_dev, void* stream);
/* The scalars of one RAdam step as the opaque block svae_radam_step_g reads from DEVICE memory (args_dev): the host
 * evaluates them with svae_radam_args (same double-precision schedule as svae_radam_step) into a pinned buffer of
 * svae_radam_args_bytes() bytes and copies it to the device before the replay. */
SVAE_API int32_t svae_radam_args_bytes(void);
SVAE_API int svae_radam_args(double lr, double beta1, double beta2, double eps, double weight_decay, int64_t step, void* args_out);
SVAE_API int svae_radam_step_g(int32_t n, void* const* params, void* const* grads, void* const* exp_avg, void* const* exp_avg_sq,
                      const int64_t* numel, const void* args_dev, void* stream);

/* ---- LayerNorm of the pre-LN decoder blocks (SURVEY 2.1 #11; reference core/transformer_layer.py:17-24) ---- */
/* x: [rows, n] contiguous (x_dtype), n in {128, 256, 512, 1024}; gamma/beta fp32 [n] (beta may be NULL).
 * y = (x - mean) * rstd * gamma + beta written in y_dtype (fp32 statistics; a 16-bit y equals the rounded fp32
 * result, i.e. what autocast's cast in front of the consuming Linear produces); mean, rstd: fp32 [rows]. */
SVAE_API int svae_layernorm_supported(int32_t n);
SVAE_API int svae_layernorm_fwd(const void* x, int32_t x_dtype, const float* gamma, const float* beta, int64_t rows,
                       int32_t n, float eps, void* y, int32_t y_dtype, float* mean, float* rstd, void* stream);
SVAE_API int64_t svae_layernorm_bwd_workspace_floats(int64_t rows, int32_t n);
/* dx (x_dtype, may be NULL), dgamma / dbeta (fp32 [n], may be NULL) from dy (y_dtype) in ONE pass over x and dy;
 * dx_residual (x_dtype, may be NULL; may equal dx) is added to dx: the gradient that reaches x through the residual
 * connection around the norm (core/transformer_layer.py:35-61), saving autograd's separate accumulation pass;
 * dx_low (y_dtype, may be NULL) receives the same dx rounded to y_dtype -- the gradient of a 16-bit branch that was
 * added to the stream right before this norm (svae_residual_layernorm);
 * workspace: device scratch of svae_layernorm_bwd_workspace_floats(rows, n) floats (deterministic two-level sum). */
SVAE_API int svae_layernorm_bwd(const void* dy, int32_t y_dtype, const void* x, int32_t x_dtype, const float* gamma,
                       const float* mean, const float* rstd, int64_t rows, int32_t n, void* dx, const void* dx_residual,
                       void* dx_low, float* dgamma, float* dbeta, float* workspace, int64_t workspace_floats,
                       void* stream);

/* ---- vocabulary cross-entropy (SURVEY 8f row 2; reference core/language_model.py:98-113,161-170) ---- */
/* logits: [rows, vocab] (dtype), row stride ld elements, vocab = 8192*k (k <= 4).  nll[r] = logsumexp(row) -
 * row[labels[r]] (fp32); if write_grad & 1, the row is overwritten with weight[r] * (softmax(row) - onehot(labels[r]))
 * (write_grad & 2, 16-bit logits: the one-row-per-CTA kernel instead of the streamed one -- a cross-check for tests).
 * weight[r] == 0 marks an ignored row (nll 0, zero gradient).  One read + one write of the logits. */
SVAE_API int svae_vocab_ce_supported(int32_t vocab);
SVAE_API int svae_vocab_ce(void* logits, int32_t dtype, int64_t rows, int32_t vocab, int64_t ld, const int64_t* labels,
                  const float* weight, float* nll, int32_t write_grad, void* stream);

/* ---- per-token log-likelihood under the vocabulary head, logits never materialised (reference
 *      core/continuous_autoencoder.py:62-88 estimate_log_prob_iw / p_of_x_given_z) ---- */
/* h: [rows, d], w: [vocab, d], bias: [vocab] or NULL -- all `dtype` (bf16 / fp16), row strides ldh / ldw elements
 * (multiples of 8, 16-byte aligned); vocab = 256*k, d = 64*k <= 512.  logit = round_dtype(h . w[c] + bias[c]) with fp32
 * accumulation (what the library GEMM returns), logp[r] = logit[r, labels[r]] - logsumexp_c logit[r, c] in fp32, and
 * logp[r] = 0 where labels[r] == 0 (column 0 still counts in the normaliser).  One tcgen05 GEMM with a running
 * log-sum-exp in its epilogue; deterministic (fixed combination order, no atomics). */
SVAE_API int svae_vocab_logprob_supported(int32_t vocab, int32_t d, int32_t dtype);
SVAE_API int svae_vocab_logprob(const void* h, int64_t ldh, const void* w, int64_t ldw, const void* bias, int32_t dtype,
                       int64_t rows, int32_t vocab, int32_t d, const int64_t* labels, float* logp, void* stream);

/* ---- bias gradient of the decoder blocks' nn.Linear layers (reference core/attention.py:33-39, ------
 *      core/transformer_layer.py:20-24): out[c] = sum_r x[r, c], fp32 accumulation, deterministic two-stage sum. */
/* x: [rows, n] (dtype), row stride ld elements, n % 8 == 0; out: fp32 [n];
 * workspace: device scratch of svae_colsum_workspace_floats(rows, n) floats.
 * counters: NULL (two launches) or svae_colsum_counters(n) device uint32 that are ZERO on entry; they are zero again
 * when the launch has run, so one array can be reused by consecutive calls on ONE stream (not by concurrent ones):
 * the last block of each column group sums the partial results, in a fixed order, inside the same launch. */
SVAE_API int64_t svae_colsum_workspace_floats(int64_t rows, int32_t n);
SVAE_API int32_t svae_colsum_counters(int32_t n);
SVAE_API int svae_colsum(const void* x, int32_t dtype, int64_t rows, int32_t n, int64_t ld, float* out, float* workspace,
                int64_t workspace_floats, uint32_t* counters, void* stream);

/* ---- weight gradient of the token embedding (reference core/transformer_language_model.py:47-53) ---- */
/* grad: [n, d] contiguous (dtype); perm: the positions 0..n-1 ordered by token id, equal ids in position order (the
 * indices of `torch.sort(ids, stable=True)`); bounds: int64 [vocab + 1], bounds[v] = first index of token v in that order
 * (`torch.searchsorted(sorted_ids, arange(vocab + 1))`); dweight: fp32 [vocab, d], every row written (zeros for absent
 * tokens).  Row v = sum of grad[perm[j]], bounds[v] <= j < bounds[v + 1], in that order: bit-deterministic, no atomics. */
SVAE_API int svae_embedding_bwd(const void* grad, int32_t dtype, const int64_t* bounds, const int64_t* perm, int64_t n,
                       int32_t vocab, int32_t d, float* dweight, void* stream);

/* ---- erf-GELU of the feed-forward blocks (reference core/transformer_layer.py:20-24: nn.GELU() between the two
 *      ffn projections; core/transformer_language_model.py:58 output_layer) ---- */
/* x, y, dy, dx: [rows, n] contiguous 16-bit (dtype), n % 8 == 0, 16-byte aligned.  y = x * Phi(x); dx = dy * (Phi(x) +
 * x * phi(x)), dx may alias dy.  colsum (optional, fp32 [n]): column sums of dx before its 16-bit rounding -- the bias gradient of the
 * projection that feeds the GELU -- from the same pass; needs `workspace` (svae_gelu_bwd_workspace_floats(rows, n)
 * floats) and svae_gelu_bwd_counters(n) device uint32 that are ZERO on entry and zero again afterwards (see
 * svae_colsum).  Deterministic.  Phi is evaluated as 2^-(1 + a Q(a)): |error| <= 2e-6 absolute, 7e-6 relative in the tail. */
SVAE_API int32_t svae_gelu_supported(int32_t dtype, int64_t rows, int32_t n);
SVAE_API int svae_gelu_fwd(const void* x, void* y, int32_t dtype, int64_t rows, int32_t n, void* stream);
SVAE_API int64_t svae_gelu_bwd_workspace_floats(int64_t rows, int32_t n);
SVAE_API int32_t svae_gelu_bwd_counters(int32_t n);
SVAE_API int svae_gelu_bwd(const void* dy, const void* x, void* dx, int32_t dtype, int64_t rows, int32_t n, float* colsum,
                  float* workspace, int64_t workspace_floats, uint32_t* counters, void* stream);

/* ---- rotary position encoding of q / k (SURVEY 8f row 1; reference core/attention.py:194-208) ---- */
/* x, out: [rows, d_model] contiguous (dtype), row r sits at position r % seq_len; cos / sin tables: [seq_len,
 * d_model/2] (table_dtype) built by the caller with the reference's own ops.  Pairs (2i, 2i+1) are rotated.
 * table_dtype == dtype: one rounding per product and per sum in `dtype` (the reference outside autocast).
 * table_dtype == F32 with a 16-bit dtype: the reference under autocast (fp32 cos/sin, promoted products): forward
 * in fp32 rounded once to `dtype`, backward with each product cast to `dtype` before the sum.
 * conj != 0 rotates by the negative angle (= the backward pass).  x == out is allowed. */
SVAE_API int svae_rotary(const void* x, const void* cos_table, const void* sin_table, void* out, int32_t dtype,
                int32_t table_dtype, int64_t rows, int32_t seq_len, int32_t d_model, int32_t conj, void* stream);

/* q and k of one attention layer in ONE launch (same tables), each rotated exactly like svae_rotary; sum_a / sum_b
 * (both or neither; fp32 [d_model]): column sums of the two outputs, bit-identical to svae_colsum of them -- the bias
 * gradients of the q / k projections when the launch is the backward rotation (conj = 1) of dq / dk.  workspace:
 * svae_rotary_pair_workspace_floats(rows, d_model) floats; counters: svae_colsum_counters(d_model) ZEROED device
 * uint32, zero again afterwards.  in_ld / out_ld: row strides (elements, >= d_model, multiples of 8) of the inputs /
 * outputs, so q and k may be column slices of one [rows, 3 d_model] projection output or gradient buffer.  xa may equal
 * oa (in place, in_ld == out_ld), likewise xb / ob. */
SVAE_API int64_t svae_rotary_pair_workspace_floats(int64_t rows, int32_t d_model);
SVAE_API int svae_rotary_pair(const void* xa, const void* xb, const void* cos_table, const void* sin_table, void* oa, void* ob,
                     int32_t dtype, int32_t table_dtype, int64_t rows, int32_t seq_len, int32_t d_model, int32_t conj,
                     int64_t in_ld, int64_t out_ld, float* sum_a, float* sum_b, float* workspace, int64_t workspace_floats,
                     uint32_t* counters, void* stream);

/* ---- token-by-token decoding (SURVEY 8f row 3) ----------------------------------------------------------------
 * One sparse-attention layer's step of TransformerVAE.sample (reference transformer_vae.py:112-126 ->
 * core/attention.py:60-100 with the KV cache of :107-142): rotary position encoding of the new q / k rows at the
 * position read from the DEVICE counter `position` (so the call can be replayed inside a CUDA graph), append of
 * k / v to the caches, and attention of the new query over the visible keys.
 *   q, k, v               [B, H*head_dim] `dtype`, `in_stride` elements between samples (slices of one fused
 *                         [B, 3*H*head_dim] projection are fine); out [B, H*head_dim] contiguous
 *   cos_table, sin_table  [table_rows, H*head_dim/2] fp32, row p = position p (positions >= table_rows clamp)
 *   key_cache, value_cache[B, (window+1)*block, H*head_dim] `dtype`: slots [0, block) = positions 0..block-1, the
 *                         rest a ring over later positions; identical to the reference's cache while
 *                         position < (window+1)*block, so the first tokens may be decoded by the ATen path.
 * Visible keys = block 0 and key blocks max(1, b-window+1)..b of the current block b = position / block, i.e.
 * the causal include_cls rows of svae_layout_build. */
SVAE_API int svae_decode_attn_supported(int32_t head_dim, int32_t window, int32_t block);
SVAE_API int svae_decode_attn(const void* q, const void* k, const void* v, const float* cos_table,
                     const float* sin_table, void* key_cache, void* value_cache, void* out,
                     const int32_t* position, int32_t B, int32_t H, int32_t head_dim, int32_t window, int32_t block,
                     int32_t table_rows, int64_t in_stride, int32_t dtype, float scale, void* stream);

/* The same step for a DENSE causal attention layer (reference core/attention.py:107-142 with `cfg is None`): rotary
 * of the new q / k rows at the DEVICE counter `position` (same arithmetic and tables as svae_decode_attn), append of
 * k / v at slot `position`, and attention of the new query over slots 0..position (fp32 softmax and accumulation).
 *   q, k, v, out, cos_table, sin_table  as for svae_decode_attn
 *   key_cache, value_cache [B, cache_len, H*head_dim] `dtype`: slot p holds position p (the reference's cache), so the
 *                         first tokens may be decoded by the ATen path.
 *   workspace             svae_decode_attn_dense_workspace_bytes(B, H, head_dim, cache_len) bytes, 16-byte aligned
 *                         (may be null when that is 0); holds the per-split partial results.
 * Split-KV: the live slots are dealt out to a number of CTAs per (sample, head) fixed by B, H and cache_len, and their
 * partial softmax results are merged in a fixed order (no atomics): bit-identical from run to run, graph-capturable.
 * position >= cache_len reads and writes nothing.  head_dim 32 | 64, cache_len 1..65536. */
SVAE_API int svae_decode_attn_dense_supported(int32_t head_dim, int32_t cache_len);
SVAE_API size_t svae_decode_attn_dense_workspace_bytes(int32_t B, int32_t H, int32_t head_dim, int32_t cache_len);
SVAE_API int svae_decode_attn_dense(const void* q, const void* k, const void* v, const float* cos_table,
                           const float* sin_table, void* key_cache, void* value_cache, void* out,
                           const int32_t* position, void* workspace, size_t workspace_bytes, int32_t B, int32_t H,
                           int32_t head_dim, int32_t cache_len, int32_t table_rows, int64_t in_stride, int32_t dtype,
                           float scale, void* stream);

/* Residual-stream update under autocast (reference core/transformer_layer.py:41,49,61 `x = x + h`): out = x + h with
 * x, out fp32 and h 16-bit, numel % 8 == 0, 16-byte aligned; out == x is allowed. */
SVAE_API int svae_residual_add(const float* x, const void* h, int32_t h_dtype, float* out, int64_t numel, void* stream);

/* The same with dropout on the branch (training mode of core/transformer_layer.py:61 `x + self.dropout(ffn(...))`):
 * out = x + dropout_p(h), h scaled by 1/(1-p) and rounded to its dtype where kept.  The keep mask is a pure function of
 * (seed, offset, element index) -- Philox4x32-10 -- and is regenerated, not stored, by svae_dropout_branch_grad:
 * dh = dtype(dtype(g) / (1-p)) where kept, 0 elsewhere.  The caller advances its generator offset by 4 per launch. */
SVAE_API int svae_residual_dropout_add(const float* x, const void* h, int32_t h_dtype, float* out, int64_t numel, float p,
                              uint64_t seed, uint64_t offset, void* stream);
SVAE_API int svae_dropout_branch_grad(const float* g, void* dh, int32_t h_dtype, int64_t numel, float p, uint64_t seed,
                             uint64_t offset, void* stream);

/* x_out = x + h (fp32 stream + branch), then y = LayerNorm(x_out) with the arithmetic of svae_layernorm_fwd (reference
 * core/transformer_layer.py:35-61: `x = x + h` followed by the next sub-layer's norm).  x_out == x updates the stream
 * in place (token-by-token decoding); training passes a new buffer and mean / rstd [rows] for the backward pass. */
SVAE_API int svae_residual_layernorm(const float* x, const void* h, int32_t h_dtype, const float* gamma, const float* beta,
                            int64_t rows, int32_t n, float eps, void* y, int32_t y_dtype, float* x_out, float* mean,
                            float* rstd, void* stream);

/* One-launch restatement of GenerationState.process_logits with its default settings (reference
 * core/generation.py:40-72): repetition penalty over the last `penalty_window` generated tokens, temperature, nucleus
 * filtering (largest set of most likely tokens with mass <= top_p, never empty), one categorical draw per row by
 * inverse CDF from uniforms[b] in [0, 1), then the bookkeeping of :66-71: ids[b, *column] = token if alive[b];
 * alive[b] cleared and *finished incremented when the token is end_token.
 *   logits [B, vocab] 16-bit, contiguous (not modified); ids [B, ids_stride] int64; column: device scalar. */
SVAE_API int svae_sample_top_p_supported(int32_t vocab, int32_t dtype);
SVAE_API int svae_sample_top_p(const void* logits, int32_t dtype, int32_t B, int32_t vocab, int64_t* ids, int64_t ids_stride,
                      const int64_t* column, const float* uniforms, uint8_t* alive, int32_t* finished,
                      int32_t penalty_window, float repetition_penalty, float temperature, float top_p,
                      int64_t end_token, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* SPARSE_VAE_B200_H_ */
