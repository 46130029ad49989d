/*
 * l32_ffn.h -- C ABI of the B200-native (sm_100a) Add-RMSNorm + SwiGLU feed-forward hot path.
 *
 * This is the drop-in boundary for the LLaMA-3.2 text-decoder block's hot path of
 * emmanuelalo52/LLaMA-3.2-Multimodal.  Every entry point cites the reference interface it replaces
 * (paths relative to the reference repository root).  The Python extension modules `rmsnorm` and
 * `swiglu_fused` (same names as the reference's setup.py:11-41 targets) bind these symbols; see
 * INTEGRATION.md for the binding a maintainer of the reference would add.
 *
 * Conventions
 *   - All pointers are DEVICE pointers unless stated otherwise; tensors are row-major and contiguous
 *     along the last dimension.  `dtype` is L32_DTYPE_BF16 or L32_DTYPE_FP16 (storage type of every
 *     activation / weight / gradient); all arithmetic accumulates in fp32.
 *   - `stream` is a cudaStream_t passed as void*; kernels are enqueued asynchronously, nothing
 *     synchronises, nothing allocates (CUDA-graph capturable).  Scratch memory is caller-provided.
 *   - Return value: 0 on success, negative L32_ERR_* for argument errors, positive = cudaError_t.
 *   - Inputs are borrowed; outputs are written in place into caller-owned buffers.
 *   - Weight layout is the Python/HF one: w_gate, w_up are [inter, hidden]; w_down is [hidden, inter]
 *     (reference Tools/swiglu/FusedSwiglu.py:63-64, Model/model.py:214).
 *   - WEIGHTS MUST BE FINAL BEFORE THE PREVIOUS KERNEL OF THE STREAM STARTS.  Every kernel here is launched with
 *     programmatic dependent launch and prefetches its weight operands (norm weight, w_gate / w_up / w_down, LoRA
 *     matrices) BEFORE it waits for the preceding kernel of the stream; only activations / gradients are read after that
 *     wait.  A weight that is itself produced on the same stream (a dtype cast, an optimiser step, an l32_gemm output
 *     used as a weight) must therefore be separated from its consumer by at least one other kernel or event -- the
 *     Python layer (ops.py) caches cast / contiguous weight copies so that it never launches such a producer itself.
 */
#ifndef L32_FFN_H_
#define L32_FFN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define L32_API __attribute__((visibility("default")))
#else
#define L32_API
#endif

#define L32_DTYPE_BF16 0
#define L32_DTYPE_FP16 1

#define L32_OK 0
#define L32_ERR_BAD_DTYPE (-1)
#define L32_ERR_BAD_SHAPE (-2)
#define L32_ERR_BAD_ALIGN (-3)
#define L32_ERR_NULL (-4)
#define L32_ERR_DRIVER (-5)
#define L32_ERR_WORKSPACE (-6)
#define L32_ERR_NOT_RESIDENT (-7)

/* ABI version of this header (bumped on any signature change).  2: tensor-parallel, LoRA and block-tail entry points.
 * 3: tensor-parallel backward; the all-gather entry points accept an A buffer distinct from the published one;
 *    l32_rmsnorm_backward_add, l32_block_tail_forward_ex, l32_linear_lora_forward / _backward, l32_lm_head_ce_*,
 *    l32_rope_kv_append, l32_gqa_attention_forward; later, additively: l32_gqa_attention_forward_train / _backward, and
 *    the tensor-parallel attention GEMMs l32_tp_linear_group_forward_allgather, l32_tp_linear_forward_allgather and
 *    l32_tp_linear_group_backward_dx_reduce_scatter, the paged KV cache l32_rope_kv_append_paged and
 *    l32_gqa_attention_forward_paged, its cascade decode l32_gqa_attention_forward_paged_cascade, next-token
 *    sampling l32_sample_tokens, and speculative decoding l32_gqa_attention_forward_paged_verify,
 *    l32_gqa_attention_verify_workspace_bytes, l32_ngram_draft_paged and l32_speculative_accept. */
L32_API int l32_abi_version(void);
/* Number of CUDA kernels this library has launched in the calling process so far (monotonic). */
L32_API unsigned long long l32_kernel_launch_count(void);
/* Human-readable text for a return code of this library (static storage). */
L32_API const char* l32_error_string(int code);

/* ---------------------------------------------------------------------------------------------
 * Fused residual Add-RMSNorm forward.
 *   h = x + residual (fp32, residual may be NULL);  y = h * rsqrt(mean(h^2) + eps) * weight
 * Replaces: rmsnorm_forward, Tools/rmsnorm/rmsnorm.cu:7-32 (kernel Tools/rmsnorm/rmsnorm.cuh:13-108),
 *           i.e. python `rmsnorm.forward(input, weight, residual, eps) -> [output, rms]`;
 *           module-level spec LLAMARMSNorm.forward, Model/model.py:164-171.
 *   x, residual, y, h_out : [rows, hidden]      weight : [hidden]      rms : [rows] fp32
 *   h_out   : optional; receives h rounded to `dtype` (saved for backward).  May alias `residual`
 *             (that reproduces the reference kernel's in-place `residual := x + residual`).
 *   rms     : optional; receives sqrt(mean(h^2) + eps)  (the reference returns rms, not rstd).
 */
L32_API int l32_add_rmsnorm_forward(const void* x, const void* residual, const void* weight, void* y, void* h_out,
                            float* rms, int64_t rows, int hidden, float eps, int dtype, void* stream);

/* RMSNorm backward.
 *   dx = rstd * (dy*w - xhat * mean(dy*w*xhat)),  xhat = h * rstd,  rstd = 1 / rms
 *   dweight[c] = sum_rows dy * xhat            (fp32 accumulation, deterministic two-stage reduction)
 * Replaces: rmsnorm_backward, Tools/rmsnorm/rmsnorm.cu:35-61 (kernel rmsnorm.cuh:110-154),
 *           python `rmsnorm.backward(grad_out, input, weight, rms) -> [d_input, d_weight]`, with
 *           `h` = the NORMALISED INPUT x + residual (the reference wrapper wrongly passes pre-add x,
 *           Model/model.py:144).  d_residual == dx.
 *   workspace : l32_rmsnorm_backward_workspace_bytes(rows, hidden) bytes, 16-byte aligned.
 *   dweight   : optional [hidden] in `dtype`.
 */
L32_API size_t l32_rmsnorm_backward_workspace_bytes(int64_t rows, int hidden);
L32_API int l32_rmsnorm_backward(const void* dy, const void* h, const void* weight, const float* rms, void* dx,
                         void* dweight, void* workspace, size_t workspace_bytes, int64_t rows, int hidden,
                         int dtype, void* stream);
/* Same, with dx = (norm backward) + addend: `addend` [rows, hidden] is a gradient that reaches the same tensor around the
 * norm -- the "+ attn_out" of the block tail (Model/model.py:273) -- added in the store pass instead of a separate kernel.
 *   dx_plain : optional [rows, hidden]; receives the norm backward WITHOUT the addend (the residual's gradient when the
 *              residual and the normalised input's other summand need different gradients, Model/model.py:271-273). */
L32_API int l32_rmsnorm_backward_add(const void* dy, const void* h, const void* weight, const float* rms, const void* addend,
                                     void* dx, void* dx_plain, void* dweight, void* workspace, size_t workspace_bytes,
                                     int64_t rows, int hidden, int dtype, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SwiGLU forward: act = silu(x w_gate^T + b_gate) * (x w_up^T + b_up)
 * Replaces: swiglu_forward_cuda, Tools/swiglu/swiglu.cu:277-316 (python `swiglu_fused.forward`,
 *           Tools/swiglu/swiglu_binding.cpp:7-12); math spec = the PyTorch path
 *           Tools/swiglu/FusedSwiglu.py:18-20.
 *   x : [tokens, hidden]   w_gate, w_up : [inter, hidden]   b_gate, b_up : optional [inter]
 *   act : [tokens, inter]  gate_cache, up_cache : optional [tokens, inter] (both or neither; the
 *   pre-activation gate / up projections, needed by l32_swiglu_backward).
 * One tcgen05 kernel: the gate/up accumulators live in TMEM and SiLU*mul is applied in the epilogue,
 * so gate and up never touch HBM unless the caches are requested.  tokens <= 128 takes the
 * weight-streaming small-M kernel (weights as the UMMA M operand, cluster split-K; same fused epilogue).
 */
L32_API int l32_swiglu_forward(const void* x, const void* w_gate, const void* w_up, const void* b_gate,
                       const void* b_up, void* act, void* gate_cache, void* up_cache, int64_t tokens,
                       int hidden, int inter, int dtype, void* stream);

/* SwiGLU backward (SiLU and SiLU' recomputed in registers from the gate cache).
 * Replaces: swiglu_backward_cuda, declared Tools/swiglu/swiglu.cuh:18-25 and bound at
 *           swiglu_binding.cpp:15-21 but never defined in the reference (kernel sketch swiglu.cu:179-223).
 *   d_act : [tokens, inter]  ->  dx : [tokens, hidden] (optional), dw_gate, dw_up : [inter, hidden]
 *   (optional, both or neither).
 *   workspace : l32_swiglu_backward_workspace_bytes(tokens, inter) bytes (holds d_gate, d_up).
 */
L32_API size_t l32_swiglu_backward_workspace_bytes(int64_t tokens, int inter);
L32_API int l32_swiglu_backward(const void* d_act, const void* x, const void* w_gate, const void* w_up,
                        const void* gate_cache, const void* up_cache, void* dx, void* dw_gate, void* dw_up,
                        void* workspace, size_t workspace_bytes, int64_t tokens, int hidden, int inter,
                        int dtype, void* stream);

/* Linear forward y = a w^T + bias, w : [out_features, in_features] (nn.Linear layout).
 * Replaces: the w_down nn.Linear call of FusedFeedforward.forward, Model/model.py:214-217. */
L32_API int l32_linear_forward(const void* a, const void* w, const void* bias, void* y, int64_t tokens, int in_features,
                       int out_features, int dtype, void* stream);

/* Up to three projections of the SAME activations, y_i = a w_i^T (no bias), as one launch: the W_query / W_key / W_value
 * calls of GroupQueryAttention.forward (Model/model.py:231-233; three nn.Linear calls in the reference).  tokens <= 128: the
 * weight-streaming kernel walks the row blocks of all weights in one grid (one launch ramp and one tail instead of three);
 * otherwise one grouped tcgen05 GEMM launch whose problems share the persistent tile loop.
 *   w, y, out_features : arrays of `count` (1..3) entries; w[i] : [out_features[i], in_features], y[i] : [tokens, out_features[i]]. */
L32_API int l32_linear_group_forward(const void* a, const void* const* w, void* const* y, const int* out_features, int count,
                             int64_t tokens, int in_features, int dtype, void* stream);

/* Whole feed-forward forward: y = (silu(x w_gate^T) * (x w_up^T)) w_down^T.
 * Replaces: swiglu_down_forward_cuda, Tools/swiglu/swiglu.cu:319-364 (python `swiglu_fused.forward_down`,
 *           swiglu_binding.cpp:24-31); module-level spec FusedFeedforward.forward, Model/model.py:216-217.
 *   act_ws : [tokens, inter] scratch in `dtype` (the intermediate; L2/HBM resident between the two GEMMs).
 *   gate_cache / up_cache : optional, as in l32_swiglu_forward.
 */
L32_API int l32_ffn_forward(const void* x, const void* w_gate, const void* w_up, const void* w_down, const void* b_gate,
                    const void* b_up, const void* b_down, void* y, void* act_ws, void* gate_cache, void* up_cache,
                    int64_t tokens, int hidden, int inter, int dtype, void* stream);

/* Tail of the decoder block in one call: normed = rmsnorm(attn_out + residual) * norm_weight;
 * out = attn_out + ff(normed)   -- the "+ attn_out" rides in the epilogue of the down GEMM.
 * Replaces: TransformerBlock.forward lines norm2 / ff / return, Model/model.py:270-273 (three module calls and one
 *           elementwise add in the reference).  The reference drops `residual` from the block output (SURVEY.md
 *           section 0.6); so does this.  Inference only (no caches).  The sum is formed the way the reference's
 *           16-bit path forms it: ff_out rounded to `dtype`, then added to attn_out and rounded again.
 *   normed_ws : [tokens, hidden] scratch;  act_ws : [tokens, inter] scratch;  out may NOT alias attn_out.
 */
L32_API int l32_block_tail_forward(const void* attn_out, const void* residual, const void* norm_weight, float eps,
                                   const void* w_gate, const void* w_up, const void* w_down, void* out, void* normed_ws,
                                   void* act_ws, int64_t tokens, int hidden, int inter, int dtype, void* stream);

/* The same with everything a training step and the NEXT block need (every extra pointer optional):
 *   h_out, rms_out          : attn_out + residual (rounded to `dtype`; only written when residual != NULL) and the row
 *                             statistic sqrt(mean(h^2) + eps) -- the operands of l32_rmsnorm_backward(_add);
 *   gate_cache, up_cache    : both or neither, the operands of l32_ffn_backward;
 *   next_norm_weight (+ next_eps, next_normed, next_rms): when given, the sum `out` is normalised once more with that weight
 *                             -- the next block's norm1, or final_norm after the last block (Model/model.py:267, :346) --
 *                             in the same call, while `out` is still L2-resident, so the next block starts from next_normed.
 */
L32_API int l32_block_tail_forward_ex(const void* attn_out, const void* residual, const void* norm_weight, float eps,
                                      const void* w_gate, const void* w_up, const void* w_down, void* out, void* normed_ws,
                                      void* act_ws, void* h_out, float* rms_out, void* gate_cache, void* up_cache,
                                      const void* next_norm_weight, float next_eps, void* next_normed, float* next_rms,
                                      int64_t tokens, int hidden, int inter, int dtype, void* stream);

/* Whole feed-forward backward (down projection included).
 *   dy : [tokens, hidden].  Outputs (each optional): dx [tokens, hidden], dw_gate / dw_up [inter, hidden]
 *   (both or neither), dw_down [hidden, inter].
 *   workspace : l32_ffn_backward_workspace_bytes(tokens, inter) bytes (d_gate, d_up, recomputed act).
 * No reference counterpart exists (the reference's backward never ran, SURVEY.md section 0.4); the
 * gradient oracle is autograd over Tools/swiglu/FusedSwiglu.py:18-20 + Model/model.py:217.
 */
L32_API size_t l32_ffn_backward_workspace_bytes(int64_t tokens, int inter);
L32_API int l32_ffn_backward(const void* dy, const void* x, const void* w_gate, const void* w_up, const void* w_down,
                     const void* gate_cache, const void* up_cache, void* dx, void* dw_gate, void* dw_up,
                     void* dw_down, void* workspace, size_t workspace_bytes, int64_t tokens, int hidden, int inter,
                     int dtype, void* stream);

/* Feed-forward whose down projection carries a LoRA adapter: y = act w_down^T + (act lora_a^T) lora_bs^T.
 * Replaces: Linear_LORA.forward (Model/model.py:120-121) swapped into FusedFeedforward.w_down by the fine-tuning
 *           recipe of README.md:179-188 (rank 16, alpha 32); the adapter rides in the down GEMM as a second
 *           accumulation phase of K = rank, so the [tokens, hidden] LoRA term never exists in HBM.
 *   lora_a  : [rank, inter];  lora_bs : [hidden, rank], ALREADY multiplied by alpha / rank;  rank % 8 == 0, rank <= 64.
 *   t_out   : [tokens, rank] receives act lora_a^T (needed by the backward);  act_ws : [tokens, inter] scratch.
 *   (LoRA dropout is the caller's business: with p > 0 in training mode the host layer uses the unfused path.)
 */
L32_API int l32_ffn_lora_forward(const void* x, const void* w_gate, const void* w_up, const void* w_down, const void* lora_a,
                                 const void* lora_bs, void* y, void* act_ws, void* t_out, void* gate_cache, void* up_cache,
                                 int64_t tokens, int hidden, int inter, int rank, int dtype, void* stream);

/* Backward of l32_ffn_lora_forward with a frozen base w_down (no dw_down).
 *   Outputs (each optional): dx, dw_gate / dw_up (both or neither), dlora_a [rank, inter], dlora_bs [hidden, rank]
 *   (gradient w.r.t. the SCALED matrix; multiply by alpha / rank for lora_b).
 *   workspace : l32_ffn_lora_backward_workspace_bytes(tokens, inter, rank) bytes.
 */
L32_API size_t l32_ffn_lora_backward_workspace_bytes(int64_t tokens, int inter, int rank);
L32_API int l32_ffn_lora_backward(const void* dy, const void* x, const void* w_gate, const void* w_up, const void* w_down,
                                  const void* lora_a, const void* lora_bs, const void* t, const void* gate_cache,
                                  const void* up_cache, void* dx, void* dw_gate, void* dw_up, void* dlora_a, void* dlora_bs,
                                  void* workspace, size_t workspace_bytes, int64_t tokens, int hidden, int inter, int rank,
                                  int dtype, void* stream);

/* Any Linear_LORA layer (Model/model.py:107-121; the attention projections q/k/v/out of README.md:179-188 as well as
 * w_down): y = x w^T + bias + (dropout(x) lora_a^T) lora_bs^T with the adapter as a second accumulation phase of the base
 * GEMM.
 *   x_lora : optional [tokens, in], the adapter's input dropout(x) (Model/model.py:121) when LoRA dropout is active -- the
 *            mask is the caller's (exact nn.Dropout semantics); NULL = x itself.
 *   lora_bs: [out, rank], already multiplied by alpha / rank;  t_out : [tokens, rank] receives dropout(x) lora_a^T.
 */
L32_API int l32_linear_lora_forward(const void* x, const void* x_lora, const void* w, const void* bias, const void* lora_a,
                                    const void* lora_bs, void* y, void* t_out, int64_t tokens, int in_features,
                                    int out_features, int rank, int dtype, void* stream);
/* Backward with a frozen base weight: u = dy lora_bs (written to u_out [tokens, rank]);
 *   dx      = dy w + u lora_a                    (dx_addend == NULL: ONE GEMM, two accumulation phases), or
 *   dx      = dy w + dx_addend                   (LoRA dropout: the caller forms mask * (u lora_a) / (1 - p) and the epilogue
 *                                                 of the base GEMM adds it);
 *   dlora_a = u^T x_lora  [rank, in];  dlora_bs = dy^T t  [out, rank] (gradient w.r.t. the SCALED matrix).
 * Every output is optional; u_out may be NULL only for a pure `dx = dy w + dx_addend` call (no dlora_a). */
L32_API int l32_linear_lora_backward(const void* dy, const void* x_lora, const void* w, const void* lora_a, const void* lora_bs,
                                     const void* t, const void* dx_addend, void* dx, void* dlora_a, void* dlora_bs, void* u_out,
                                     int64_t tokens, int in_features, int out_features, int rank, int dtype, void* stream);

/* lm_head + cross entropy (SURVEY.md 8f rank 4).
 * Replaces: `logits = self.language_model.lm_head(hidden_states)` followed by
 *           `nn.CrossEntropyLoss(ignore_index)(shift_logits.view(-1, V), shift_labels.view(-1))`, Model/model.py:429-438
 *           (lm_head = nn.Linear(hidden, vocab, bias=False), Model/model.py:354, tied to tok_emb by tie_weights, :363-364).
 * ONE tcgen05 GEMM whose epilogue stores the logits (16-bit, the model's output) and gathers each row's softmax statistics
 * per 256-column tile, then two tiny reductions: no fp32 [tokens, vocab] tensor and no second pass over the logits.
 *   labels        : [tokens] int64, ALREADY SHIFTED by the caller (row (b, s) carries labels[b, s + 1], the last position
 *                   of every sequence carries ignore_index); values outside [0, vocab) never match;
 *   logits        : [tokens, vocab] in `dtype`;  lse : [tokens] fp32 log-sum-exp of the stored (rounded) logits;
 *   loss_rows     : [tokens] fp32, lse - logit[label] (0 for ignored rows);
 *   loss_and_count: [2] fp32 = { mean of loss_rows over the valid rows (nan when there is none, like torch), #valid rows };
 *   workspace     : l32_lm_head_ce_workspace_bytes(tokens, vocab) bytes.
 */
L32_API size_t l32_lm_head_ce_workspace_bytes(int64_t tokens, int vocab);
L32_API int l32_lm_head_ce_forward(const void* hidden_states, const void* w, const int64_t* labels, long long ignore_index,
                                   void* logits, float* lse, float* loss_rows, float* loss_and_count, void* workspace,
                                   size_t workspace_bytes, int64_t tokens, int hidden, int vocab, int dtype, void* stream);
/* Backward: dlogits = (softmax(logits) - onehot(labels)) * grad_loss / #valid (from the stored logits and lse; `dlogits` may
 * alias `logits`; grad_loss = DEVICE pointer to the fp32 upstream gradient of the scalar loss, NULL = 1), d_hidden = dlogits w (optional), dw = dlogits^T hidden_states (optional, [vocab, hidden]). */
L32_API int l32_lm_head_ce_backward(const void* logits, const float* lse, const int64_t* labels, long long ignore_index,
                                    const float* loss_and_count, const float* grad_loss, const void* hidden_states, const void* w,
                                    void* dlogits, void* d_hidden, void* dw, int64_t tokens, int hidden, int vocab, int dtype,
                                    void* stream);

/* ---------------------------------------------------------------------------------------------
 * Grouped-query attention with a preallocated KV cache (SURVEY.md 8f rank 3).
 * Replaces: GroupQueryAttention.forward between the projections, Model/model.py:238-253 -- RoPE (apply_rotary_pos_emb,
 *           :195-198, angles of LLAMARotaryEmbedding :176-186), KVCache.update (:21-29, one torch.cat per layer per step),
 *           repeat_kv (:124-132), the materialised [B, heads, S, S] scores + dense additive mask + softmax + P V (:246-252).
 * Layouts: q, ctx : [batch, q_len, heads * head_dim] (what W_query / out_proj produce / consume, no transposes);
 *          k_new, v_new : [batch, q_len, kv_heads * head_dim];  cache_k, cache_v : [batch, kv_heads, max_len, head_dim],
 *          ZERO-INITIALISED by the caller (rows past the current length are multiplied by zero probabilities).
 */
/* RoPE on q (in place) and on k_new while it is stored at cache_k[:, :, past_len : past_len + q_len]; v_new is stored next
 * to it.  position_ids : [batch, q_len] int64 absolute positions (pass them explicitly in decode: the reference's default
 * restarts at 0 every step, SURVEY.md 0.9).  rope_base = config.rope_base (500000).  Angles in fp32. */
L32_API int l32_rope_kv_append(void* q, const void* k_new, const void* v_new, const int64_t* position_ids, void* cache_k,
                               void* cache_v, int batch, int q_len, int heads, int kv_heads, int head_dim, int max_len,
                               int past_len, float rope_base, int dtype, void* stream);
/* ctx = softmax(q k^T / sqrt(head_dim) + mask) v over keys [0, kv_len) of the cache, flash-style on tcgen05 (scores never
 * leave the SM).  Query i of the call sits at position past_len + i.  causal != 0: key j is visible iff j <= past_len + i
 * (the reference's triu(-inf, 1) mask, Model/model.py:314-317); key_keep: optional [batch, kv_len] bytes, 0 = padded key
 * (the reference's padding term, :318).  A row without any visible key yields zeros.  head_dim 64 or 128.
 * workspace (optional): l32_gqa_attention_workspace_bytes(...) bytes.  With it a decode step (q_len == 1) splits the cached
 * keys over several CTAs per KV head (fp32 partials + a merge kernel, fixed order: deterministic), which is what keeps small
 * batches with long contexts from running on a handful of SMs; without it (or when the function returns 0) one CTA per KV head
 * walks the whole cache.  The function returns non-zero exactly when the call will split: q_len == 1, no key_keep, a group
 * heads / kv_heads of 2 to 128, and enough keys.  Cache rows at or beyond kv_len are never read (whatever they hold). */
L32_API size_t l32_gqa_attention_workspace_bytes(int batch, int q_len, int heads, int kv_heads, int head_dim, int kv_len);
L32_API int l32_gqa_attention_forward(const void* q, const void* cache_k, const void* cache_v, const uint8_t* key_keep,
                                      void* ctx, void* workspace, size_t workspace_bytes, int batch, int q_len, int heads,
                                      int kv_heads, int head_dim, int max_len, int kv_len, int past_len, int causal, int dtype,
                                      void* stream);

/* Training calls (no KV cache): keys are [0, q_len) of cache_k / cache_v (rows [q_len, max_len), if any, must hold finite
 * values: they are multiplied by zero probabilities), query i sits at position i.  Same masks as l32_gqa_attention_forward.  Deterministic: no floating-point atomics, the same inputs give the
 * same bits.
 * forward_train: ctx as l32_gqa_attention_forward, and lse [batch, heads, q_len] fp32: the log-sum-exp of each row's scaled
 *   scores in the log2 domain, +inf for a row that sees no key.
 * backward: from d_ctx (the gradient of ctx) and the forward's q_rot, K / V, ctx and lse: dq [batch, q_len, heads * head_dim],
 *   dk / dv [batch, q_len, kv_heads * head_dim] -- the gradients of the projection outputs BEFORE RoPE (the inverse rotation at
 *   position_ids [batch, q_len], rope_base as in l32_rope_kv_append, is applied).  A row that sees no key gets dq = 0 and
 *   contributes nothing (the reference gives it a uniform softmax, whose loss a model ignores); a padded key gets dk = dv = 0.
 *   workspace: l32_gqa_attention_backward_workspace_bytes(...) bytes, 16-byte aligned.  Enqueues three kernels; nothing
 *   allocates or synchronises (graph-capturable). */
L32_API int l32_gqa_attention_forward_train(const void* q_rot, const void* cache_k, const void* cache_v, const uint8_t* key_keep,
                                            void* ctx, float* lse, int batch, int q_len, int heads, int kv_heads, int head_dim,
                                            int max_len, int causal, int dtype, void* stream);
L32_API size_t l32_gqa_attention_backward_workspace_bytes(int batch, int q_len, int heads);
L32_API int l32_gqa_attention_backward(const void* d_ctx, const void* q_rot, const void* cache_k, const void* cache_v, const void* ctx,
                                       const float* lse, const uint8_t* key_keep, const int64_t* position_ids, void* dq, void* dk,
                                       void* dv, void* workspace, size_t workspace_bytes, int batch, int q_len, int heads,
                                       int kv_heads, int head_dim, int max_len, int causal, float rope_base, int dtype,
                                       void* stream);

/* ---------------------------------------------------------------------------------------------
 * Paged KV cache: per-sequence lengths in device memory, keys in fixed-size pages named by a block table (inference only).
 * Layout:
 *   page       : L32_KV_PAGE = 64 tokens, the attention kernel's key tile (one key tile is exactly one page).
 *   pool_k / pool_v : [num_pages, kv_heads, L32_KV_PAGE, head_dim] per layer, one (page, kv head) slice = 64 x head_dim
 *                contiguous elements.  Page index p names the same slot in every layer's pool (one allocator serves all layers).
 *   block_table : int32 [batch, max_pages_per_seq]; logical page j of sequence b is block_table[b][j].
 *   past_lens   : int32 [batch], tokens already cached for sequence b.
 *   new_lens    : int32 [batch] or NULL: tokens this call appends for sequence b (NULL: every row has q_len).  The keys a call
 *                sees for sequence b are [0, past_lens[b] + new_lens[b]); its query i sits at position past_lens[b] + i.
 *   q, ctx      : [batch, q_len, heads * head_dim], right-padded: query rows i >= new_lens[b] are padding.
 * CONTRACT on stale rows: every row of a page at or beyond its sequence's length must hold FINITE values (they are multiplied by
 *   zero probabilities, and 0 * NaN is NaN in P V).  Pools that start zeroed and are written only by l32_rope_kv_append_paged
 *   keep this without zeroing a page when it is handed to another sequence.
 * The table and length values live in device memory and are TRUSTED: every page index must lie in [0, num_pages), every
 *   past_lens[b] + new_lens[b] must be <= max_pages_per_seq * 64 (and <= max_kv_len for the attention) and every page a call
 *   reads or writes must be in the table.  The caller (the Python PagedKVCache) checks them when it builds them.
 * Same rules as the other entry points: nothing allocates or synchronises, everything is graph-capturable, and argument errors
 * return L32_ERR_* before any launch.
 */
#define L32_KV_PAGE 64
/* RoPE on q (in place, every row) and on k_new while it is stored at position past_lens[b] + t of sequence b, i.e. row
 * (pos % 64) of page block_table[b][pos / 64]; v_new stored next to it.  Tokens t >= new_lens[b] write nothing to the pools.
 * position_ids [batch, q_len] int64 as in l32_rope_kv_append.  head_dim 64 or 128. */
L32_API int l32_rope_kv_append_paged(void* q, const void* k_new, const void* v_new, const int64_t* position_ids, void* pool_k,
                                     void* pool_v, const int32_t* block_table, const int32_t* past_lens, const int32_t* new_lens,
                                     int batch, int q_len, int heads, int kv_heads, int head_dim, int num_pages, int max_pages_per_seq,
                                     float rope_base, int dtype, void* stream);
/* ctx = causal attention of each sequence's queries over its own keys (for one query per sequence that is no mask at all).
 * Padded query rows yield exact zeros.  max_kv_len: a host bound >= every past_lens[b] + new_lens[b]; it sizes the split-KV
 * plan of a decode step (q_len == 1) exactly as kv_len does for l32_gqa_attention_forward, so the workspace is
 * l32_gqa_attention_workspace_bytes(batch, q_len, heads, kv_heads, head_dim, max_kv_len) (optional, as there).  With uniform
 * lengths, max_kv_len equal to them and the same keys laid out in pages, the result is bit-identical to
 * l32_gqa_attention_forward's. */
L32_API int l32_gqa_attention_forward_paged(const void* q, const void* pool_k, const void* pool_v, const int32_t* block_table,
                                            const int32_t* past_lens, const int32_t* new_lens, void* ctx, void* workspace,
                                            size_t workspace_bytes, int batch, int q_len, int heads, int kv_heads, int head_dim,
                                            int num_pages, int max_pages_per_seq, int max_kv_len, int dtype, void* stream);

/* Cascade decode over a paged cache whose sequences share prefix pages (forked sequences: PagedKVCache.fork).  One decode step
 * (one query per sequence, group = heads / kv_heads in [2, L32_CASCADE_TILE_ROWS]) computed as
 *   prefix pass : per (kv head, prefix work item) one query tile of L32_CASCADE_TILE_ROWS rows holding the `group` query
 *                 heads of up to floor(128 / group) member sequences, over the item's shared key tiles (read once for all
 *                 its members);
 *   own-key pass: per (sequence, kv head, split) the packed paged decode over the sequence's keys from its shared tiles on;
 *   combine     : the row's prefix partials, then its split partials, merged in that fixed order.
 * Same layout and stale-row contract as l32_gqa_attention_forward_paged (q_len = 1; new_lens NULL means one new token per
 * sequence, 0 marks a row that yields zeros).  The plan, int32 in device memory, TRUSTED like the table:
 *   plan_items  : [1 + 5 * max_items]: the item count n <= max_items, then per item (first_seq, tile0, tiles, member0,
 *                 members): keys [tile0 * 64, (tile0 + tiles) * 64) read through block_table row first_seq, for the query
 *                 rows of sequences plan_members[member0 .. member0 + members), members * group <= 128.
 *   plan_members: [batch] sequence indices.
 *   plan_seq    : [batch][4] per sequence (shared_tiles, first_item, items, row0): its keys [0, shared_tiles * 64) are covered
 *                 by items first_item .. first_item + items - 1, where it is member row0 / group (query tile rows row0 ..
 *                 row0 + group - 1); items = 0 for a sequence outside the prefix pass (shared_tiles = 0).
 *   The prefix tiles of a sequence must be full pages of ITS table (the same pages as first_seq's) and lie below
 *   past_lens[b]: they are read with no mask.  Items past n are ignored, as is every workspace slot the plan does not name.
 * max_items: the plan's capacity; it fixes the launch shape, so a CUDA graph captured once stays valid while the plan's
 * contents change between replays.  max_kv_len: as for l32_gqa_attention_forward_paged (sizes the own-key split plan).
 * workspace: l32_gqa_attention_cascade_workspace_bytes(...) bytes, 16-byte aligned (required).  Enqueues two kernels.
 * Deterministic: the same inputs give the same bits. */
#define L32_CASCADE_TILE_ROWS 128
#define L32_CASCADE_MAX_ITEMS 65535
L32_API size_t l32_gqa_attention_cascade_workspace_bytes(int batch, int heads, int kv_heads, int head_dim, int max_kv_len,
                                                         int max_items);
L32_API int l32_gqa_attention_forward_paged_cascade(const void* q, const void* pool_k, const void* pool_v, const int32_t* block_table,
                                                    const int32_t* past_lens, const int32_t* new_lens, const int32_t* plan_items,
                                                    const int32_t* plan_members, const int32_t* plan_seq, void* ctx, void* workspace,
                                                    size_t workspace_bytes, int batch, int heads, int kv_heads, int head_dim,
                                                    int num_pages, int max_pages_per_seq, int max_kv_len, int max_items, int dtype,
                                                    void* stream);

/* ---------------------------------------------------------------------------------------------
 * Speculative decoding on the paged KV cache (inference only; the paged layout, stale-row and trusted-table rules above hold).
 *
 * Verify attention: l32_gqa_attention_forward_paged for a step in which each sequence has up to q_len = t new tokens (its
 * drafts), computed with one query tile per (sequence, kv head) that holds the group = heads / kv_heads query heads of each of
 * the t tokens, so every key is read once per kv head.  Same arguments, layout and result (up to the order of the softmax
 * sums) as l32_gqa_attention_forward_paged; query rows i >= new_lens[b] and rows with new_lens[b] == 0 yield exact zeros.
 * Requires 2 <= group and group * q_len <= L32_VERIFY_TILE_ROWS (L32_ERR_BAD_SHAPE otherwise).  The split-KV plan is the
 * packed decode's for max_kv_len; workspace: l32_gqa_attention_verify_workspace_bytes(...) bytes (optional: without it the
 * call runs in one pass).  Enqueues one kernel, or two with the split.  Deterministic. */
#define L32_VERIFY_TILE_ROWS 128
L32_API size_t l32_gqa_attention_verify_workspace_bytes(int batch, int q_len, int heads, int kv_heads, int head_dim, int max_kv_len);
L32_API int l32_gqa_attention_forward_paged_verify(const void* q, const void* pool_k, const void* pool_v, const int32_t* block_table,
                                                   const int32_t* past_lens, const int32_t* new_lens, void* ctx, void* workspace,
                                                   size_t workspace_bytes, int batch, int q_len, int heads, int kv_heads, int head_dim,
                                                   int num_pages, int max_pages_per_seq, int max_kv_len, int dtype, void* stream);
/* Token history: token_pool int32 [num_pages, L32_KV_PAGE], named by the same block table as K / V: token i of sequence b is
 * token_pool[block_table[b][i / 64]][i % 64].  A sequence's history holds exactly past_lens[b] tokens (its KV length); the
 * sampled token whose K / V is not computed yet (the pending token) is kept by the caller.
 *
 * N-gram drafts, one row per sequence b < batch: S = history [0, past_lens[b]) followed by pending[b].  For n = n_max down to
 * n_min (n <= |S| - 1), j is the largest index with S[j, j + n) == S[|S| - n, |S|) and j + n < |S|; the first n with such a j
 * proposes S[j + n, j + n + k) cut at |S|.  Writes ids[b][0] = pending[b], ids[b][1 .. k] = the proposal, padded with its last
 * token (with pending[b] when there is none), and draft_len[b] = the proposal's length (optional).  ids: int64 [batch, k + 1].
 * 1 <= k, 1 <= n_min <= n_max <= L32_NGRAM_MAX.  Deterministic; one launch. */
#define L32_NGRAM_MAX 16
L32_API int l32_ngram_draft_paged(const int32_t* token_pool, const int32_t* block_table, const int32_t* past_lens,
                                  const int64_t* pending, int64_t* ids, int32_t* draft_len, int batch, int k, int n_min, int n_max,
                                  int num_pages, int max_pages_per_seq, void* stream);
/* Acceptance.  ids int64 [batch, width] (the pending token, then the drafts), sampled int64 [batch * width], where row i of
 * sequence b was sampled at position past_lens[b] + i + 1.  For each b with n = min(new_lens[b], width) > 0: a = the number
 * of leading i < n - 1 with ids[b][i + 1] == sampled[b][i]; ids[b][0 .. a] are written to the history at positions
 * past_lens[b] .. past_lens[b] + a, and out[b] (int64 [batch, width + 1]) = (a + 1, sampled[b][0 .. a], then -1).  Rows with
 * new_lens[b] == 0 are not touched.  sampled == NULL keeps all n tokens of the row (a prompt written into the history) and
 * writes only out[b][0] = n when out is given.  The pages written must be in the table and not shared.  One launch. */
L32_API int l32_speculative_accept(const int64_t* ids, const int64_t* sampled, int32_t* token_pool, const int32_t* block_table,
                                   const int32_t* past_lens, const int32_t* new_lens, int64_t* out, int batch, int width,
                                   int num_pages, int max_pages_per_seq, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Next-token sampling: one token per row of 16-bit logits [batch, vocab] (row pitch = vocab), written to tokens_out [batch]
 * (int64).  Replaces the torch sampler of the reference's decode loop (Inference/Inference.py, select_next_token).
 * Per-row parameters, device arrays of `batch` entries: temperature (f32), top_k (i32), top_p (f32), seed (u64),
 * position (i64, the position of the token being sampled).  For row r:
 *   1. Greedy: temperature <= 0 or NaN -> the smallest index among the maximal logits (torch.argmax's choice).
 *   2. Otherwise z_i = logit_i / temperature in fp32.
 *   3. Top-k, if 0 < top_k < vocab: keep every token with logit_i >= v_k, the top_k-th largest logit counted with
 *      multiplicity; all ties at v_k survive.
 *   4. Top-p, if top_p < 1: over the survivors' softmax of z, keep every token with logit_i >= v_p, the largest logit value
 *      whose survivors at or above it carry at least top_p of the survivors' mass (top_p <= 0: only the maximal value).
 *   5. -inf is never kept.
 *   6. Return the argmax over kept i of z_i + g_i (smallest index on ties), g_i = -log(-log(u_i)): an exact sample of the
 *      kept set's softmax.  u_i = ((out[i & 3] >> 8) + 0.5) * 2^-24 with out = Philox4x32-10 of counter
 *      (i >> 2, 0, position_lo, position_hi) under key (seed_lo, seed_hi).
 * A draw is a function of (logits row, parameters, seed, position) only: not of the batch, the row index or graph capture.
 * Values outside the contract are clamped: top_k <= 0 or >= vocab means no top-k, top_p >= 1 or NaN means no top-p.
 * A row without a finite logit returns 0.  The parameter values are TRUSTED (the Python TokenSampler validates them).
 * kept_min_logit: optional [batch] f32, the smallest kept logit of each row (greedy: the maximum; no finite logit: -inf);
 * with it NULL nothing extra is computed.  8 <= vocab <= L32_SAMPLE_MAX_VOCAB, vocab % 8 == 0, logits 16-byte aligned;
 * batch == 0 is a no-op.  One launch (a cluster of up to 8 CTAs per row), deterministic, graph-capturable. */
#define L32_SAMPLE_MAX_VOCAB 262144
L32_API int l32_sample_tokens(const void* logits, const float* temperature, const int32_t* top_k, const float* top_p,
                              const uint64_t* seed, const int64_t* position, int64_t* tokens_out, float* kept_min_logit, int batch,
                              int vocab, int dtype, void* stream);

/* General tiled GEMM used by the entry points above (exposed for tests, tuning and the tensor-parallel
 * host code):  D[m,n] = A[m,k] B[n,k]^T  (+ A1 B1^T when a1 != NULL).
 *   *_mn_major = 0: operand stored [rows][k];  1: stored [k][rows] (i.e. the transpose is consumed in place).
 *   cta_group: 0 auto, 1, or 2 (CTA pair, UMMA M = 256).  max_ctas: 0 = all SMs.
 */
L32_API int l32_gemm(const void* a, int64_t lda, int a_mn_major, const void* b, int64_t ldb, int b_mn_major, const void* a1,
             int64_t lda1, const void* b1, int64_t ldb1, void* d, int64_t ldd, int m, int n, int k, int k1, int dtype,
             int cta_group, int max_ctas, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Tensor-parallel feed-forward (one process per GPU; gate/up column-parallel, down row-parallel).
 * No reference counterpart: the reference has no distributed code (SURVEY.md section 8e); these entry points
 * implement the sharding of Tools/swiglu/FusedSwiglu.py:63-64 / Model/model.py:214 that BASELINE.json asks for.
 * "peer" pointers are device pointers of OTHER ranks' buffers mapped into this process (CUDA IPC / symmetric
 * memory); the arrays holding them are HOST arrays of `world` entries (world <= 8), entry [rank] = own buffer.
 * Flags are uint32 step counters ("epoch", monotonic, starting at 1) living in each rank's own memory.
 */

/* flag[index] := value on every rank, after everything this stream did before is visible system-wide.
 * zero8 : optional, 8 uint32 of this rank's memory cleared by the same kernel (the `done` counters of the next
 *         l32_tp_swiglu_forward_allgather -- saves a memset launch). */
L32_API int l32_tp_signal(void* const* peer_flags, int world, int index, uint32_t value, uint32_t* zero8, void* stream);

/* Plain SM copy between (peer) buffers: the NVLink bandwidth reference for the fused kernels (pull when src is peer
 * memory, push when dst is).  bytes % 16 == 0; `ctas` CTAs of `warps` warps, `unroll` (4, 8 or 16) loads in flight per lane.
 * seg_bytes = 0: linear copy; otherwise the buffer is walked like a GEMM epilogue walks its output (runs of seg_bytes
 * contiguous bytes at a row pitch of 8192 bytes), to measure what short contiguous runs cost on NVLink. */
L32_API int l32_tp_peer_copy(void* dst, const void* src, size_t bytes, int ctas, int warps, int unroll, int seg_bytes,
                             void* stream);

/* Fused all-gather + gate/up projection + SiLU*mul.
 *   x_full   : this rank's [tokens, hidden] activation buffer.  If x_full == peer_x[rank] (gather in place) only rows
 *              [rank*rows_per_rank, ...) are valid on entry; otherwise the own rows are copied from peer_x[rank] too and
 *              x_full may be a tensor the caller keeps (the saved input of the weight gradients).  The kernel PULLS the other ranks' rows out of peer_x[s] (NVLink loads issued by the spare
 *              warps of the tcgen05 GEMM CTAs) while the tensor cores already work on the rows that have arrived;
 *              tiles are visited starting at the own rows, then rank+1, rank+2, ... (the pull order).
 *   ready    : own flags, ready[s] >= epoch once rank s has written its rows (see l32_tp_signal).
 *   done     : own scratch counters, 8 uint32, cleared by this call (cudaMemsetAsync on `stream`).
 *   w_gate, w_up : this rank's shard [inter_local, hidden]; act : [tokens, inter_local].
 */
L32_API int l32_tp_swiglu_forward_allgather(void* x_full, const void* const* peer_x, const uint32_t* ready, uint32_t* done,
                                            uint32_t epoch, int rank, int world, int64_t rows_per_rank, const void* w_gate,
                                            const void* w_up, const void* b_gate, const void* b_up, void* act,
                                            void* gate_cache, void* up_cache, int64_t tokens, int hidden, int inter_local,
                                            int dtype, void* stream);

/* Fused down projection + reduce-scatter: y_partial = a w^T is stored row by row straight into the slot of the rank
 * that owns the row: peer_slots[o] = base of rank o's [rows_per_rank, out_features] slot for THIS rank's partial.
 *   a : [tokens, in_local]; w : this rank's shard [out_features, in_local] (contiguous copy of w_down[:, shard]).
 */
L32_API int l32_tp_linear_forward_reduce_scatter(const void* a, const void* w, void* const* peer_slots, int rank, int world,
                                                 int64_t rows_per_rank, int64_t tokens, int in_local, int out_features,
                                                 int dtype, void* stream);

/* Tensor-parallel BACKWARD of the feed-forward (mirror image of the two forward calls: all-gather of dY pulled inside
 * the d_act GEMM, reduce-scatter of the partial dX pushed from the two-phase dX GEMM; the weight gradients are local
 * l32_gemm calls on the shard).  No reference counterpart (SwiGLUFunction.backward, Tools/swiglu/FusedSwiglu.py:32-40,
 * never ran and the reference has no distributed code); the gradient oracle is autograd over FusedSwiglu.py:18-20 +
 * Model/model.py:217.
 *   dy_full  : this rank's [tokens, hidden] buffer for the gathered output gradient (rows of rank s pulled from
 *              peer_dy[s]; when peer_dy[rank] != dy_full the own rows are copied in as well, so dy_full can be a tensor
 *              the caller keeps for the w_down weight gradient).
 *   w_down   : this rank's shard [hidden, inter_local] (consumed MN-major, no transpose);
 *   gate_cache, up_cache : [tokens, inter_local] from the forward;  d_gate, d_up : [tokens, inter_local] outputs;
 *   act_out  : optional [tokens, inter_local], the recomputed act = silu(gate) * up (operand of dW_down).
 */
L32_API int l32_tp_ffn_backward_dact_allgather(void* dy_full, const void* const* peer_dy, const uint32_t* ready,
                                               uint32_t* done, uint32_t epoch, int rank, int world, int64_t rows_per_rank,
                                               const void* w_down, const void* gate_cache, const void* up_cache,
                                               void* d_gate, void* d_up, void* act_out, int64_t tokens, int hidden,
                                               int inter_local, int dtype, void* stream);
/*   partial dx = d_gate w_gate_shard + d_up w_up_shard (ONE GEMM, two accumulation phases), every row stored into the
 *   slot of the rank that owns it (peer_slots as in l32_tp_linear_forward_reduce_scatter); the owner then sums the
 *   slots with l32_tp_reduce_partials. */
L32_API int l32_tp_ffn_backward_dx_reduce_scatter(const void* d_gate, const void* d_up, const void* w_gate, const void* w_up,
                                                  void* const* peer_slots, int rank, int world, int64_t rows_per_rank,
                                                  int64_t tokens, int hidden, int inter_local, int dtype, void* stream);

/* Tensor-parallel attention (heads sharded by KV group: rank r owns query heads [r H/p, (r+1) H/p) and KV heads
 * [r kv/p, (r+1) kv/p)).  No reference counterpart (the reference has no distributed code); the oracle is
 * Model/model.py:238-253 with the shards summed.
 *
 * Up to three projections of the SAME gathered activations in one persistent launch: y[i] = x_full w[i]^T, w[i]
 * [out_features[i], in_features] K-major (the shard's rows of W_query / W_key / W_value), y[i] [tokens, out_features[i]].
 * The all-gather of x_full is pulled inside the kernel exactly as in l32_tp_swiglu_forward_allgather (same meaning of
 * x_full, peer_x, ready, done, epoch, rows_per_rank); every problem's tiles start at the own rows.  At world == 1 this is
 * the tiled path of l32_linear_group_forward. */
L32_API int l32_tp_linear_group_forward_allgather(void* x_full, const void* const* peer_x, const uint32_t* ready,
                                                  uint32_t* done, uint32_t epoch, int rank, int world, int64_t rows_per_rank,
                                                  const void* const* w, void* const* y, const int* out_features, int count,
                                                  int64_t tokens, int in_features, int dtype, void* stream);
/* y [tokens, out_features] = a_full w^T with the all-gather of a_full pulled in (arguments as above).  w_mn_major = 0:
 * w is [out_features, in_features]; w_mn_major = 1: w is [in_features, out_features] (e.g. d_ctx = dY_full out_proj_shard
 * with the out_proj shard [hidden, heads_local * head_dim] as it is). */
L32_API int l32_tp_linear_forward_allgather(void* a_full, const void* const* peer_a, const uint32_t* ready, uint32_t* done,
                                            uint32_t epoch, int rank, int world, int64_t rows_per_rank, const void* w,
                                            int w_mn_major, void* y, int64_t tokens, int in_features, int out_features,
                                            int dtype, void* stream);
/* partial dx [tokens, hidden] = sum_{i < num_phases} dy[i] w[i] (ONE GEMM, up to three accumulation phases): dy[i]
 * [tokens, k[i]], w[i] [k[i], hidden] (row slices of W_query / W_key / W_value, consumed MN-major); every row is stored
 * into the slot of the rank that owns it (peer_slots as in l32_tp_linear_forward_reduce_scatter). */
L32_API int l32_tp_linear_group_backward_dx_reduce_scatter(const void* const* dy, const void* const* w, const int* k,
                                                           int num_phases, void* const* peer_slots, int rank, int world,
                                                           int64_t rows_per_rank, int64_t tokens, int hidden, int dtype,
                                                           void* stream);

/* The two forward calls above as ONE persistent kernel: gate/up tiles (all-gather pulled in) and down tiles (reduce-scatter pushed
 * out) share the tile loop -- the down tiles of one group of rows are interleaved with the gate/up tiles of the next
 * group, so the NVLink pushes overlap the (twice as long) gate/up math instead of only the down projection, and the
 * intermediate act is consumed while it is still in L2.
 *   act_ws   : [tokens, inter_local] scratch;  act_done : ceil(tokens / 256) uint32 scratch (cleared by this call);
 *   other arguments as in l32_tp_swiglu_forward_allgather / l32_tp_linear_forward_reduce_scatter.
 */
L32_API int l32_tp_ffn_forward_fused(void* x_full, const void* const* peer_x, const uint32_t* ready, uint32_t* done,
                                     uint32_t epoch, int rank, int world, int64_t rows_per_rank, const void* w_gate,
                                     const void* w_up, const void* w_down, void* act_ws, uint32_t* act_done,
                                     void* const* peer_slots, int64_t tokens, int hidden, int inter_local, int dtype,
                                     void* stream);

/* y[rows, hidden] = sum_s slots[s][rows, hidden] (+ addend), fp32 accumulation in rank order, after waiting until
 * flags[s] >= epoch for every s != rank.  slots : own [world, slot_rows, hidden] buffer the peers pushed into. */
L32_API int l32_tp_reduce_partials(const void* slots, const uint32_t* flags, uint32_t epoch, int world, int rank,
                                   const void* addend, void* y, int64_t rows, int64_t slot_rows, int hidden, int dtype,
                                   void* stream);

/* Host-side view of the persistent kernels' tile sequences (no GPU needed; used by the CPU tests).
 *   kind 0: plain / reduce-scatter order, cfg = {tiles_m, tiles_n, group, m_rotate, il_world, il_tiles_per_chunk, il_rank}
 *   kind 1: one-kernel feed-forward order, cfg = {tiles_m, n_tiles_gate_up, n_tiles_down, group, m_rotate, prefix}
 *   out3 = {problem (0 gate/up or plain, 1 down), m_tile, n_tile} of the t-th tile. */
L32_API int l32_debug_tile_order(int kind, int t, const int* cfg, int* out3);

/* Launch plan of the tiled GEMM for one (not grouped) problem D[m, n], as the library would launch it (no GPU needed).
 *   epilogue : 0 plain store (256-column tiles), 1 fused gate/up + SwiGLU (n = intermediate size), 2 SwiGLU backward,
 *              4 lm_head + cross entropy
 *   cta_group: 0 = auto (2 above 128 rows), 1 or 2;  max_ctas: 0 = every SM;  num_sms: 0 = the current device's
 *   out[7]   = {cta_group, tiles_m, tiles_n, n_act (act columns per tile of epilogue 1, else 128), raster_group (m-tiles
 *              per raster group), num_tiles, ctas launched}.
 * Reads the L32_SWIGLU_TILE_N and L32_RASTER_GROUP overrides like the launch does. */
L32_API int l32_debug_gemm_plan(int epilogue, int m, int n, int cta_group, int max_ctas, int num_sms, int* out);

/* Elementwise helpers (unfused reference points for tests / benchmarks of the fusion saving). */
L32_API int l32_swiglu_act(const void* gate, const void* up, void* act, int64_t n, int dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* L32_FFN_H_ */
