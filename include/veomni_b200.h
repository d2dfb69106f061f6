/*
 * veomni_b200 C ABI — the drop-in boundary of the B200-native hot path.
 *
 * The reference (ByteDance-Seed/VeOmni) has no native code: its "FFI" for this path is the
 * set of Python hooks listed in SURVEY.md §8(b) (OpSlot kernels, the Ulysses all-to-all choke
 * point, the EP dispatch/combine functions, and PyTorch FSDP2's custom AllGather/ReduceScatter
 * hooks).  Every entry point below is what the Python side of one of those hooks binds through
 * ctypes (veomni_b200/_lib.py); each cites the reference call site it replaces.
 *
 * Conventions
 *   - plain pointers + sizes, no torch types; all device pointers unless stated otherwise
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream)
 *   - return 0 on success, negative VB200_E* on failure; vb200_last_error() has the text
 *   - no allocation inside compute calls; no hidden global state except the explicit
 *     vb200_comm handle (peer pointers + signal pads)
 *   - bf16 = __nv_bfloat16 bit pattern (uint16_t) unless stated otherwise
 */
#ifndef VEOMNI_B200_H_
#define VEOMNI_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VB200_OK 0
#define VB200_EINVAL (-1)   /* bad argument / unsupported shape */
#define VB200_ECUDA (-2)    /* CUDA runtime error, see vb200_last_error() */
#define VB200_ESTATE (-3)   /* comm handle in wrong state */
#define VB200_ETIMEOUT (-4) /* peer signal wait exceeded its bound */

#define VB200_ABI_VERSION 1

/* ---- runtime ------------------------------------------------------------------------- */
int vb200_abi_version(void);
const char* vb200_last_error(void);
/* Number of kernels this library has launched in this process (bench.py "gpu_launches"). */
int64_t vb200_launch_count(void);
void vb200_reset_launch_count(void);

/* ---- RMSNorm --------------------------------------------------------------------------
 * Replaces OpSlot("rms_norm","standard") (veomni/ops/liger/__init__.py:28-59) i.e.
 * Qwen3RMSNorm.forward (veomni/models/transformers/qwen3/generated/
 * patched_modeling_qwen3_gpu.py:88-97):  y = w * bf16(x * rsqrt(mean(x^2) + eps)).
 * x,y: [rows, cols] bf16 row-major (cols % 8 == 0, cols <= 16384); w: [cols] bf16;
 * rstd: [rows] fp32 (saved for backward).                                                 */
int vb200_rmsnorm_fwd(const void* x, const void* w, void* y, float* rstd, int64_t rows, int64_t cols,
                      float eps, void* stream);
/* dx: [rows, cols] bf16; dw_partial: [vb200_rmsnorm_bwd_partials(rows, cols), cols] fp32
 * workspace; dw: [cols] fp32 = column sums (deterministic two-pass reduction).            */
int64_t vb200_rmsnorm_bwd_partials(int64_t rows, int64_t cols);
/* Fused residual add + RMSNorm (SURVEY.md §8(f)1, the `hidden_states = residual + hidden_states` line before every
 * Qwen3RMSNorm in the decoder layer, patched_modeling_qwen3_gpu.py:369-375).
 *   fwd: h_out = bf16(x + residual), y = RMSNorm(h_out) * w, rstd[rows];  cols in {1024, 2048, 4096, 5120, 8192}
 *   bwd: dx = rmsnorm_bwd(dy; x = h_out, w, rstd) + dres (bf16 sum), dw as vb200_rmsnorm_bwd; dres NULL = plain bwd */
int vb200_add_rmsnorm_fwd(const void* x, const void* residual, const void* w, void* h_out, void* y, float* rstd,
                          int64_t rows, int64_t cols, float eps, void* stream);
int vb200_rmsnorm_bwd_add(const void* dy, const void* x, const void* w, const float* rstd, const void* dres, void* dx,
                          float* dw_partial, float* dw, int64_t rows, int64_t cols, void* stream);
int vb200_rmsnorm_bwd(const void* dy, const void* x, const void* w, const float* rstd, void* dx,
                      float* dw_partial, float* dw, int64_t rows, int64_t cols, void* stream);

/* ---- RoPE -----------------------------------------------------------------------------
 * Replaces OpSlot("rotary_pos_emb","full") (patched_modeling_qwen3_gpu.py:208-223):
 *   out = x*cos + rotate_half(x)*sin  for q and k, cos/sin: [tokens, head_dim] bf16.
 * q,k are addressed as [tokens, heads, head_dim] with explicit element strides so both the
 * reference's transposed [B,H,S,D] views and packed [S,H,D] buffers work without a copy.
 * `inverse` != 0 applies the transposed rotation (the backward of the op).
 * head_dim in {64,128,256}; out may alias in (in-place).                                   */
int vb200_rope(const void* q_in, void* q_out, const void* k_in, void* k_out, const void* cos,
               const void* sin, int64_t tokens, int32_t q_heads, int32_t k_heads, int32_t head_dim,
               int64_t q_stride_tok, int64_t q_stride_head, int64_t k_stride_tok, int64_t k_stride_head,
               int64_t qo_stride_tok, int64_t qo_stride_head, int64_t ko_stride_tok,
               int64_t ko_stride_head, int32_t inverse, void* stream);

/* Fused q/k head RMSNorm + RoPE (Qwen3Attention.forward, patched_modeling_qwen3_gpu.py:305-310:
 * q_norm/k_norm over head_dim followed by apply_rotary_pos_emb) in one pass over q and k.
 * x: [tokens, heads, head_dim] bf16 contiguous, normalised per (token, head) with weight
 * wq/wk [head_dim]; rstd_{q,k}: [tokens, heads] fp32 saved for backward.                   */
int vb200_qknorm_rope_fwd(const void* q_in, const void* k_in, const void* wq, const void* wk,
                          const void* cos, const void* sin, void* q_out, void* k_out, float* rstd_q,
                          float* rstd_k, int64_t tokens, int32_t q_heads, int32_t k_heads,
                          int32_t head_dim, float eps, void* stream);
int vb200_qknorm_rope_bwd(const void* dq_out, const void* dk_out, const void* q_in, const void* k_in,
                          const void* wq, const void* wk, const void* cos, const void* sin,
                          const float* rstd_q, const float* rstd_k, void* dq_in, void* dk_in,
                          float* dw_partial, float* dwq, float* dwk, int64_t tokens, int32_t q_heads,
                          int32_t k_heads, int32_t head_dim, void* stream);
int64_t vb200_qknorm_rope_bwd_partials(int64_t tokens);

/* ---- SwiGLU ---------------------------------------------------------------------------
 * Replaces the elementwise part of OpSlot("swiglu_mlp","standard")
 * (veomni/ops/liger/__init__.py:119-142; eager: patched_modeling_qwen3_gpu.py:121-127):
 *   out = silu(gate) * up.  n elements bf16, n % 8 == 0.
 * gate/up/out are [rows, cols] with a row stride in elements so a merged [rows, 2*cols]
 * fc1 output (MoE: EPMergedFc1GroupGemm, veomni/distributed/moe/moe_layer.py:339-346) can be
 * consumed as two strided views.                                                           */
int vb200_swiglu_fwd(const void* gate, const void* up, void* out, int64_t rows, int64_t cols,
                     int64_t in_stride, int64_t out_stride, void* stream);
/* dgate = dout * up * dsilu(gate); dup = dout * silu(gate)                                 */
int vb200_swiglu_bwd(const void* dout, const void* gate, const void* up, void* dgate, void* dup,
                     int64_t rows, int64_t cols, int64_t in_stride, int64_t dout_stride,
                     int64_t dgrad_stride, void* stream);

/* ---- gradient clipping: multi-tensor L2 norm and in-place scale ---------------------------
 * Replaces the two passes of torch.nn.utils.clip_grad_norm_ under veomni_clip_grad_norm
 * (veomni/distributed/clip_grad_norm.py:7-20 -> fsdp2/clip_grad_norm.py:21-51 dense,
 * :73-153 expert groups): _foreach_norm over the local gradient shards and _foreach_mul_ by the
 * clip coefficient.  ptrs_dev / numels_dev: device arrays of n entries (an entry is a whole
 * tensor or a piece of one; keep entries <= 2^20 elements for balance); dtype 0 = bf16, 1 = f32.
 *   vb200_multi_sumsq : total[0] = sum over entries of sum(x^2)  (fp32, fixed reduction order);
 *                       per_entry (optional) [n] the per-entry sums; partials: workspace of
 *                       vb200_multi_sumsq_partials(n) floats.
 *   vb200_multi_scale : x *= *coef_dev for every entry; returns without touching memory when
 *                       *coef_dev == 1 (no clipping needed).                                  */
int64_t vb200_multi_sumsq_partials(int32_t n_entries);
int vb200_multi_sumsq(const void* const* ptrs_dev, const int64_t* numels_dev, int32_t n_entries, int32_t dtype,
                      float* partials, float* total, float* per_entry, void* stream);
int vb200_multi_scale(void* const* ptrs_dev, const int64_t* numels_dev, int32_t n_entries, int32_t dtype,
                      const float* coef_dev, void* stream);

/* AdamW step over a device table of entries (SURVEY.md §8(f)4: the reference builds torch.optim.AdamW(fused=True),
 * veomni/optim/optimizer.py:261-328).  Same arithmetic as PyTorch's fused kernel (ADAMW mode, no amsgrad / maximize) on
 * fp32 parameters and moments; gradients fp32 (grad_dtype 1) or bf16 (0); bias_correction1 = 1 - beta1^step,
 * bias_correction2_sqrt = sqrt(1 - beta2^step), computed by the caller.  grad_scale_dev (optional device scalar, e.g.
 * the gradient-clip coefficient) multiplies every gradient first.  lp_params_dev (optional): a second pointer table —
 * the updated parameter is also stored there rounded to bf16 (master-weight training without FSDP: the world_size-1
 * path of build_parallelize_model, veomni/distributed/torch_parallelize.py:438-443,465).                              */
int vb200_multi_adamw(void* const* params_dev, const void* const* grads_dev, void* const* exp_avgs_dev,
                      void* const* exp_avg_sqs_dev, void* const* lp_params_dev, const int64_t* numels_dev,
                      int32_t n_entries, int32_t grad_dtype, float lr, float beta1, float beta2, float eps,
                      float weight_decay, float bias_correction1, float bias_correction2_sqrt,
                      const float* grad_scale_dev, void* stream);

/* ---- softmax cross-entropy over the vocabulary ------------------------------------------
 * Replaces the arithmetic of eager_cross_entropy -> transformers fixed_cross_entropy
 * (veomni/ops/kernels/cross_entropy/eager.py:23-38) and of the liger fused-linear-cross-entropy
 * element kernel (veomni/ops/kernels/cross_entropy/liger.py) as bound by ForCausalLMLoss
 * (veomni/ops/kernels/cross_entropy/__init__.py:89-221).
 *   logits  [rows, vocab], dtype 0 = bf16, 1 = f32, row stride in elements
 *   labels  [rows] int64; rows with label == ignore_index contribute loss 0 and gradient 0
 *   loss_rows[r] = logsumexp(x_r) - x_r[label_r]   (fp32, natural log; may be NULL)
 *   lse[r]       = logsumexp(x_r): written when lse_given == 0 (may be NULL), read when lse_given != 0
 *                  (backward-only call: the max/sum pass is skipped)
 *   grad         = (softmax(x) - onehot(label)) * scale * (*scale_dev) * (*upstream), same dtype as
 *                  logits; NULL = forward only; may alias logits (in place). scale_dev / upstream are
 *                  optional device scalars (e.g. 1/valid-token-count and the incoming dLoss), so the
 *                  mean reduction needs no host synchronisation.                            */
int vb200_cross_entropy(const void* logits, int32_t dtype, int64_t rows, int64_t vocab, int64_t row_stride,
                        const int64_t* labels, int64_t ignore_index, float* loss_rows, float* lse,
                        int32_t lse_given, void* grad, int64_t grad_stride, float scale,
                        const float* scale_dev, const float* upstream, void* stream);
/* ---- per-token log-probs, entropy and top-k forward-KL distillation -------------------------
 * Replaces the arithmetic of _ChunkedLinearLogProbs (veomni/ops/kernels/cross_entropy/chunk_logprobs.py:126-268)
 * and _ChunkedLinearTopkDistill (chunk_topk_distill.py:79-326) on one logits chunk, as reached through
 * ForCausalLMLoss(return_log_probs=True) (__init__.py:130-177).
 *   logits [rows, vocab], dtype 0 = bf16, 1 = f32, row stride in elements; rows, vocab < 2^31
 *   x = round_dtype(logits / temperature) (a true division in fp32, then rounded: chunk_logprobs.py:173-176)
 *   lse[r] = logsumexp(x_r) (may be NULL); logp[r] = x_r[label_r] - lse[r]; entropy[r] = lse[r] - sum softmax(x_r) x_r
 *   k = 0: no distillation. 0 < k <= 1024: topk_ids [rows, k] int64, topk_logp [rows, k] (topk_dtype 0 = bf16,
 *   1 = f32) and   slp = x[id] - lse,  student_mass = sum exp(slp),  teacher_mass = sum exp(tlp),
 *                  distill = sum exp(tlp') (tlp' - slp'),  ' = max(., clamp) when has_clamp
 *   Every output is 0 where label == ignore_index; logp is NaN for a label outside [0, vocab).           */
int vb200_token_logprobs(const void* logits, int32_t dtype, int64_t rows, int64_t vocab, int64_t row_stride,
                         const int64_t* labels, int64_t ignore_index, float temperature, float* lse, float* logp,
                         float* entropy, int32_t k, const int64_t* topk_ids, const void* topk_logp, int32_t topk_dtype,
                         int32_t has_clamp, float clamp, float* distill, float* student_mass, float* teacher_mass,
                         void* stream);
/* Gradient of sum_r dlogp[r] logp[r] + dentropy[r] entropy[r] + ddistill[r] distill[r] w.r.t. the logits
 * (chunk_logprobs.py:230-258, chunk_topk_distill.py:252-313), written to grad (same dtype; may alias logits).
 * lse / entropy are the forward's outputs; each upstream pointer may be NULL (= 0). With p = softmax(x):
 *   g_v = dlogp (d(v=label) - p_v) - dentropy p_v (x_v - lse + entropy)
 *         + ddistill (teacher_mass_eff p_v - pt[v]),  pt[v] = sum_{k: id_k = v} exp(tlp'_k) [slp_k >= clamp],
 *   teacher_mass_eff = sum_v pt[v];  grad = round_dtype(round_dtype(g) / temperature).  0 at ignored rows. */
int vb200_token_logprobs_bwd(const void* logits, int32_t dtype, int64_t rows, int64_t vocab, int64_t row_stride,
                             const int64_t* labels, int64_t ignore_index, float temperature, const float* lse,
                             const float* entropy, const float* dlogp, const float* dentropy, const float* ddistill,
                             int32_t k, const int64_t* topk_ids, const void* topk_logp, int32_t topk_dtype,
                             int32_t has_clamp, float clamp, void* grad, int64_t grad_stride, void* stream);
/* out2[0] = 1 / count(labels != ignore_index) (0 if none), out2[1] = that count; device scalars. */
int vb200_count_valid_labels(const int64_t* labels, int64_t n, int64_t ignore_index, float* out2,
                             void* stream);

/* ---- packed (varlen) causal attention ---------------------------------------------------
 * Replaces flash_attn_varlen_func as called by flash_attention_forward
 * (veomni/ops/kernels/attention/__init__.py:304-320 through HF _flash_attention_forward's
 * padding-free branch): q [total, Hq, D], k/v [total, Hk, D] packed sequences delimited by
 * cu_seqlens (int32 [num_seqs+1], device), causal inside each sequence, GQA (Hq % Hk == 0),
 * D in {64,128}.  strides: int64 host array of (token stride, head stride) element pairs for
 * q,k,v,o (fwd: 8 values) and q,k,v,o,dout,dq,dk,dv (bwd: 16 values); last dim contiguous.
 * lse: [Hq, total] fp32 = log-sum-exp of scaled scores (natural log), consumed by the backward.
 * Backward is deterministic (no atomics): delta [Hq,total] fp32 workspace, then dq, dk, dv.  */
int vb200_attn_varlen_fwd(const void* q, const void* k, const void* v, void* o, float* lse,
                          const int32_t* cu_seqlens, int32_t num_seqs, int32_t max_seqlen, int32_t total,
                          int32_t q_heads, int32_t k_heads, int32_t head_dim, const int64_t* strides,
                          float scale, int32_t causal, void* stream);
/* Same contract as vb200_attn_varlen_fwd for head_dim == 128, on the tcgen05 tensor cores (TMEM-resident
 * S and PV tiles, softmax warps on tcgen05.ld).                                                   */
int vb200_attn_varlen_fwd_tc(const void* q, const void* k, const void* v, void* o, float* lse,
                             const int32_t* cu_seqlens, int32_t num_seqs, int32_t max_seqlen, int32_t total,
                             int32_t q_heads, int32_t k_heads, int32_t head_dim, const int64_t* strides,
                             float scale, int32_t causal, void* stream);
/* tcgen05 backward (head_dim 128): delta = rowsum(dO*O) first, then dq / dk / dv. strides: (token, head)
 * element strides of q, k, v, dout, dq, dk, dv (14 values). Deterministic (no atomics).           */
int vb200_attn_bwd_delta(const void* o, const void* dout, float* delta, int32_t total, int32_t q_heads,
                         int32_t head_dim, int64_t o_stride_tok, int64_t o_stride_head, int64_t do_stride_tok,
                         int64_t do_stride_head, void* stream);
int vb200_attn_varlen_bwd_tc(const void* q, const void* k, const void* v, const void* dout, const float* lse,
                             const float* delta, void* dq, void* dk, void* dv, const int32_t* cu_seqlens,
                             int32_t num_seqs, int32_t max_seqlen, int32_t total, int32_t q_heads, int32_t k_heads,
                             int32_t head_dim, const int64_t* strides, float scale, int32_t causal, void* stream);
/* Debugging aid (tools/attn_trace.py): with bit 13 of `causal` set, vb200_attn_varlen_bwd_tc records clock64 stamps of the
 * hand-offs of block 0 of the dQ kernel; this copies them out (8 events x 64 tiles of int64).                         */
int vb200_attn_debug_trace(int64_t* out512);
int vb200_attn_varlen_bwd(const void* q, const void* k, const void* v, const void* o, const void* dout,
                          const float* lse, float* delta, void* dq, void* dk, void* dv,
                          const int32_t* cu_seqlens, int32_t num_seqs, int32_t max_seqlen, int32_t total,
                          int32_t q_heads, int32_t k_heads, int32_t head_dim, const int64_t* strides,
                          float scale, int32_t causal, void* stream);

/* ---- peer-memory runtime (NVLink / NVSwitch) --------------------------------------------
 * One process per GPU. vb200_symm_alloc returns zeroed device memory that can be exported with
 * vb200_ipc_get_handle (64-byte opaque handle, exchanged by the host through torch.distributed)
 * and mapped by peers with vb200_ipc_open_handle.  vb200_comm_create takes, for every rank of the
 * group, the locally mapped base pointer of that rank's symmetric data region and signal pad
 * (vb200_comm_signal_bytes() bytes, zero-initialised); entries for `rank` itself are the local
 * allocations.  world <= 8.  Collectives use `channel` (0..31) as an independent epoch/flag
 * lane: calls on one channel must be issued in the same order on every rank.  `region_offset`
 * (256-byte aligned) is where THIS rank's buffer for the call lives inside its own region; it is
 * published to the peers with the ready flag, so offsets may differ between ranks.            */
int vb200_symm_alloc(void** ptr, int64_t bytes);
int vb200_symm_free(void* ptr);
int vb200_ipc_get_handle(const void* ptr, void* handle64);
int vb200_ipc_open_handle(const void* handle64, void** ptr);
int vb200_ipc_close_handle(void* ptr);
int64_t vb200_comm_signal_bytes(void);
int vb200_comm_create(void** comm, int32_t rank, int32_t world, void* const* peer_data,
                      void* const* peer_signal, int64_t data_bytes);
int vb200_comm_destroy(void* comm);
int vb200_comm_check(void* comm); /* VB200_ETIMEOUT if a peer wait ever timed out (synchronises) */
int vb200_comm_barrier(void* comm, int32_t channel, void* stream);

/* FSDP2 unit all-gather, replaces DefaultAllGather.__call__
 * (torch/distributed/fsdp/_fully_shard/_fsdp_collectives.py:81-95) behind
 * FSDPModule.set_custom_all_gather: rank p's shard (shard_bytes, any dtype) already sits at
 * region_offset + p*shard_bytes of its own symmetric region (FSDP's copy-in wrote it there);
 * on return every rank's region holds all N shards.                                          */
int vb200_allgather(void* comm, int32_t channel, int64_t region_offset, int64_t shard_bytes,
                    int32_t num_ctas, void* stream);
/* FSDP2 unit reduce-scatter, replaces DefaultReduceScatter.__call__ (:116-131) incl. the
 * AVG / pre-multiplied-SUM scaling (:701-759): every rank holds N chunks of chunk_elems fp32 at
 * region_offset; out[i] = scale * sum_{p=0..N-1} chunk_rank(p)[i], summed in rank order.      */
int vb200_reduce_scatter_f32(void* comm, int32_t channel, int64_t region_offset, int64_t chunk_elems,
                             float scale, float* out, int32_t num_ctas, void* stream);
/* Same reduce-scatter with bf16 inputs (N chunks of chunk_elems bf16 at region_offset), fp32 accumulation
 * in rank order and fp32 output: bit-identical to vb200_reduce_scatter_f32 on the fp32 copies of the same
 * gradients (bf16 -> fp32 is exact), at half the NVLink bytes.                                       */
int vb200_reduce_scatter_bf16(void* comm, int32_t channel, int64_t region_offset, int64_t chunk_elems,
                              float scale, float* out, int32_t num_ctas, void* stream);
/* Reduce-scatter copy-in, replaces foreach_reduce_scatter_copy_in -> torch._chunk_cat
 * (torch/distributed/fsdp/_fully_shard/_fsdp_collectives.py:667-675) for bf16 gradients WITHOUT the
 * conversion to the reduce dtype: out[r, off_p : off_p + chunk_p] = chunk r of parameter p
 * (dim-0 zero-padded to a multiple of world), bf16.  desc: host array of n x {src pointer, numel,
 * chunk elements, row offset}; src_dtype 0 = bf16, 1 = f32 (rounded to bf16).  With world = 1 and
 * f32 sources it is also the all-gather copy-in (all_gather_copy_in_cuda, :175-188): the fp32 master
 * shards cast into the bf16 all-gather input in one pass.                                            */
int vb200_fsdp_pack_bf16(const int64_t* desc, int32_t n, int32_t world, int64_t row_elems, void* out,
                         int32_t src_dtype, void* stream);
/* FSDP2 unit all-gather with the copy-out fused in: replaces DefaultAllGather.__call__ (:81-95) AND the
 * fsdp::split_with_sizes_copy of foreach_all_gather_copy_out (:196-212, :346-412). As for vb200_allgather, rank p's
 * shard row sits at region_offset + p*shard_bytes of its own region; table: host array of n x {byte offset of the
 * parameter inside a shard row, bytes of one rank's shard of it, destination pointer}: rank p's piece of parameter i
 * is pulled over NVLink straight into dst_i + p*bytes_i (the parameter's unsharded tensor, any local memory).       */
int vb200_allgather_scatter(void* comm, int32_t channel, int64_t region_offset, int64_t shard_bytes,
                            const int64_t* table, int32_t n, int32_t num_ctas, void* stream);
/* FSDP2 unit reduce-scatter with the copy-in fused in: replaces foreach_reduce_scatter_copy_in -> torch._chunk_cat
 * (:667-675), DefaultReduceScatter.__call__ (:116-131) and the divide (:701-759) for bf16 gradients reduced in fp32.
 * desc: host array of n x {gradient pointer (bf16, contiguous, local), numel, chunk elements = ceil(dim0/world)*inner};
 * row_elems = sum of chunks. Chunk p of every gradient (dim-0 zero-padded) is pushed to rank p's staging buffer
 * [world, row_elems] bf16 at region_offset of its region (slot = source rank); then
 * out[i] = scale * sum_{s=0..N-1} staging[s][i] in rank order, fp32.                                               */
int vb200_reduce_scatter_push_bf16(void* comm, int32_t channel, int64_t region_offset, const int64_t* desc, int32_t n,
                                   int64_t row_elems, float scale, float* out, int32_t num_ctas, void* stream);
/* Strided chunk exchange, replaces dist.all_to_all_single + the reshape/cat copies of
 * _all_to_all_single (veomni/distributed/sequence_parallel/ulysses.py:86-122).
 * desc: n_desc x 8 int64 = {src_off, src_rank_stride, src_row_stride, dst pointer,
 * dst_peer_stride, dst_row_stride, rows, seg_bytes} (bytes; all multiples of 16): for every peer p
 * and row, copy seg_bytes from p's buffer at src_off + rank*src_rank_stride + row*src_row_stride
 * to dst + p*dst_peer_stride + row*dst_row_stride.                                            */
int vb200_all_to_all(void* comm, int32_t channel, int64_t region_offset, int32_t n_desc, const int64_t* desc,
                     int32_t num_ctas, void* stream);
/* Variable-size block pull for the EP token exchange (veomni/distributed/moe/comm.py:36-42) and the uneven image-row
 * exchange (_AlltoAllRegion, veomni/distributed/sequence_parallel/ulysses.py:298-316):
 * chunks = device array of {int64 src_off, int64 dst_off, int64 bytes, int32 peer, int32 pad}.  */
int vb200_chunk_pull(void* comm, int32_t channel, int64_t region_offset, const void* chunks, int32_t nchunks,
                     void* dst, int32_t num_ctas, void* stream);

/* ---- MoE routing / permutation -----------------------------------------------------------
 * Replaces expert_histogram + `argsort(stable).argsort()` + moe_scatter / moe_gather of the fused
 * MoE path (veomni/ops/kernels/moe/group_gemm.py:277-345; kernels in
 * veomni/ops/kernels/moe/_kernels/kernel/moe.py:53-159,253-333).
 * expert_index: [num_slots] = flattened [tokens, topk] expert ids (int64 if index_is_int64 else int32).
 * splits[e] = tokens routed to e; cumsum = inclusive prefix sum of splits; scatter_index[i] = row of
 * slot i in the expert-sorted activation (stable: ties keep slot order) — integer-exact.
 * workspace: vb200_moe_route_workspace(num_slots, num_experts) bytes.                          */
int64_t vb200_moe_route_workspace(int64_t num_slots, int32_t num_experts);
int vb200_moe_route(const void* expert_index, int32_t index_is_int64, int64_t num_slots, int32_t num_experts,
                    int32_t* splits, int32_t* cumsum, int32_t* scatter_index, void* workspace, void* stream);
/* out[scatter_index[t,k], :] = x[t, :]; with w_in and w_out: also w_out[scatter_index[t,k]] = w_in[t,k];
 * with w_in only: the copied row is scaled by w_in[t,k] (bf16 rounding) — backward of the weighted
 * combine (veomni/distributed/moe/moe_utils.py:44-72).                                           */
int vb200_moe_scatter(const void* x, const int32_t* scatter_index, void* out, const void* w_in, void* w_out,
                      int64_t tokens, int32_t topk, int64_t hidden, void* stream);
/* out[t,:] = sum_k x[scatter_index[t,k],:] (fp32 accumulation in k order, one rounding); with
 * weights != NULL each row is first scaled by weights[t,k] and rounded to bf16 (EP combine,
 * veomni/distributed/moe/moe_utils.py:44-72).                                                  */
int vb200_moe_gather(const void* x, const int32_t* scatter_index, const void* weights, void* out, int64_t tokens,
                     int32_t topk, int64_t hidden, void* stream);
/* out[t,k] = <g[t,:], x[scatter_index[t,k],:]> (fp32): gradient of the weighted combine with respect to the routing
 * weights (autograd of veomni/distributed/moe/moe_utils.py:44-72, `unpermute` with `probs`). hidden: multiple of 256.   */
int vb200_moe_weight_grad(const void* g, const void* x, const int32_t* scatter_index, float* out, int64_t tokens,
                          int32_t topk, int64_t hidden, void* stream);

/* ---- ragged MoE GroupGEMM (tcgen05 tensor cores) ------------------------------------------
 * Replaces group_gemm_same_nk / group_gemm_same_mn
 * (veomni/ops/kernels/moe/_kernels/kernel/group_gemm.py:157-234, 357-397).  bf16 in, fp32 accumulate,
 * bf16 out.  cumsum: int32 [num_groups] inclusive row prefix (device).  total_rows = rows of `a`.
 *   mode 0 (NT, transpose_b=True):  c[rows g] = a[rows g] (x k) * b[g]^T,  b [G, n, k]
 *   mode 1 (NN, transpose_b=False): c[rows g] = a[rows g] (x k) * b[g],    b [G, k, n]
 *   mode 2 (TN, same_mn wgrad):     c[g] (m x n) = a[rows g]^T * b[rows g], a [rows, m], b [rows, n];
 *                                   zero-filled when the group is empty.
 * m, n, k multiples of 8.  Rows of c past cumsum[G-1] are not written.                          */
int vb200_group_gemm(int32_t mode, const void* a, const void* b, void* c, const int32_t* cumsum,
                     int32_t num_groups, int64_t total_rows, int32_t m, int32_t n, int32_t k, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VEOMNI_B200_H_ */
