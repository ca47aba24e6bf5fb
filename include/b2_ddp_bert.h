/* b2_ddp_bert.h — C ABI of libb2ddpbert.so: the sm_100a kernels behind the DDP BERT fine-tuning step.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference (taishan1994/pytorch-distributed-NLP) has no
 * native code; the work these entry points replace is issued by third-party Python modules that
 * `multi-gpu-distributed-cls.py` drives.  Each declaration cites the reference-side call it stands in for
 * (paths relative to the reference tree, or `SP/` = site-packages of the pinned dependencies).
 *
 * Conventions
 *   - plain C: device pointers (borrowed; the library never allocates tensors), int64 sizes, explicit stream
 *     (`cudaStream_t` passed as void*).  No torch types.  No CPU fallback of any kind.
 *   - every function returns 0 on success, negative on error; `b2_last_error()` returns a thread-local message.
 *     The Python host turns a non-zero status into `RuntimeError(b2_last_error())`.
 *   - re-entrant: forward runs on the main thread, backward / DDP hooks on the autograd thread.
 *   - bf16 activations / weights / gradients, fp32 accumulation and statistics, fp32 master weights and
 *     AdamW moments.
 */
#ifndef B2_DDP_BERT_H_
#define B2_DDP_BERT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------------ */
/* library                                                                                                */
/* ------------------------------------------------------------------------------------------------------ */
const char* b2_last_error(void);
int32_t b2_abi_version(void);             /* bumped when a struct below changes */
#define B2_ABI_VERSION 18
int64_t b2_launch_count(void);            /* kernels launched by this library so far (process-wide) */

/* ------------------------------------------------------------------------------------------------------ */
/* GEMM (tcgen05 + TMA)                                                                                   */
/*   replaces: cuBLAS addmm issued by SP/transformers/models/bert/modeling_bert.py:179-181 (Q,K,V),       */
/*   :295 (attention output dense), :340 (intermediate dense), :353 (output dense) and the dgrad/wgrad    */
/*   GEMMs autograd runs for them inside `loss.backward()` (multi-gpu-distributed-cls.py:173).            */
/* ------------------------------------------------------------------------------------------------------ */
enum { B2_MAJOR_K = 0, B2_MAJOR_MN = 1 };
enum {
  B2_EPI_NONE = 0,                  /* D = acc                                  (dgrad / wgrad)               */
  B2_EPI_BIAS = 1,                  /* D = acc + bias[n]                        (QKV projection)              */
  B2_EPI_BIAS_GELU = 2,             /* aux_out = acc + bias; D = gelu_erf(aux_out)   (BertIntermediate)       */
  B2_EPI_BIAS_DROPOUT_RESIDUAL = 3, /* D = dropout(acc + bias) + aux_in         (BertSelfOutput / BertOutput) */
  B2_EPI_RESIDUAL = 4,              /* D = acc + aux_in                         (dgrad joining a residual)    */
  B2_EPI_GELU_BWD = 5,              /* D = acc * gelu_erf'(aux_in)              (dgrad through GELU)          */
  B2_EPI_RESIDUAL_F32 = 6,          /* D(fp32) = acc + aux_in(fp32); ldd / ld_aux_in count fp32 elements      */
  B2_EPI_ACCUM_F32 = 7,             /* D(fp32) += acc (vector reductions at L2; D holds the residual stream;   */
                                    /* split-K slices add in place, summation order unspecified)               */
  B2_EPI_PARTIAL_F32 = 100          /* internal: split-K partials                                           */
};

typedef struct b2_gemm_args {
  int64_t M, N, K;        /* D is [M,N]; K is the contraction length                                         */
  const void* A;          /* bf16. a_major K : A[m*lda + k];  MN : A[k*lda + m]                              */
  int64_t lda;
  int32_t a_major;
  const void* B;          /* bf16. b_major K : B[n*ldb + k];  MN : B[k*ldb + n]                              */
  int64_t ldb;
  int32_t b_major;
  void* D;                /* bf16 [M, ldd]                                                                   */
  int64_t ldd;
  int32_t epilogue;
  const void* bias;       /* bf16 [N] or NULL                                                                */
  const void* aux_in;     /* bf16 [M, ld_aux_in]: residual (3,4) or saved pre-activation (5)                 */
  int64_t ld_aux_in;
  void* aux_out;          /* bf16 [M, ld_aux_out]: pre-activation saved by (2)                               */
  int64_t ld_aux_out;
  float dropout_p;        /* (3) only                                                                        */
  const void* rng_state;  /* device uint64[2] = {seed, step}; see b2_rng_*                                   */
  uint32_t rng_site;      /* distinct per dropout site                                                       */
  void* workspace;        /* fp32 scratch for split-K (may be NULL -> never split)                           */
  int64_t workspace_bytes;
  int32_t force_bn;       /* 0 = auto, else 128 / 192 / 256 (tests, tuning)                                  */
  int32_t force_splits;   /* 0 = auto, else >= 1                                                             */
  int32_t force_kernel;   /* 0 = auto, 1 = single-CTA 128xBN kernel, 2 = CTA-pair (cta_group::2) 256xBN kernel        */
  void* debug_timing;     /* NULL, or device int64[grid][8]: clock64 phase stamps (CTA-pair GEMM, b2_gemm_ln_fwd)    */
  float* colsum_out;      /* NULL, or fp32 [N]: += column sums of the (bf16-rounded) output D, by atomic add        */
} b2_gemm_args_t;

int32_t b2_gemm_bf16(const b2_gemm_args_t* args, void* stream);

/* `count` independent problems behind one launch where they allow it (all TN = both operands MN-major, plain bf16
 * output, N % 256 == 0, one K; at most 4): the four weight-gradient GEMMs of an encoder layer (autograd's
 * addmm backward nodes for BertSelfAttention/BertSelfOutput/BertIntermediate/BertOutput, modeling_bert.py:179-356).
 * Other mixes are issued one by one; results are identical either way.                                         */
int32_t b2_gemm_bf16_grouped(const b2_gemm_args_t* args, int32_t count, void* stream);

/* BertSelfOutput.forward / BertOutput.forward in ONE launch (SP/transformers/models/bert/modeling_bert.py:294-298,
 * :352-356): y = LayerNorm(dropout(x W^T + b) + residual).  `args` as for b2_gemm_bf16 with epilogue
 * B2_EPI_BIAS_DROPOUT_RESIDUAL, NT layouts, N = hidden in {768, 1024} -- EXCEPT that args->aux_in is the residual as
 * FP32 [M, N] (ld_aux_in in elements): the residual stream stays in fp32 end to end.  D receives the pre-LayerNorm sum
 * rounded to bf16 (kept for the backward), y the normalised output as bf16 (the next GEMM's operand), y_f32 (optional)
 * the same as fp32 (the next block's residual), mean / rstd (fp32 [M]) the row statistics -- computed from the
 * UNROUNDED fp32 sum.  A row's N columns are spread over a cluster of N / 256 CTA pairs; the row statistics travel
 * through distributed shared memory.
 * b2_gemm_ln_max_clusters(hidden): how many such clusters the device can hold at once (0 = shape / device not
 * supported: issue b2_gemm_bf16 + b2_layernorm_fwd instead).                                                    */
int32_t b2_gemm_ln_fwd(const b2_gemm_args_t* args, const void* gamma, const void* beta, float eps, void* y,
                       int64_t ldy, float* y_f32, int64_t ldyf, float* mean, float* rstd, void* stream);
int32_t b2_gemm_ln_max_clusters(int64_t hidden);

/* ------------------------------------------------------------------------------------------------------ */
/* memory-bound kernels                                                                                   */
/* ------------------------------------------------------------------------------------------------------ */

/* BertEmbeddings.forward (SP/transformers/models/bert/modeling_bert.py:72-112): word + position + token-type
 * gather, add, LayerNorm(eps), dropout.  ids are the int64 tensors the reference's Collate produces
 * (multi-gpu-distributed-cls.py:88-97).  Writes y (bf16 [rows,H]), the pre-LN sum (bf16, for backward),
 * mean/rstd (fp32 [rows]) and ids32/tt32 (int32 copies used by the backward scatter).                      */
int32_t b2_embed_fwd(const int64_t* input_ids, const int64_t* token_type_ids, int64_t batch, int64_t seq,
                     const void* word_emb, const void* pos_emb, const void* type_emb, const void* gamma,
                     const void* beta, int64_t hidden, int64_t vocab, int64_t type_vocab, float eps, float dropout_p,
                     const void* rng_state, uint32_t rng_site, void* y, float* y_f32 /* optional fp32 copy of y: first residual of the fp32 stream */, void* pre_ln, float* mean, float* rstd,
                     int32_t* ids32, int32_t* tt32, void* stream);

/* arms the owner table used by b2_embed_bwd (int32[vocab] = INT_MAX); call once after allocation */
int32_t b2_embed_owner_init(int32_t* owner, int64_t vocab, void* stream);

/* backward of the above: LN backward, then the three scatter-adds (deterministic: one owner CTA per touched
 * vocabulary row sums its duplicates in token order).  d_word must be zeroed by the caller (b2_zero).  The row
 * `pad_token_id` gets no gradient (nn.Embedding padding_idx semantics, modeling_bert.py:58).                 */
int32_t b2_embed_bwd(const void* dy /* bf16, or fp32 when dy_fp32 */, int32_t dy_fp32, const void* pre_ln, const float* mean, const float* rstd, const void* gamma,
                     const int32_t* ids32, const int32_t* tt32, int64_t batch, int64_t seq, int64_t hidden,
                     int64_t vocab, int64_t type_vocab, int64_t pad_token_id /* -1: none */, float dropout_p,
                     const void* rng_state, uint32_t rng_site, void* d_word, void* d_pos, void* d_type, void* d_gamma, void* d_beta, void* scratch_dx,
                     float* scratch_partials, int64_t scratch_partials_bytes, int32_t* owner, void* stream);

/* LayerNorm over the last dim (BertSelfOutput / BertOutput LayerNorm, modeling_bert.py:297,355).
 * x is the already-summed (dropout(dense)+residual) input produced by the GEMM epilogue.                   */
int32_t b2_layernorm_fwd(const void* x, const void* gamma, const void* beta, int64_t rows, int64_t hidden,
                         float eps, void* y, float* mean, float* rstd, void* stream);

/* LayerNorm backward.  dy: grad wrt LN output.  Produces
 *   dx        grad wrt LN input (goes to the residual branch),
 *   dx_drop   dx * dropout-mask / (1-p) of the dense output that fed this LN (NULL when p == 0: use dx),
 *   d_gamma, d_beta, d_bias (bias grad of that dense = column sums of dx_drop)  — all bf16 [hidden].
 * `dy_add` (optional) is added to dy first (second consumer of the LN output, e.g. a residual path).       */
int32_t b2_layernorm_bwd(const void* dy, const void* dy_add, const void* x, const float* mean, const float* rstd,
                         const void* gamma, int64_t rows, int64_t hidden, float dropout_p, const void* rng_state,
                         uint32_t rng_site, int32_t grad_fp32 /* 1: dy, dy_add, dx are fp32 (dx_drop stays bf16 and
                         is then always written: it is what the GEMMs consume) */,
                         void* dx, void* dx_drop, void* d_gamma, void* d_beta, void* d_bias,
                         float* scratch_partials, int64_t scratch_partials_bytes,
                         int32_t* deferred_nparts /* host pointer or NULL.  NULL: d_gamma/d_beta/d_bias are final in
                         stream order.  Else only the per-block partials are written, *deferred_nparts receives their
                         count and the caller finishes with b2_colsum_finish (takes the reduction off the critical
                         path, e.g. onto another stream) */,
                         void* stream);

/* The training engine's form of b2_layernorm_bwd (fp32 gradient stream: dy fp32 in, dx fp32 out, dx_drop bf16 out,
 * dropout mask on the input branch): the three column-sum sets are ADDED into accum (fp32 [3][hidden]: d_gamma,
 * d_beta, d_bias) instead of going through partials + b2_colsum_finish; the caller converts them with
 * b2_accum_finish.                                                                                             */
int32_t b2_layernorm_bwd_accum(const float* dy, const void* x, const float* mean, const float* rstd,
                               const void* gamma, int64_t rows, int64_t hidden, float dropout_p,
                               const void* rng_state, uint32_t rng_site, float* dx, void* dx_drop, float* accum,
                               void* stream);

/* partials [nparts][nsets][cols] fp32 -> up to three bf16 [cols] outputs (the second half of b2_layernorm_bwd) */
int32_t b2_colsum_finish(const float* partials, int32_t nparts, int32_t nsets, int64_t cols, void* out0, void* out1,
                         void* out2, void* stream);

/* column sums of a bf16 [rows, cols] matrix -> bf16 [cols]   (bias gradients of QKV / intermediate dense)  */
int32_t b2_colsum(const void* x, int64_t rows, int64_t cols, int64_t ldx, void* out, float* scratch_partials,
                  int64_t scratch_partials_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------ */
/* attention (BertSelfAttention core, modeling_bert.py:115-140 eager_attention_forward + :206 head merge)    */
/*   qkv  bf16 [batch*seq, 3*hidden]  (Q | K | V column blocks, heads of 64 inside each)                    */
/*   mask int64 [batch, seq] of {0,1} as produced by the reference Collate, or NULL (= all ones)            */
/*   ctx  bf16 [batch*seq, hidden]    lse fp32 [batch, heads, seq]                                          */
/*   keep_bits  NULL, or uint64 [batch, heads, seq, seq/64]: cache of the forward's dropout decisions; used  */
/*              (written by fwd, read by bwd instead of regenerating Philox) when seq == 128 and dropout_p > 0,*/
/*              ignored otherwise.  Pass the same buffer to both calls of a step, or NULL to both.            */
/* ------------------------------------------------------------------------------------------------------ */
int32_t b2_attention_fwd(const void* qkv, const int64_t* attention_mask, int64_t batch, int64_t seq,
                         int64_t heads, int64_t head_dim, float dropout_p, const void* rng_state,
                         uint32_t rng_site, void* ctx, float* lse, uint64_t* keep_bits, void* stream);
int32_t b2_attention_bwd(const void* qkv, const int64_t* attention_mask, const void* ctx, const void* d_ctx,
                         const float* lse, int64_t batch, int64_t seq, int64_t heads, int64_t head_dim,
                         float dropout_p, const void* rng_state, uint32_t rng_site, void* d_qkv,
                         float* dq_accum /* fp32 [batch*seq, hidden], only for seq > 128 */,
                         float* dbias_accum /* NULL, or fp32 [3*hidden]: += column sums of d_qkv (QKV bias grad) */,
                         const uint64_t* keep_bits, void* stream);

/* ------------------------------------------------------------------------------------------------------ */
/* head: BertPooler (modeling_bert.py:462-468) + dropout + classifier (:1123-1124) + CrossEntropyLoss       */
/*   (multi-gpu-distributed-cls.py:169,343).  fp32 logits/loss as the reference exposes them.               */
/* ------------------------------------------------------------------------------------------------------ */
int32_t b2_head_fwd(const void* hidden_states /* bf16 [batch*seq, hidden] */, int64_t batch, int64_t seq,
                    int64_t hidden, const void* pool_w, const void* pool_b, const void* cls_w, const void* cls_b,
                    int64_t num_labels, float dropout_p, const void* rng_state, uint32_t rng_site,
                    void* pooled /* bf16 [batch, hidden] */, float* logits /* [batch, num_labels] */,
                    void* stream);
/* mean cross-entropy and d(loss)/d(logits); labels int64 [batch]; loss_scale multiplies dlogits (DDP: 1)    */
int32_t b2_ce_fwd_bwd(const float* logits, const int64_t* labels, int64_t batch, int64_t num_labels,
                      float* loss /* scalar */, float* dlogits /* [batch, num_labels] or NULL */, void* stream);
/* backward of b2_head_fwd: from dlogits to d(hidden_states[:,0]) and the four head parameter grads (bf16)  */
int32_t b2_head_bwd(const float* dlogits, const void* hidden_states, const void* pooled, int64_t batch,
                    int64_t seq, int64_t hidden, const void* pool_w, const void* cls_w, int64_t num_labels,
                    float dropout_p, const void* rng_state, uint32_t rng_site, void* d_pool_w, void* d_pool_b,
                    void* d_cls_w, void* d_cls_b, void* d_hidden /* [batch*seq, hidden], rows != CLS zeroed */,
                    int32_t d_hidden_fp32 /* 0: bf16, 1: fp32 */, float* scratch /* fp32 [2, batch, hidden] */,
                    void* stream);

/* ------------------------------------------------------------------------------------------------------ */
/* packed bins (SURVEY.md §8 f3): the reference tokenises with padding="max_length" (multi-gpu-distributed-cls.py */
/* :76) although its rows average 18 of 128 tokens.  The host packs the valid prefixes of several sequences into  */
/* 128-token bins (pytorch-distributed-nlp_b200/packing.py); these variants of the entry points above take        */
/*   position_ids  int64 [bins * 128]   position of every token inside its own sequence                           */
/*   segments      int32 [bins * 128]   lo | hi << 16: the row may attend to rows [lo, hi) of its bin only        */
/*   cls_rows      int64 [batch]        flat row of every sequence's first token (what the pooler reads)          */
/* Everything else (GEMMs, LayerNorm, GELU) is token-wise and simply runs on bins * 128 rows.                     */
/* ------------------------------------------------------------------------------------------------------ */
int32_t b2_embed_fwd_packed(const int64_t* input_ids, const int64_t* token_type_ids, const int64_t* position_ids,
                            int64_t max_positions, int64_t bins, int64_t seq, const void* word_emb,
                            const void* pos_emb, const void* type_emb, const void* gamma, const void* beta,
                            int64_t hidden, int64_t vocab, int64_t type_vocab, float eps, float dropout_p,
                            const void* rng_state, uint32_t rng_site, void* y, float* y_f32, void* pre_ln, float* mean,
                            float* rstd, int32_t* ids32, int32_t* tt32, int32_t* pos32, void* stream);
int32_t b2_embed_bwd_packed(const void* dy, int32_t dy_fp32, const void* pre_ln, const float* mean, const float* rstd,
                            const void* gamma, const int32_t* ids32, const int32_t* tt32, const int32_t* pos32,
                            int64_t bins, int64_t seq, int64_t hidden, int64_t vocab, int64_t type_vocab,
                            int64_t pad_token_id, float dropout_p, const void* rng_state, uint32_t rng_site,
                            void* d_word, void* d_pos, void* d_type, void* d_gamma, void* d_beta, void* scratch_dx,
                            float* scratch_partials, int64_t scratch_partials_bytes, int32_t* owner, void* stream);
int32_t b2_attention_fwd_packed(const void* qkv, const int32_t* segments, int64_t bins, int64_t heads,
                                int64_t head_dim, float dropout_p, const void* rng_state, uint32_t rng_site,
                                void* ctx, float* lse, uint64_t* keep_bits, void* stream);
int32_t b2_attention_bwd_packed(const void* qkv, const int32_t* segments, const void* ctx, const void* d_ctx,
                                const float* lse, int64_t bins, int64_t heads, int64_t head_dim, float dropout_p,
                                const void* rng_state, uint32_t rng_site, void* d_qkv, float* dbias_accum,
                                const uint64_t* keep_bits, void* stream);
int32_t b2_head_fwd_packed(const void* hidden_states, const int64_t* cls_rows, int64_t batch, int64_t hidden,
                           const void* pool_w, const void* pool_b, const void* cls_w, const void* cls_b,
                           int64_t num_labels, float dropout_p, const void* rng_state, uint32_t rng_site,
                           void* pooled, float* logits, void* stream);
int32_t b2_head_bwd_packed(const float* dlogits, const void* hidden_states, const void* pooled,
                           const int64_t* cls_rows, int64_t tokens, int64_t batch, int64_t hidden,
                           const void* pool_w, const void* cls_w, int64_t num_labels, float dropout_p,
                           const void* rng_state, uint32_t rng_site, void* d_pool_w, void* d_pool_b, void* d_cls_w,
                           void* d_cls_b, void* d_hidden, int32_t d_hidden_fp32, float* scratch, void* stream);

/* b2_head_bwd / b2_head_bwd_packed (cls_rows NULL: row of sequence b = b * seq) with the two parameter-gradient
 * kernels launched on `weight_stream` (ordered behind the data-gradient part by an event; the same stream when NULL): they
 * are off the critical path of the backward.  Whatever reads the four head gradients must be ordered behind
 * `weight_stream`.                                                                                               */
int32_t b2_head_bwd_split(const float* dlogits, const void* hidden_states, const void* pooled,
                          const int64_t* cls_rows, int64_t tokens, int64_t batch, int64_t seq, int64_t hidden,
                          const void* pool_w, const void* cls_w, int64_t num_labels, float dropout_p,
                          const void* rng_state, uint32_t rng_site, void* d_pool_w, void* d_pool_b, void* d_cls_w,
                          void* d_cls_b, void* d_hidden, int32_t d_hidden_fp32, float* scratch, void* stream,
                          void* weight_stream);

/* ------------------------------------------------------------------------------------------------------ */
/* optimizer + gradient exchange                                                                          */
/*   replaces: HF AdamW.step (transformers 4.28.1 optimization.py, built at multi-gpu-distributed-cls.py    */
/*   :100-111, stepped :174), optimizer.zero_grad (:172), and the DDP Reducer's bucket all-reduce            */
/*   (SP/torch/nn/parallel/distributed.py:1255-1280, reducer.hpp:276-286) for world > 1.                     */
/* ------------------------------------------------------------------------------------------------------ */
typedef struct b2_adamw_hparams {
  double lr, beta1, beta2, eps, weight_decay; /* python doubles, rounded to fp32 the way torch rounds them */
  int32_t correct_bias;
  /* optional DEVICE pointer to the fp32 loss scale of a torch.cuda.amp.GradScaler (the reference's -amp scripts,
   * multi-gpu-distributed-mp-amp-cls.py:160-171): gradients are divided by *grad_scale before the update.
   * NULL = unscaled gradients.                                                                                */
  const float* grad_scale;
  /* optional DEVICE pointer to the GradScaler's fp32 inf/nan indicator: a non-zero value skips the update (and the
   * step count), as GradScaler.step() skips optimizer.step().  NULL = always update.                            */
  const float* found_inf;
  /* optional DEVICE uint8 per 8-element vector (indexed like decay_flags): non-zero = this vector was already
   * updated elsewhere (b2_gemm_bf16_grouped_adamw) and is skipped.  NULL = update everything in [begin, end).     */
  const uint8_t* skip_flags;
} b2_adamw_hparams_t;

/* The layer's weight gradients AND their HF-AdamW update in one launch (single-GPU step: no exchange between the
 * gradient and the update): b2_gemm_bf16_grouped whose epilogue, for every output element, rounds the gradient to
 * bf16 (still written to D_i), updates exp_avg / exp_avg_sq / the fp32 master weight of the same element in place
 * and writes the bf16 shadow weight.  targets[i] addresses the optimizer state of problem i's [M_i, N_i] block
 * (row pitch = args[i].ldd elements); decay != 0 applies hp->weight_decay.  Same arithmetic as
 * b2_bucket_reduce_adamw; hp->grad_scale / found_inf must be NULL.  The problems must be groupable (see
 * b2_gemm_bf16_grouped) -- this entry point fails instead of falling back.                                       */
typedef struct b2_fused_adamw_target {
  float* master;
  float* exp_avg;
  float* exp_avg_sq;
  void* shadow; /* bf16 */
  int32_t decay;
} b2_fused_adamw_target_t;
int32_t b2_gemm_bf16_grouped_adamw(const b2_gemm_args_t* args, const b2_fused_adamw_target_t* targets, int32_t count,
                                   const b2_adamw_hparams_t* hp, const int64_t* step_counter, void* stream);

/* Fused update of one contiguous slice [begin, end) (element indices, multiples of 8) of the flat parameter
 * space.  world == 1: grads read from `grad_local`.  world > 1: element-wise mean over `peer_grads[0..world)`
 * (peer-mapped bf16 buffers, fixed rank order => bit-identical on every rank), then the HF AdamW update on the
 * fp32 master / moments, then the bf16 shadow weights are stored to every non-NULL `peer_shadow[r]`
 * (peer_shadow[rank] must be set; NULL elsewhere = that peer's copy travels by b2_copy_async).
 * decay_flags: uint8 per 8-element vector (1 = apply weight decay).  step_counter: device int64, read here
 * (t = *step_counter + 1 for the bias correction); bumped separately by b2_step_advance.                     */
int32_t b2_bucket_reduce_adamw(const void* const* peer_grads, void* const* peer_shadow, int32_t world,
                               int32_t rank, float* master, float* exp_avg, float* exp_avg_sq,
                               const uint8_t* decay_flags, int64_t begin, int64_t end,
                               const b2_adamw_hparams_t* hp, const int64_t* step_counter, void* stream);

/* Single-GPU background form of the same update (world == 1, no GradScaler state): blocks of 128 threads x 32
 * registers and no shared memory, i.e. shaped to become resident BESIDE a 640-thread GEMM CTA instead of waiting for the
 * gaps between GEMM kernels; launched per bucket on the optimizer stream while the backward pass is still running.
 * `step_size` = the bias-corrected step of this update, a device float written by b2_adamw_prepare (lr * sqrt(1 - b2^t)
 * / (1 - b1^t), t = *step_counter + 1, in double like the host would); call b2_adamw_prepare once per step, after
 * b2_step_advance.  Same arithmetic as b2_bucket_reduce_adamw.                                                  */
int32_t b2_adamw_prepare(const b2_adamw_hparams_t* hp, const int64_t* step_counter, float* step_size, void* stream);
int32_t b2_adamw_background(const void* grads, void* shadow, float* master, float* exp_avg, float* exp_avg_sq,
                            const uint8_t* decay_flags, int64_t begin, int64_t end, const b2_adamw_hparams_t* hp,
                            const float* step_size, void* stream);

/* ++step (AdamW t) and ++rng step (dropout stream) on the device: keeps CUDA-graph replays stateful.
 * found_inf (optional device fp32, see b2_adamw_hparams_t): non-zero leaves the AdamW step count untouched.   */
int32_t b2_step_advance(int64_t* step_counter, void* rng_state, const float* found_inf, void* stream);
int32_t b2_rng_seed(void* rng_state, uint64_t seed, uint64_t step, void* stream);

/* segments[i] = {src element offset in `src` (fp32), dst element offset in `dst` (bf16), count}: dst <- bf16(src), then
 * src <- 0.  One launch turns the per-step fp32 bias-gradient accumulators (filled by atomics from the GEMM and
 * attention-backward epilogues) into bf16 gradients and re-arms them.                                           */
int32_t b2_accum_finish(float* src, void* dst, const int64_t* segments /* device [n][3] */, int64_t n_segments,
                        int64_t max_count, void* stream);

/* Gradient accumulation over [begin, end) of the flat space (multiples of 8).
 * mode 0 (ADD):    acc[e] += scale * float(grads[e])
 * mode 1 (FINISH): grads[e] = bf16(acc[e] + scale * float(grads[e])); acc[e] = 0
 * acc fp32, grads bf16 (this micro-batch's gradient, as the backward left it).  128-thread blocks of at most 32
 * registers and no shared memory: shaped like b2_adamw_background to run per bucket beside the backward's GEMMs. */
#define B2_ACCUM_ADD 0
#define B2_ACCUM_FINISH 1
int32_t b2_grad_accumulate(float* acc, void* grads, int64_t begin, int64_t end, float scale, int32_t mode,
                           void* stream);

/* bf16 <- fp32 cast of a flat range (initial shadow weights, load_state_dict) and zero fill                 */
int32_t b2_cast_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream);
int32_t b2_cast_bf16_to_f32(const void* src, float* dst, int64_t n, void* stream);
int32_t b2_zero(void* dst, int64_t bytes, void* stream);
/* stream-ordered device-to-device copy; with an IPC-mapped peer pointer on one side it is a copy-engine transfer
 * over NVLink (the DMA form of the gradient exchange: peers' slices in, updated bf16 weights out)             */
int32_t b2_copy_async(void* dst, const void* src, int64_t bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------ */
/* peer memory over NVLink / NVSwitch (one process per GPU; handles exchanged by the host through           */
/* torch.distributed).  replaces dist.all_reduce / all_gather / barrier call sites                          */
/* (multi-gpu-distributed-cls.py:141,148,153,171) on the step path.                                          */
/* ------------------------------------------------------------------------------------------------------ */
#define B2_IPC_HANDLE_BYTES 64
int32_t b2_comm_alloc(int64_t bytes, void** ptr);                       /* cudaMalloc'ed, IPC-exportable     */
int32_t b2_comm_free(void* ptr);
int32_t b2_comm_export(void* ptr, uint8_t handle[B2_IPC_HANDLE_BYTES]);
int32_t b2_comm_import(const uint8_t handle[B2_IPC_HANDLE_BYTES], void** ptr);
int32_t b2_comm_unimport(void* ptr);

/* Device-side barrier across ranks through flag words in each rank's signal pad.
 * peer_flags[r] points at rank r's pad (uint32[world * B2_FLAG_SLOTS]); `slot` selects the flag family; `epoch` is a
 * device counter incremented by the kernel so graph replays stay in lock-step.  Bounded spin -> trap.       */
#define B2_FLAG_SLOTS 64
int32_t b2_peer_barrier(void* const* peer_flags, int32_t world, int32_t rank, int32_t slot, uint32_t* epoch,
                        void* stream);

/* Trainer.output_reduce (multi-gpu-distributed-cls.py:145-155): every rank stores its [rows, row_bytes] block
 * into slot `rank` of every peer's gather buffer, then a barrier.                                           */
int32_t b2_allgather_rows(const void* src, int64_t bytes, void* const* peer_dst, void* const* peer_flags,
                          int32_t world, int32_t rank, int32_t slot, uint32_t* epoch, void* stream);
/* Trainer.loss_reduce (:139-143): mean of one fp32 scalar over ranks                                        */
int32_t b2_scalar_allreduce_mean(const float* src, float* dst, float* const* peer_scratch,
                                 void* const* peer_flags, int32_t world, int32_t rank, int32_t slot,
                                 uint32_t* epoch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2_DDP_BERT_H_ */
