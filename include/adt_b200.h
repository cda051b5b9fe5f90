/* libadt_b200.so -- C ABI of the B200-native ADT hot path (SASRec-ADT training step + full-catalog eval).
 *
 * The reference (defineZYP/ADT) is pure Python/PyTorch and has no FFI layer of its own; the seam it offers is
 * the torch.nn.Module (`SASRecADT.forward/predict`, /root/reference/sasrec/model.py:67-97) plus the loss /
 * optimiser lines of its training loop (/root/reference/sasrec/main.py:146-173).  Each entry point below
 * replaces the span of reference code it cites; `adt_b200/model.py` binds them with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (fp32 activations/weights, int32 ids), 16-byte aligned;
 *   - activations are row-major [M = B*L, H]; H % 4 == 0, H <= 256, (H/nh) % 4 == 0, L <= 256, nh <= 8; longer sequences (L <= 2048)
 *     and wider rows (256 < H <= 512: precision 1, H % 64 == 0, H/nh a multiple of 32 up to 128) as stated where they apply;
 *   - all calls are asynchronous on `stream` (a cudaStream_t), never synchronise, allocate nothing;
 *   - return 0 on success, a negative ADT_E_* otherwise; adt_last_error() gives the thread-local message;
 *   - gradient buffers are ACCUMULATED into (+=, atomics) unless stated: zero them once per step.
 */
#ifndef ADT_B200_H
#define ADT_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef void* adt_stream_t; /* cudaStream_t */

#define ADT_OK 0
#define ADT_E_SHAPE (-1)
#define ADT_E_ALIGN (-2)
#define ADT_E_ARCH (-3)
#define ADT_E_CUDA (-4)

/* Counter-based dropout site (replaces torch's global-RNG F.dropout; sasrec/modules.py:61, :626-628,
 * sasrec/model.py:20).  keep(idx) = philox4x32_10(ctr=(idx>>2, site, step), key=seed)[idx&3] >= p*2^32. */
typedef struct {
  int32_t enabled;   /* 0 -> identity (eval mode or p == 0) */
  float p;
  uint64_t seed;
  uint32_t step;
  uint32_t site;
  uint64_t base;     /* linear index offset of this rank's first element (data-parallel batch offset) */
  const uint32_t* step_dev; /* optional DEVICE counter added to `step` at run time (lets a captured CUDA graph advance) */
} adt_dropout;

int adt_version(void);
const char* adt_last_error(void);

/* Scratch / saved-activation sizes (bytes) the caller must allocate for one (B, L, H, nh, nl) training step: the library allocates
 * nothing itself.  saved = activations kept from forward for backward; scratch = backward temporaries; sort = keys/vals/tmp/hist of
 * adt_embed_sort; scatter = head/tail/has_tail of adt_embed_bwd; score_part = part_scores + part_ids of adt_score_topk for
 * (U = B, K, n_splits); wgrad_scratch = the bf16 operand copies of the hoisted weight gradients, fwd_scratch = the bf16 operands of the
 * tcgen05 forward path (both 0 when H < 128).  Sequences of 257..2048 positions need precision 1 and a head size H/nh that is a multiple of
 * 16 up to 128.  Hidden sizes of 257..512 need precision 1, H % 64 == 0 and a head size H/nh that is a multiple of 32 up to 128; the
 * block entry points then run on the tcgen05 path at every row count, so tc_scratch / wgrad_scratch are required there. */
typedef struct { int32_t B, L, H, nh, nl, K, n_splits; } adt_workspace_query;
typedef struct {
  int64_t saved, scratch, sort_keys, sort_hist, scatter_rows, scatter_flags, score_part, wgrad_scratch, fwd_scratch;
  int64_t attn_scratch;  /* L > 256: bf16 operands of the fused flash attention (O(B*L*H), one per concurrently running block; 0 for L <= 256) */
} adt_workspace_sizes;
int adt_workspace_bytes(const adt_workspace_query* q, adt_workspace_sizes* out);

/* K1. x = dropout(E[ids]*sqrt(H) + P[t]) * (ids != 0)            -- sasrec/model.py:34-41 and :53-58 */
typedef struct {
  const int32_t* ids; const float* item_emb; const float* pos_emb; float* x;
  int32_t B, L, H; adt_dropout drop;
} adt_embed_fwd_args;
int adt_embed_fwd(const adt_embed_fwd_args* a, adt_stream_t stream);

/* attention weights of one nn.MultiheadAttention / MultiheadAttentionADT (packed in-projection) */
typedef struct { const float* in_w; const float* in_b; const float* out_w; const float* out_b; } adt_mha_w;
typedef struct { float* in_w; float* in_b; float* out_w; float* out_b; } adt_mha_g;
typedef struct { const float* w1; const float* b1; const float* w2; const float* b2; } adt_ffn_w; /* Conv1d k=1 == [H,H] */
typedef struct { float* w1; float* b1; float* w2; float* b2; } adt_ffn_g;
/* Optional bf16 mirror of the flat fp32 parameter buffer: the bf16 copy of a weight W lives at bf16 + (W - base32).  Kept current by
 * adt_adam (mirror / mirror_n) or adt_to_bf16; base32 segments must start on 8-element boundaries.  bf16 == NULL: kernels convert the
 * fp32 weights on the fly. */
typedef struct { const float* base32; const void* bf16; } adt_wmirror;
/* 1 when the sequence-resident encoder forward (evaluation; one CTA per sequence, a whole block per launch) serves this shape / precision */
int adt_seq_kernels_apply(int32_t L, int32_t H, int32_t nh, int32_t precision);

/* Encoder block -- EncoderLayer.forward, sasrec/modules.py:644-655 (+ MultiheadAttentionADT :270-527,
 * PointWiseFeedForward :629-633, SparseInputLinear :696-703).  rec is written in TRUE [B,L,nh,nh] layout. */
typedef struct {
  const float* x; const int32_t* ids;                     /* block input [M,H], log_seqs (keep = ids != 0) */
  const float* ln1_w; const float* ln1_b; adt_mha_w attn; const float* ln2_w; const float* ln2_b; adt_ffn_w ffn;
  const float* sparse_w; const float* sparse_b;
  float* q; float* k; float* v; float* ctx; float* lse;    /* saved for backward: [M,H] x4, [B,nh,L] */
  float* y; float* h1;                                     /* saved for backward (may be NULL when training == 0) */
  float* out; float* rec;                                  /* outputs: [M,H], [M,nh,nh] (rec may be NULL) */
  double* nll_acc;                                         /* += -sum_{r,c} rec[r][c][c]   (may be NULL) */
  int32_t B, L, H, nh, training, mask_mode;                /* mask_mode 0 causal, 1 key-padding (bidirectional) */
  adt_dropout drop_attn, drop_ffn1, drop_ffn2;
  int32_t precision;                                       /* 0: fp32 FFMA GEMM cores; 1: bf16 tensor-core cores (fp32 accumulate) */
  int32_t phase;   /* 0: whole block; 1: LN + q/k/v projections + attention only (writes q, k, v, ctx, lse); 2: the rest of the
                      block from ctx (out-projection, residual, LN, FFN, pad mask).  Phase 2 is row-wise, so it may be called on
                      a row subset with B = rows, L = 1: predict() reads only the last position (sasrec/model.py:89) and runs
                      the tail of the LAST block on those rows only */
  adt_wmirror wm;  /* optional bf16 mirror of the parameters (see adt_wmirror) */
  float* out_last; /* optional [B][H]: the block output of the LAST position of every sequence (predict reads nothing else,
                      sasrec/model.py:89); `out` may then be NULL.  Only honoured by the sequence-resident kernel (phase 0, training 0,
                      precision 1, H == 64, L <= 64, nh in {1,2,4}); otherwise ignored, so callers must check adt_seq_kernels_apply() first */
  void* tc_scratch; /* optional, adt_workspace_sizes.fwd_scratch bytes (precision 1, H >= 128, H % 64 == 0, phase 0): every linear layer
                       then runs as one tcgen05 GEMM over all rows (block_tc.cuh) instead of inside the row-tile kernels (at >= 512 rows
                       up to H = 256).  Required beyond H = 256, with y, h1 and out, in every phase */
  void* attn_scratch; /* adt_workspace_sizes.attn_scratch bytes, required when L > 256 (fused flash attention; NULL otherwise) */
} adt_enc_block_fwd_args;
int adt_enc_block_fwd(const adt_enc_block_fwd_args* a, adt_stream_t stream);

typedef struct {
  const float* x; const int32_t* ids;
  const float* ln1_w; const float* ln1_b; adt_mha_w attn; const float* ln2_w; const float* ln2_b; adt_ffn_w ffn;
  const float* sparse_w; const float* sparse_b;
  const float* q; const float* k; const float* v; const float* ctx; const float* lse; const float* y; const float* h1;
  const float* dout;          /* grad wrt block output (NULL = 0) */
  const float* dx_extra;      /* extra grad wrt block input, e.g. the reconstruction-MSE grad (NULL = 0) */
  const float* drec;          /* external grad wrt rec (compat mode, NULL = none) */
  float nll_coef;             /* fused independence loss: lambda2 / (M_global*nh), 0 = off */
  float* dq; float* dk; float* dv; float* dctx; float* dy;   /* scratch [M,H] each */
  float* dx;                  /* out: grad wrt block input (overwritten) */
  float* g_ln1_w; float* g_ln1_b; adt_mha_g g_attn; float* g_ln2_w; float* g_ln2_b; adt_ffn_g g_ffn;
  float* g_sparse_w; float* g_sparse_b;
  int32_t B, L, H, nh, mask_mode;
  adt_dropout drop_attn, drop_ffn1, drop_ffn2;
  int32_t precision;
  adt_wmirror wm;
  void* wgrad_scratch;        /* optional, adt_workspace_sizes.wgrad_scratch bytes (precision 1, H >= 128): the row-tile kernels then only write
                                 bf16 copies of their dY / X tiles and every weight gradient becomes ONE split-K tcgen05 GEMM over all rows
                                 (>= 512 rows: the whole backward on the tcgen05 path).  Required beyond H = 256 */
  void* attn_scratch;         /* as in adt_enc_block_fwd_args */
} adt_enc_block_bwd_args;
int adt_enc_block_bwd(const adt_enc_block_bwd_args* a, adt_stream_t stream);

/* Decoder block -- DecoderLayer.forward, sasrec/modules.py:666-677 (two stock nn.MultiheadAttention + FFN). */
typedef struct {
  const float* x; const float* feats; const int32_t* ids;  /* decoder input, encoder features, dec_seqs */
  const float* ln_w; const float* ln_b; adt_mha_w slf; adt_mha_w enc; adt_ffn_w ffn;
  const float* enc_in;                                     /* reconstruction target for the fused MSE (may be NULL) */
  float* d; float* q1; float* k1; float* v1; float* ctx1; float* lse1; float* a;
  float* q2; float* k2; float* v2; float* ctx2; float* lse2; float* c; float* h1;
  float* out;
  double* mse_acc;                                         /* += sum (enc_in - out)^2   (may be NULL) */
  int32_t B, L, H, nh, training, mask_mode;
  adt_dropout drop_slf, drop_enc, drop_ffn1, drop_ffn2;
  int32_t precision;
  int32_t phase;   /* 0: whole block; 1: only LN + self-attention (independent of the encoder -> may run beside it on another
                    * stream); 2: the rest (cross-attention on `feats`, FFN) */
  adt_wmirror wm;
  void* tc_scratch; /* as in adt_enc_block_fwd_args (phases 0, 1 and 2) */
  void* attn_scratch; /* as in adt_enc_block_fwd_args */
} adt_dec_block_fwd_args;
int adt_dec_block_fwd(const adt_dec_block_fwd_args* a, adt_stream_t stream);

typedef struct {
  const float* x; const float* feats; const int32_t* ids;
  const float* ln_w; const float* ln_b; adt_mha_w slf; adt_mha_w enc; adt_ffn_w ffn;
  const float* d; const float* q1; const float* k1; const float* v1; const float* ctx1; const float* lse1; const float* a;
  const float* q2; const float* k2; const float* v2; const float* ctx2; const float* lse2; const float* c; const float* h1;
  const float* out; const float* enc_in; float mse_coef;   /* fused MSE: lambda1*2/(M_global*H); enc_in NULL = off */
  const float* dout;                                       /* grad wrt block output (NULL = 0) */
  float* denc;                                             /* out: grad wrt enc_in (overwritten; may be NULL) */
  float* dq; float* dk; float* dv; float* dctx; float* dd; float* dq2; float* dk2; float* dv2; float* dctx2; /* scratch [M,H] each */
  float* dfeats;                                           /* accumulated (+=) */
  float* dx;                                               /* out: grad wrt decoder block input */
  float* g_ln_w; float* g_ln_b; adt_mha_g g_slf; adt_mha_g g_enc; adt_ffn_g g_ffn;
  int32_t B, L, H, nh, mask_mode;
  adt_dropout drop_slf, drop_enc, drop_ffn1, drop_ffn2;
  int32_t precision;
  int32_t phase;   /* 0: whole block; 2: FFN + cross-attention adjoints (produce dfeats, dctx, dd); 1: self-attention + LN adjoints
                    * (produce dx; nothing the encoder backward needs -> may run beside it on another stream) */
  adt_wmirror wm;
  void* wgrad_scratch;        /* as in adt_enc_block_bwd_args */
  void* attn_scratch;         /* as in adt_enc_block_fwd_args */
} adt_dec_block_bwd_args;
int adt_dec_block_bwd(const adt_dec_block_bwd_args* a, adt_stream_t stream);

/* last LayerNorm + pos/neg logits + BCE sums -- sasrec/model.py:48,72-76 and sasrec/main.py:151-153.
 * acc[0] += sum softplus(-pos_logit), acc[1] += sum softplus(neg_logit), acc[2] += #valid   over pos != 0.
 * ln_w == NULL skips the LayerNorm (SuperSASRecModel has none, sasrec/supersasrec.py:56-58).
 * pos == NULL: only feats are produced (predict path, model.py:83-89). */
typedef struct {
  const float* x; const float* ln_w; const float* ln_b; const float* item_emb; const int32_t* pos; const int32_t* neg;
  float* feats; float* pos_logits; float* neg_logits; double* acc; int32_t M, H;
} adt_final_fwd_args;
int adt_final_logits_loss_fwd(const adt_final_fwd_args* a, adt_stream_t stream);

typedef struct {
  const float* x; const float* ln_w; const float* item_emb; const int32_t* pos; const int32_t* neg;
  const float* pos_logits; const float* neg_logits; const float* dfeats_in;
  const double* n_valid; float bce_weight; const float* dpl_ext; const float* dnl_ext;
  float* dx; float* cpos; float* cneg; float* g_ln_w; float* g_ln_b; int32_t M, H;
} adt_final_bwd_args;
int adt_final_logits_loss_bwd(const adt_final_bwd_args* a, adt_stream_t stream);

/* K2. embedding backward for the four lookups of one step (seq, dec, pos, neg): stable LSD radix sort of the
 * 4*M (id, element) pairs followed by a deterministic segmented scatter-add into d_item_emb (rows touched are
 * OVERWRITTEN, so d_item_emb must be zeroed once per step), plus the pos_emb gradient.
 * Replaces torch's embedding_dense_backward for sasrec/model.py:34,37,53,56,72,73.
 * adt_embed_sort only depends on the ids and may run on a side stream as soon as the batch is on the device. */
typedef struct {
  const int32_t* seq; const int32_t* dec; const int32_t* pos; const int32_t* neg; int32_t M; int32_t max_id;
  int32_t* keys; int32_t* vals;            /* out: sorted ids / element indices, 4*M each */
  int32_t* keys_tmp; int32_t* vals_tmp;    /* scratch 4*M each */
  int32_t* hist;                           /* scratch: 256 * ceil(4*M/256) ints */
} adt_embed_sort_args;
int adt_embed_sort(const adt_embed_sort_args* a, adt_stream_t stream);

typedef struct {
  const int32_t* keys; const int32_t* vals; const int32_t* seq; const int32_t* dec; int32_t B, L, H;
  const float* dx_enc; const float* dx_dec; const float* feats; const float* cpos; const float* cneg;
  adt_dropout drop_enc, drop_dec;
  float* d_item_emb; float* d_pos_emb;      /* d_pos_emb accumulated */
  float* head; float* tail; int32_t* has_tail;   /* scratch: ceil(4*M/32) x H floats (x2), ceil(4*M/32) ints */
  float emb_scale;                               /* factor on the dx_enc/dx_dec rows; 0 -> sqrt(H) (SASRec, model.py:35) */
} adt_embed_bwd_args;
int adt_embed_bwd(const adt_embed_bwd_args* a, adt_stream_t stream);

/* K6. optimiser pieces -- sasrec/main.py:170-173 (wd*||E||, clip_grad_norm_, Adam). */
int adt_sumsq(const float* x, int64_t n, double* out /* += */, adt_stream_t stream);
int adt_norm_decay_grad(float* g, const float* w, int64_t n, float wd, const double* normsq, adt_stream_t stream);
/* the two above in one pass over the FLAT gradient / parameter buffers: g[i] += wd/sqrt(*normsq) * w[i] for i >= decay_off (the item
 * table is the trailing segment), then *out += sum g^2 over all n elements.  decay_off % 4 == 0. */
int adt_sumsq_decay(float* g, const float* w, int64_t n, int64_t decay_off, float wd, const double* normsq, double* out, adt_stream_t stream);
typedef struct {
  float* p; float* g; float* m; float* v; int64_t n;
  float lr, beta1, beta2, eps, weight_decay; int32_t step; float max_norm; const double* gnormsq;
  const int32_t* step_dev;  /* optional DEVICE step count t (overrides `step`; for CUDA-graph replay) */
  void* mirror; int64_t mirror_n;   /* optional: bf16 copy of p[0 .. mirror_n) written in the same pass (adt_wmirror) */
} adt_adam_args;
int adt_adam(const adt_adam_args* a, adt_stream_t stream);
/* torch.optim.Adam's PER-PARAMETER semantics on the flat buffers (sasrec/evolution.py:111,316-318): parameters whose .grad is None
 * are skipped entirely (no moment decay, no weight decay, no step increment) and every parameter keeps its own step count.  The
 * caller lists the active segments (active_seg[n_active], indices into seg_step) and a work list of chunks of those segments
 * (chunk_start / chunk_len in elements, chunk_seg = owning segment); seg_step[] (device int32, one per segment) is incremented for
 * the active segments and then read for the bias corrections.  a->step / a->step_dev are ignored; clipping uses a->gnormsq. */
typedef struct {
  const int64_t* chunk_start; const int32_t* chunk_len; const int32_t* chunk_seg; int32_t n_chunks;
  int32_t* seg_step; const int32_t* active_seg; int32_t n_active;
} adt_adam_segments;
int adt_adam_segmented(const adt_adam_args* a, const adt_adam_segments* g, adt_stream_t stream);
/* *out = #{i < n : ids[i] != 0} (double): the BCE normaliser of sasrec/main.py:151-153, which depends on the batch only */
int adt_count_nonzero(const int32_t* ids, int32_t n, double* out, adt_stream_t stream);

/* K7. full-catalog scoring with fused per-user top-K -- replaces predict(full=True) + the host-side
 * mask / argpartition / sort of the whole score row (sasrec/model.py:91-96, sasrec/utils.py:718-731,
 * stosa/trainer.py:604-614).  scores[u][i] = <feats[u], item_emb[i]>, items whose GLOBAL id (item_offset + i) is in
 * the user's sorted seen-list are skipped; ties are ordered by ascending id.  Item-sharded evaluation calls this
 * once per shard (item_offset = first global id of the shard) and merges the per-shard lists. */
typedef struct {
  const float* feats; int32_t U, H;
  const float* item_emb; int32_t n_items; int32_t item_offset;
  const int32_t* seen_indptr; const int32_t* seen_idx;   /* CSR over users, ids ascending (NULL = no mask) */
  int32_t K;                                             /* <= 64 */
  int32_t n_splits;                                      /* catalog splits per 64-user tile (<= 256) */
  float* part_scores; int32_t* part_ids;                 /* scratch [n_splits][U][K] */
  float* out_scores; int32_t* out_ids;                   /* [U][K], best first; -inf / -1 padded */
  /* optional fused metric epilogue (get_full_sort_score, sasrec/utils.py:686-708, :530-569, :629-648): answers[u] = the held-out
   * item of user u; metric_acc[6] += {HIT@5, NDCG@5, HIT@10, NDCG@10, MRR over the K-list, #users}.  Both NULL = off. */
  const int32_t* answers; double* metric_acc;
  const int32_t* user_mask;   /* optional [U]: only users with a non-zero entry are scored and written (the exact re-run of the users
                                 adt_score_topk_tc flagged, issued unconditionally so that the whole evaluation stays capturable) */
  const float* item_bias;     /* optional [n_items], indexed like item_emb (local to the shard): scores[u][i] = <feats[u], item_emb[i]>
                                 + item_bias[i], the bias added in fp32 once after the full dot product (Bert4Rec's tied head +
                                 mask_bias).  NULL = no bias */
} adt_score_topk_args;
int adt_score_topk(const adt_score_topk_args* a, adt_stream_t stream);

/* item-sharded evaluation (SURVEY 8e): merge n_lists per-shard top-K lists (all-gathered, [n_lists][U][K] with `list_stride`
 * elements between lists, each best first, id -1 = padding) into the global top-K, order (score desc, id asc); optional fused metric
 * epilogue as in adt_score_topk.  Replaces the host-side concatenate + sort of a sharded evaluate_loader_full. */
int adt_topk_merge(const float* scores, const int32_t* ids, int32_t n_lists, int64_t list_stride, int32_t U, int32_t K,
                   float* out_scores, int32_t* out_ids, const int32_t* answers, double* metric_acc, adt_stream_t stream);

/* predict(full=True), sasrec/model.py:91-96: out[u][item_offset + i] = <feats[u], item_emb[i]> for i < n_items, fp32 FFMA
 * (row stride ld floats).  Replaces `item_emb.weight.matmul(final_feat)`. */
int adt_score_full(const float* feats, int32_t U, int32_t H, const float* item_emb, int32_t n_items, int32_t item_offset,
                   float* out, int64_t ld, adt_stream_t stream);

/* predict(full=False) + evaluate_loader's ranking, sasrec/model.py:91-96 and sasrec/utils.py:407-427:
 * scores[u][c] = <feats[u], item_emb[idx[u*idx_stride + c]]> (idx_stride 0 = one candidate list for all users),
 * rank[u] = #{c > 0 : scores[u][c] > scores[u][0]} (= `(-pred).argsort().argsort()[:,0]` without ties),
 * metric_acc[7] += {HR@5, NDCG@5, HR@10, NDCG@10, sum 1/(rank+1), #users, sum (C+1-(rank+1))/C}  (AUC with the reference's
 * candidates_size = 1 + C, quirk B7).  scores / rank / metric_acc may be NULL. */
typedef struct {
  const float* feats; const float* item_emb; const int32_t* idx; float* scores; int32_t* rank; double* metric_acc;
  int64_t idx_stride; int32_t U, H, C, n_rows;
} adt_candidate_scores_args;
int adt_candidate_scores(const adt_candidate_scores_args* a, adt_stream_t stream);

/* K7 on the tensor cores (H % 64 == 0, H <= 512; beyond 256 the catalog ring holds one 64-column K block per stage): bf16
 * TMA-fed tcgen05.mma GEMM (fp32 accumulators in TMEM) with a fused
 * streaming top-KC epilogue per (catalog split, user), then an exact fp32 re-score of the <= n_splits*KC candidates
 * per user and the final top-K.  flags[u] = 1 when the bf16 rounding bound cannot prove that the fp32 top-K is
 * contained in the candidate set; the caller re-runs those users through adt_score_topk (exact).  n_splits*KC <= 2048. */
int adt_to_bf16(const float* x, void* y_bf16, int64_t rows, int32_t H, float* max_normsq /* atomicMax'ed, may be NULL */,
                adt_stream_t stream);
typedef struct {
  const float* feats; const void* feats_bf16; int32_t U, H;          /* [U,H] fp32 and its bf16 copy */
  const float* item_emb; const void* item_emb_bf16; int32_t n_items; int32_t item_offset;
  const float* max_normsq;                                           /* device scalar: max_i |item_emb[i]|^2 */
  const int32_t* seen_indptr; const int32_t* seen_idx;
  int32_t K, KC, n_splits;
  float* part_scores; int32_t* part_ids; float* part_thr;            /* scratch [n_splits][U][KC], [2*n_splits][U] */
  float* out_scores; int32_t* out_ids; int32_t* flags;               /* [U][K], [U][K], [U] */
  const int32_t* answers; double* metric_acc;   /* fused metric epilogue as in adt_score_topk, for the users whose result is proven
                                                   exact (flags[u] == 0); flagged users are accumulated by the exact re-run */
  const float* item_bias;     /* optional [n_items] per-item fp32 bias, as in adt_score_topk (NULL = none).  It is added to every
                                 accumulator as it leaves tensor memory, so tau, the candidate lists and the exactness test all see
                                 biased scores; the re-score adds it after the fp32 dot product, bit-identical to adt_score_topk */
  const float* max_abs_bias;  /* device scalar: max_i |item_bias[i]| (required with item_bias; maintained by the caller like
                                 max_normsq).  It widens the exactness bound by the rounding of the two fp32 bias additions */
} adt_score_topk_tc_args;
int adt_score_topk_tc(const adt_score_topk_tc_args* a, adt_stream_t stream);
/* Launch plan for adt_score_topk_tc: fills the list capacity KC and the number of catalog splits to pass for (U, n_items, K).
 * Returns 1 when the call will run as two passes (catalogs of >= 65,536 rows): a sample of every 16th catalog tile fixes a per-user
 * score threshold tau with about max(192, 6K) catalog items above it, then the whole catalog is filtered against tau with an
 * append-only epilogue (tiles interleaved over the splits); 0: one streaming top-KC pass with cross-split threshold exchange. */
int adt_score_tc_plan(int32_t U, int32_t H, int32_t n_items, int32_t K, int32_t* KC, int32_t* n_splits);

/* test helper: out[i] = keep-multiplier (0 or 1/(1-p)) of element base+i of a dropout site */
int adt_philox_mask(float* out, int64_t n, const adt_dropout* d, adt_stream_t stream);

/* ---- generic ops for the post-LN backbones (Bert4Rec-ADT: /root/reference/bert4rec/model/modules.py) ---------------- */
/* y = act((x W^T + b) * scale), act 0 none / 1 relu / 2 gelu(erf) / 3 elu / 4 elu+1; pre (optional) receives the pre-activation.
 * Replaces nn.Linear (+ nn.GELU): modules.py:57-72 (q/k/v/out transfer), :128-139 (FFN), bert.py:80-90 (head). */
typedef struct {
  const float* x; const float* w; const float* b; float* y; float* pre;
  int32_t M, K, N, act; float scale; int32_t precision;
  int32_t ldy;                                 /* row stride of y/pre in floats (0 -> N): lets a wide output be produced in column blocks */
} adt_linear_fwd_args;
int adt_linear_fwd(const adt_linear_fwd_args* a, adt_stream_t stream);
/* dx = scale * dy W (dx NULL: skipped; accumulate_dx: +=) ; g_w += scale * dy^T x ; g_b += scale * colsum(dy) */
typedef struct {
  const float* x; const float* w; const float* dy; float* dx; float* g_w; float* g_b;
  int32_t M, K, N, accumulate_dx; float scale; int32_t precision;
  int32_t lddy;                                /* row stride of dy in floats (0 -> N) */
} adt_linear_bwd_args;
int adt_linear_bwd(const adt_linear_bwd_args* a, adt_stream_t stream);
int adt_act_bwd(const float* dy, const float* pre, float* dpre, int64_t n, int32_t act, adt_stream_t stream);
/* nn.Linear on tcgen05 (bert4rec/model/modules.py:57-72, :128-139, bert.py:80-90 and their autograd): c[M,N] (fp32, row stride ldc)
 * (+)= act((A[M,K] . B[N,K]^T + bias[N]) * scale), A / B bf16 row-major with row strides lda / ldb (multiples of 8 elements; use
 * adt_to_bf16_ld to make the operand copies: forward A = x, B = W; dgrad A = dy, B = W with b_mn; wgrad A = dy with a_mn, B = x with
 * b_mn -- see a_mn / b_mn below; transposed copies from adt_to_bf16_t work too).  Also every linear layer and the attention products of
 * the wide SASRec-ADT blocks (sasrec/modules.py:644-655, :666-677; vendored MHA :270-527).
 * Persistent CTAs walk 128 x 128 (or x 64) output tiles: TMA-fed ring, fp32 accumulators double-buffered in TMEM; M, N, K arbitrary
 * (zero-filled edges, masked stores).
 * pre (optional, same layout as c) receives the pre-activation values; accumulate != 0 adds into c. */
typedef struct {
  const void* a_bf16; const void* b_bf16; int64_t lda, ldb;
  float* c; float* pre; const float* bias; int64_t ldc;
  int32_t M, N, K, act, accumulate; float scale;
  int32_t a_mn, b_mn;                          /* != 0: the operand is stored MN-major, i.e. as [K][ld] with its M (or N) extent contiguous:
                                                  dgrad reads W [N,K] as b_mn, wgrad reads dy [M,N] and x [M,K] as a_mn / b_mn -- no transposes */
  int32_t split_k;                             /* > 1: that many CTAs share an output tile and add partial sums atomically (act 0, pre NULL) */
  float* c2; int32_t n_split;                  /* optional second output: columns >= n_split (multiple of 32) go to c2[:, col - n_split] (row stride ldc):
                                                  one product fills the separate k and v buffers of a packed in-projection */
  int32_t batch_inner, batch_outer;            /* > 1: a strided batch of batch_outer x batch_inner independent products in ONE launch (attention: heads x
                                                  sequences); matrix (zo, zi) of an operand starts at base + zo * x_so + zi * x_si elements */
  int64_t a_so, a_si, b_so, b_si, c_so, c_si;  /* batch strides in elements (a / b: multiples of 8, c: multiples of 4); split_k, pre, c2 unavailable */
  int32_t causal_skip;                         /* != 0: output tiles entirely above the diagonal are left untouched (causal attention scores) */
} adt_gemm_tc_args;
int adt_gemm_tc(const adt_gemm_tc_args* a, adt_stream_t stream);
/* operand copies for adt_gemm_tc: fp32 [R][C] (row stride ld) -> bf16 [R][ldy], or -> its bf16 transpose [C][ldt] */
int adt_to_bf16_ld(const float* x, int64_t ld, void* y_bf16, int64_t ldy, int64_t R, int32_t C, adt_stream_t stream);
int adt_to_bf16_t(const float* x, int64_t ld, void* y_bf16, int64_t ldt, int32_t R, int32_t C, adt_stream_t stream);
/* out[c] += sum_r x[r][c]  (bias gradient of a linear layer) */
int adt_colsum(const float* x, int64_t ld, int32_t R, int32_t C, float* out, adt_stream_t stream);
/* mode 0: y = LN(dropout(a) + r)  (DropResidualNormalizeLayer, modules.py:104-117)
 * mode 1: y = dropout(LN(a + r))  (BertEmbedding, modules.py:42-48).   r may be NULL. */
typedef struct {
  const float* a; const float* r; const float* gamma; const float* beta; float* y;
  const float* dy; float* da; float* dr; float* g_gamma; float* g_beta;     /* backward only */
  int32_t M, H, mode; float eps; adt_dropout drop;
} adt_drl_args;
int adt_drop_res_ln_fwd(const adt_drl_args* a, adt_stream_t stream);
int adt_drop_res_ln_bwd(const adt_drl_args* a, adt_stream_t stream);
/* s[row] = A[ia[row]] + B[ib[row]] + C[ic[row]] (B, C may be NULL) ; g[ids[row]] += dx[row] for ids != padding_idx */
int adt_gather3(const int32_t* ia, const float* A, const int32_t* ib, const float* B, const int32_t* ic, const float* C, float* s,
                int32_t M, int32_t H, adt_stream_t stream);
int adt_small_table_grad(const int32_t* ids, const float* dx, float* g, int32_t M, int32_t H, int32_t padding_idx, adt_stream_t stream);
/* multi-head attention core on projected q (pre-scaled), k, v [B*L, H]: softmax(q k^T + mask) -> dropout -> . v
 * mask_mode 0 causal, 1 key padding (key_ids[b][j] == 0 -> -1e9, modules.py:88-91).  lse [B,nh,L] saved for backward.
 * 1 <= L <= 2048; L > 256 needs precision 1, a head size H/nh that is a multiple of 16 up to 128, tc_scratch, and (backward) ctx. */
typedef struct {
  const float* q; const float* k; const float* v; float* ctx; float* lse; const int32_t* key_ids;   /* backward reads ctx when L > 256 */
  const float* dctx; float* dq; float* dk; float* dv;                       /* backward only */
  int32_t B, L, H, nh, mask_mode, training; adt_dropout drop; int32_t precision;
  void* tc_scratch;   /* adt_attention_scratch_bytes(B, L, H, nh, backward) bytes.  Sequences of 65..256 positions in the bf16 mode then run as
                         strided-batch tcgen05 GEMMs (q k^T, P v, and the three backward products) + one softmax / dropout row kernel
                         (optional there); sequences of 257..2048 positions run in the fused flash kernels (required there) */
} adt_attention_args;
int64_t adt_attention_scratch_bytes(int32_t B, int32_t L, int32_t H, int32_t nh, int32_t backward);
int adt_attention_fwd(const adt_attention_args* a, adt_stream_t stream);
int adt_attention_bwd(const adt_attention_args* a, adt_stream_t stream);
/* the fused flash attention (flash_tc.cu) at any 1 <= L <= 2048 (bf16, head size a multiple of 16 up to 128): the kernels every call
 * above dispatches to for L > 256, exported so that shorter sequences can be compared with the batched path on the same inputs.
 * tc_scratch: adt_attention_scratch_bytes(B, max(L, 257), H, nh, backward) bytes; the backward reads ctx. */
int adt_attention_flash_fwd(const adt_attention_args* a, adt_stream_t stream);
int adt_attention_flash_bwd(const adt_attention_args* a, adt_stream_t stream);
/* softmax cross-entropy over logits rows [R,V] (nn.CrossEntropyLoss on the rows that carry a label, trainer.py:113-115).
 * fwd: lse[r], *loss_acc += sum_r (lse[r] - logits[r][labels[r]]).  bwd: logits <- (softmax - onehot) * coef, in place. */
int adt_softmax_ce_fwd(const float* logits, const int32_t* labels, float* lse, double* loss_acc, int32_t R, int32_t V, adt_stream_t stream);
int adt_softmax_ce_bwd(float* logits, const int32_t* labels, const float* lse, float coef, int32_t R, int32_t V, adt_stream_t stream);
/* vocabulary head + softmax cross-entropy without the [R,V] logits (bert.py:80-90 + trainer.py:113-115 on the labelled rows):
 *   z[r][v] = <x[r], W[v]> + bias[v]   (bf16 operands, fp32 accumulation in TMEM, bias added in fp32 as the accumulator leaves it).
 * fwd: lse[r] = log sum_v exp z[r][v];  *loss_acc += sum_r (lse[r] - z[r][labels[r]]).  The scores stay on chip: the tcgen05 epilogue keeps
 *      a running (max, sum exp) per row and tile, a merge kernel folds the tiles.
 * bwd: per vocabulary chunk [v0, v0 + Vc): recompute z, dS = c (exp(z - lse) - onehot) with c = coef * (*coef_dev if non-NULL) rounded to
 *      bf16 in scratch; g_bias[v] += fp32 column sums of dS; dx (+)= dS W[v0:v0+Vc] and g_w[v0:v0+Vc] += dS^T x on adt_gemm_tc.
 *      dx [R][H] fp32 is overwritten, g_w [V][H] fp32 and g_bias [V] are accumulated.
 * x_bf16 [R][ldx], w_bf16 [V][ldw] (ldx, ldw >= H, multiples of 8), labels in [0, V), bias / g_bias / coef_dev may be NULL.
 * Vc is the widest multiple of 128 whose scratch fits scratch_bytes (adt_linear_ce_plan): memory O(R Vc), not O(R V). */
typedef struct {
  const void* x_bf16; const void* w_bf16; int64_t ldx, ldw;
  const float* bias; const int32_t* labels; int32_t R, V, H;
  float* lse; double* loss_acc; float coef; const float* coef_dev;
  float* dx; float* g_w; float* g_bias;
  void* scratch; int64_t scratch_bytes;
} adt_linear_ce_args;
int adt_linear_ce_fwd(const adt_linear_ce_args* a, adt_stream_t stream);
int adt_linear_ce_bwd(const adt_linear_ce_args* a, adt_stream_t stream);
/* host only: the vocabulary chunk (*vocab_chunk, = V when one chunk covers it) for scratch_bytes, and the least scratch that works (one
 * 128-column chunk).  ADT_E_SHAPE when scratch_bytes is below that. */
int adt_linear_ce_plan(int32_t R, int32_t V, int32_t H, int64_t scratch_bytes, int32_t* vocab_chunk, int64_t* min_scratch_bytes);

/* ---- STOSA-ADT (SURVEY 8a row a20) -------------------------------------------------------------------------------
 * elementwise activation y = act(x) (act codes of adt_linear_fwd); n % 4 == 0. */
int adt_act_fwd(const float* x, float* y, int64_t n, int32_t act, adt_stream_t stream);
/* Wasserstein attention core on projected streams [B*L, H] (cov streams already ELU+1) -- replaces the score / softmax /
 * dropout / context lines of DistAttention.forward and DistEDAttention.forward (stosa/modules.py:240-254, :330-344):
 *   S_ij = -( |mq_i - mk_j|^2 in matmul form + sum cq_i + sum ck_j - 2 sqrt(cq_i).sqrt(ck_j) ) / sqrt(hd) + mask_ij,
 *   mask_ij = 0 if key_ids[b][j] > 0 and j <= i else float(-2^32+1) (additive, models.py:229-233), P = dropout(softmax(S)),
 *   mctx = P mv, cctx = P^2 cv.  bwd returns the gradients of all six streams.  Needs (8 L + 64)(hd + 4) + 96 L floats of
 *   shared memory in bwd (L=100, hd=16 -> 108 KB); larger shapes return ADT_E_SHAPE (adt_wattention_resident_fits tells which).
 * adt_wattention_flash_fwd / _bwd: the same core on the tensor cores for any 1 <= L <= 2048 with a head size hd = H/nh that is a
 *   multiple of 16 up to 64 (bf16 operands centred per (sequence, head), fp32 accumulation; the same mask, dropout stream and row
 *   statistics).  tc_scratch: adt_wattention_scratch_bytes(B, L, H, nh, backward) bytes; the backward also reads the forward's outputs
 *   (mctx_in, cctx_in).  Both write every output element once: no zeroed buffers, bitwise reproducible. */
typedef struct {
  const float* mq; const float* cq; const float* mk; const float* ck; const float* mv; const float* cv;
  float* mctx; float* cctx; float* lse;            /* softmax row statistics (max, 1/sum) [B, nh, L, 2]: written by fwd, read by bwd */
  const int32_t* key_ids;                          /* [B, L] ids of the KEY sequence */
  const float* dmctx; const float* dcctx;          /* bwd only */
  float* dmq; float* dcq; float* dmk; float* dck; float* dmv; float* dcv;
  int32_t B, L, H, nh; adt_dropout drop;           /* attention-probability site (base = row offset) */
  void* tc_scratch;                                /* flash only */
  const float* mctx_in; const float* cctx_in;      /* flash bwd only: mctx, cctx of the forward */
} adt_wattention_args;
int adt_wattention_fwd(const adt_wattention_args* a, adt_stream_t stream);
int adt_wattention_bwd(const adt_wattention_args* a, adt_stream_t stream);
int adt_wattention_flash_fwd(const adt_wattention_args* a, adt_stream_t stream);
int adt_wattention_flash_bwd(const adt_wattention_args* a, adt_stream_t stream);
/* host only: 1 when the resident kernels serve (L, H/nh) in the forward (backward = 0) or the backward, 0 when not, ADT_E_SHAPE for
 * invalid dims; the scratch of the flash kernels (O(B L H), -1 for shapes they do not serve) */
int adt_wattention_resident_fits(int32_t L, int32_t H, int32_t nh, int32_t backward);
int64_t adt_wattention_scratch_bytes(int32_t B, int32_t L, int32_t H, int32_t nh, int32_t backward);
/* BPR + positive-vs-negative loss on elementwise Wasserstein distances (stosa/trainer.py:358-391).
 * fwd: acc[0] += sum_t softplus(-(d_neg - d_pos + 1e-24)), acc[1] += sum_t max(d_pos - d_pn, 0), acc[2] += sum_t (sign(d_neg-d_pos)+1)/2,
 *      acc[3] += #targets (pos id > 0).  bwd: gcoef[0] = dLoss/d(acc[0]), gcoef[1] = dLoss/d(acc[1]) (device scalars) ->
 *      gradients of the sequence streams and per-row gradients of the looked-up table rows (cov rows through ELU+1),
 *      to be scatter-added by adt_embed_sort + adt_embed_bwd. */
typedef struct {
  const float* seq_mean; const float* seq_cov;     /* [M, H] */
  const float* item_mean; const float* item_cov;   /* tables [I+1, H]; cov raw (ELU+1 applied inside) */
  const int32_t* pos; const int32_t* neg;          /* [M] */
  double* acc;                                     /* [4] */
  const float* gcoef;                              /* [2], bwd only */
  float* d_seq_mean; float* d_seq_cov; float* g_pos_mean; float* g_pos_cov; float* g_neg_mean; float* g_neg_cov;   /* [M, H], bwd only */
  int32_t M, H;
} adt_wbpr_args;
int adt_wbpr_fwd(const adt_wbpr_args* a, adt_stream_t stream);
int adt_wbpr_bwd(const adt_wbpr_args* a, adt_stream_t stream);
/* reconstruction term (F.mse_loss of sasrec/main.py:158, bert4rec/trainer.py:121, stosa/trainer.py:519-520):
 * fwd: *acc += sum (a-b)^2 ; bwd: da = 2 (a-b) * g[0] * scale, db = -da (g: device scalar, scale = lambda / n). n % 4 == 0. */
int adt_sqdiff_fwd(const float* a, const float* b, int64_t n, double* acc, adt_stream_t stream);
int adt_sqdiff_bwd(const float* a, const float* b, const float* g, float scale, float* da, float* db, int64_t n, adt_stream_t stream);
/* rows for full-sort evaluation through adt_score_topk (stosa/trainer.py:464-479, modules.py:30-43), width 2H+4:
 *   is_user = 0: [ mean_i | sqrt(elu(cov_i)+1) | -(|mean_i|^2 + sum(elu(cov_i)+1)) | 0 0 0 ]   (catalog rows, cov raw)
 *   is_user = 1: [ 2 mean_u | 2 sqrt(cov_u) | 1 | 0 0 0 ]                                        (user rows, cov already ELU+1)
 * so that <user row, catalog row> = -distance(u, i) + const(u): the largest dot product is the smallest distance. */
int adt_wcatalog_rows(const float* mean, const float* cov, float* out, int32_t n, int32_t H, int32_t is_user, adt_stream_t stream);
/* the same ranking as a centred, biased dot product for adt_score_topk / adt_score_topk_tc with item_bias.  With item rows
 * y_i = [ mean_i | sqrt(elu(cov_i)+1) ], user rows x_u = [ mean_u | sqrt(cov_u) ] and any mu,
 *   -distance(u, i) = -|x_u - y_i|^2 = <2 (x_u - mu), y_i - mu> - |y_i - mu|^2 - |x_u - mu|^2,   the last term constant per user.
 * mu = the column mean of the y_i removes the component all items share, which keeps the bf16 bound of adt_score_topk_tc tight.
 * adt_wcatalog_build: mu [2H] (fixed-order fp64 column sums: an unchanged table gives bit-identical output), rows [n][2H] = y_i - mu,
 *   bias [n] = -|rows[i]|^2, all fp32, H <= 128.  Two launches.  work: adt_wcatalog_work_bytes(H) bytes of scratch (column partials and
 *   an arrival counter), zero-filled before its first use; every call leaves it zero-filled where the counter is.
 * adt_wcatalog_user: out [U][2H] = 2 (x_u - mu) from the encoder's (mean, cov) [U][H] (cov already ELU+1); no host synchronisation. */
int adt_wcatalog_work_bytes(int32_t H, int64_t* bytes);
int adt_wcatalog_build(const float* mean, const float* cov, int32_t n, int32_t H, float* mu, float* rows, float* bias, void* work,
                       adt_stream_t stream);
int adt_wcatalog_user(const float* mean, const float* cov, const float* mu, float* out, int32_t U, int32_t H, adt_stream_t stream);

/* ---- device-side batch assembly and sampling (SURVEY 8f-1) ---------------------------------------------------------------------
 * User histories live in HBM as CSR (hist_indptr [n_users+2] indexed by user id, hist_items in interaction order, hist_sorted the same
 * rows sorted ascending for membership tests).  Every random draw is Philox4x32-10 of (seed, epoch, user, position, draw index), so
 * a sample does not depend on its batch and oracle/sampler_oracle.py reproduces it bit for bit.
 * adt_assemble_train_batch == WarpDataset.sample_data + random_neq (sasrec/utils.py:288-307, :73-77): right-aligned seq / pos,
 * dec = seq shifted right by one, neg uniform over 1..itemnum outside the user's history. */
typedef struct {
  const int32_t* users; const int32_t* hist_indptr; const int32_t* hist_items; const int32_t* hist_sorted;
  int32_t* seq; int32_t* dec; int32_t* pos; int32_t* neg;      /* out [B][L] */
  int32_t B, L, itemnum; uint64_t seed; uint32_t epoch;
} adt_train_batch_args;
int adt_assemble_train_batch(const adt_train_batch_args* a, adt_stream_t stream);
/* adt_assemble_eval_batch == EvalDataset.sample_data (sasrec/utils.py:162-191) + PopularSampler.get_negative_samples (:57-69):
 * seq = the last L history items (+ last_item[u] appended when non-zero: test mode), item_idx[u] = [answers[u], n_candidates ids drawn
 * by popularity WITHOUT replacement over ids 0..itemnum-1 (quirk B8) outside the user's seen set].  alias_prob / alias_idx: Vose alias
 * table of popular_p.  n_candidates == 0: sequences only. */
typedef struct {
  const int32_t* users; const int32_t* hist_indptr; const int32_t* hist_items;
  const int32_t* seen_indptr; const int32_t* seen_sorted;       /* per-user seen set (sorted ids), CSR by user id */
  const int32_t* last_item; const int32_t* answers;
  const float* alias_prob; const int32_t* alias_idx;
  int32_t* seq; int32_t* item_idx;                              /* out [U][L], [U][1 + n_candidates] */
  int32_t U, L, itemnum, n_candidates; uint64_t seed; uint32_t epoch;
} adt_eval_batch_args;
int adt_assemble_eval_batch(const adt_eval_batch_args* a, adt_stream_t stream);

/* adt_cloze_batch == Bert4Rec's cloze instances (bert4rec/datasets/dataset.py:70-158, SURVEY 8f-3) generated on the device instead of
 * a pre-generated Python list of dupe_factor x users tensors: instance b = window [win_start, win_start + win_len) of the user's
 * history, right aligned; per position p ~ U[0,1): p < mask_prob -> label = item and token = mask_token (p/mask_prob < 0.8), a random
 * item in 1..itemnum (< 0.9) or the item itself; the decoder copy always ends in mask_token; dup[b] < 0 = the "mask last" instance.
 * Draws are Philox(user, position in the history, dup, epoch): independent of the batch. */
typedef struct {
  const int32_t* users; const int32_t* win_start; const int32_t* win_len; const int32_t* dup;
  const int32_t* hist_indptr; const int32_t* hist_items;
  int32_t* tokens; int32_t* dec_tokens; int32_t* labels;         /* out [B][L] */
  int32_t B, L, itemnum, mask_token; float mask_prob; uint64_t seed; uint32_t epoch;
} adt_cloze_batch_args;
int adt_cloze_batch(const adt_cloze_batch_args* a, adt_stream_t stream);

/* optional per-kernel CUDA-event timing (used by bench.py for the live roofline number; off by default) */
int adt_timing_enable(int on);
int adt_debug_read(long long* out, int n);   /* clock64() phase stamps of CTA 0 of the instrumented kernels (debug) */
int adt_timing_collect(char* names_buf, int buf_len, float* total_ms, int* counts, int max_names);

#ifdef __cplusplus
}
#endif
#endif
