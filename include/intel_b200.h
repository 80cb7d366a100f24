/* libintel_b200 - C ABI of the B200-native IntEL hot path.
 *
 * The reference (JiayuLi-997/IntEL-SIGIR2023) is pure Python; it has no FFI.  Its plugin
 * surface is three Python call signatures resolved by name (IntEL/src/main.py:127-130):
 *
 *   model(batch)            -> {"weights","ens_score","intents"}   models/IntEL/IntEL.py:117-124
 *   criterion(out, batch)   -> (loss, ensemble_loss, intent_loss)  loss/Int{List,BPR,MSE}loss.py:14-19
 *   BaseRunner.evaluate_method(...) / evaluate_intents(...)        helpers/BaseRunner.py:57-150
 *
 * The entry points below are what a ctypes binding of those three calls needs; each one
 * names the reference code it replaces.  Conventions (SURVEY.md section 8b):
 *   - plain pointers + sizes, no torch types; every pointer is DEVICE memory owned by the caller
 *   - tensors arrive in the dtypes the reference's collate_batch delivers (int64 ids, float64
 *     scores / intents); conversion happens inside the kernels' loads
 *   - scratch comes from a caller workspace (query *_workspace_bytes first); the library never
 *     allocates or frees device memory and never synchronises: all work is queued on `stream`
 *   - forward calls leave their saved activations in the workspace; the matching backward call
 *     must be given the same workspace, untouched
 *   - backward entry points ACCUMULATE (+=) into the gradient buffers (dense, same shapes as the
 *     parameters, zeroed by the caller) so torch.optim.Adam(weight_decay) stays drop-in
 *   - return 0 on success, otherwise an INTEL_ERR_* code; intel_last_error() gives the message
 *     (thread-local).  No exceptions cross the ABI.
 */
#ifndef INTEL_B200_H
#define INTEL_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define INTEL_ABI_VERSION 1
#define INTEL_MAX_BERT_LAYERS 4
#define INTEL_MAX_TOPK 16
#define INTEL_ENCODER_BERT4REC 0
#define INTEL_ENCODER_GRU4REC 1

typedef void* intel_stream_t; /* cudaStream_t */

/* Shapes of one batch + model widths (flag names of IntEL.py:17-34). */
typedef struct {
    int64_t B, L, K, I;      /* sessions, padded list length, basic lists, intents */
    int64_t H1, H2;          /* padded session-history / item-history lengths */
    int64_t item_rows, class_rows, user_rows, ctx_rows;
    int32_t d_iid, d_im, d_u, d_s, d_int, d_ctx;   /* i/im/u/s/intent/context_emb_size */
    int32_t qsize;           /* cross_attn_qsize */
    int32_t heads, layers;   /* num_heads, num_layers of the two self-attention stacks */
    int32_t cross_attention; /* 1: CrossAtt pooling (default); 0: intent MLP gate */
    int32_t encoder;         /* INTEL_ENCODER_* */
    int32_t gru_hidden, bert_layers, bert_heads, history_max;
    /* nn.Dropout of the two self-attention stacks (IntEL.py:187,196), training mode only: p = 0 disables it.
     * Masks come from a counter-based hash of (seed, stream, layer, row, channel); pass a new seed per step. */
    float dropout_p;
    uint64_t dropout_seed;
    /* 1: forward only (BaseRunner.predict runs under torch.no_grad()): the fused stack kernels skip the activations they
     * would otherwise leave in the workspace for intel_ensemble_bwd, which must then not be called on this workspace. */
    int32_t inference;
} intel_dims_t;

typedef struct {             /* layers.py TransformerLayer, one block of BERT4RecEncoder */
    float *qw, *qb, *kw, *kb, *vw, *vb, *ln1w, *ln1b, *l1w, *l1b, *l2w, *l2b, *ln2w, *ln2b;
} intel_bert_layer_t;

typedef struct {             /* GeneralSeq.py:58-106 */
    float* pos;                                          /* p_embeddings [history_max+1, d] */
    intel_bert_layer_t layer[INTEL_MAX_BERT_LAYERS];
    float *w_ih, *w_hh, *b_ih, *b_hh, *w_out;            /* nn.GRU l0 + out (bias-free) */
} intel_encoder_t;

typedef struct {             /* one self-attention stack of IntEL.py:182-197 */
    float *wq, *wk, *wv, *w1, *b1, *w2, *b2, *lnw, *lnb;
} intel_selfatt_t;

/* Every parameter of the reference module (state_dict contract, SURVEY.md 8b).  The same
 * struct type carries the gradient buffers in the backward calls. */
typedef struct {
    float *iid_emb, *item_emb, *uid_emb, *ctx_emb;       /* embedding tables */
    float *intent_w, *intent_b;                          /* intent_embeddings [d_int, I] */
    float *score_w, *score_b;                            /* score_embeddings  [d_s, K]   */
    intel_selfatt_t item, score;
    float *xq_item, *xk_item, *xv_item;                  /* intent_item_attention.{query,key,value}_layer */
    float *xq_score, *xk_score, *xv_score;               /* intent_score_attention.*                      */
    float *gate_item_w0, *gate_item_b0, *gate_item_w2;   /* intent_item_embeddings.{0,2} (cross_attention=0) */
    float *gate_score_w0, *gate_score_b0, *gate_score_w2;
    float *head_w, *head_b;                              /* weight_embeddings [K, d_i+d_s+d_u+d_int] */
    intel_encoder_t enc, item_enc;                       /* encoder / item_encoder */
    float *pred_w, *pred_b;                              /* pred_layer [I, d_pred] */
} intel_tensors_t;

/* One collated batch (BaseModel.py:121-142 layout; ragged fields right-padded with 0). */
typedef struct {
    const int64_t *u_id;             /* [B]      u_id_c          */
    const int64_t *i_id;             /* [B,L]    i_id_s          */
    const int64_t *i_class;          /* [B,L]    i_class_c (NULL when class_rows == 0) */
    const int64_t *session_len;      /* [B]                      */
    const double  *scores;           /* [B,L,K]  float64         */
    const int64_t *context_mh;       /* [B]                      */
    const int64_t *his_context;      /* [B,H1]   his_context_mh  */
    const double  *his_intents;      /* [B,H1,I] float64 dense   */
    const int64_t *history_len;      /* [B]                      */
    const int64_t *his_item_id;      /* [B,H2]                   */
    const double  *his_item_int;     /* [B,H2,I] float64 one-hot */
    const int64_t *history_item_len; /* [B]                      */
    /* Opt-in compact form of the two dense history tensors (what a device-side batch builder would emit):
     * entry e of row (b,h) adds val * W[:, idx].  When the idx pointer is non-NULL the dense tensor is ignored. */
    const int32_t *his_intents_idx;  /* [B,H1,nz1] */
    const float   *his_intents_val;  /* [B,H1,nz1] */
    const int32_t *his_item_int_idx; /* [B,H2,nz2] */
    const float   *his_item_int_val; /* [B,H2,nz2] */
    int32_t nz1, nz2;
} intel_batch_t;

const char* intel_last_error(void);
int intel_abi_version(void);

/* ---- input validation ------------------------------------------------------------------- */
/* The reference's nn.Embedding raises IndexError on an id outside its table (IntEL.py:135-178) and its encoders need
 * 1 <= history_len <= H (GeneralSeq.py:64-78, 95-106).  This pass ORs one bit per offending field class into flags[0]
 * (device int32, zeroed by the caller); the model entry points themselves stay memory-safe on such input (a bad id reads
 * a zero row and is skipped by the gradient scatter) but their results are then meaningless. */
#define INTEL_BAD_USER_ID 1
#define INTEL_BAD_ITEM_ID 2
#define INTEL_BAD_CLASS_ID 4
#define INTEL_BAD_CONTEXT_ID 8
#define INTEL_BAD_SESSION_LEN 16
#define INTEL_BAD_HISTORY_LEN 32
#define INTEL_BAD_INTENT_IDX 64
int intel_batch_validate(const intel_dims_t* d, const intel_batch_t* batch, int32_t* flags, intel_stream_t stream);

/* ---- model forward / backward -------------------------------------------------------- */
/* IntEL.predict_intent (IntEL.py:126-155): intents_out f32 [B,I] = softmax(pred_layer(...)). */
size_t intel_intent_workspace_bytes(const intel_dims_t* d);
int intel_intent_fwd(const intel_dims_t* d, const intel_tensors_t* params, const intel_batch_t* batch,
                     float* intents_out, void* workspace, size_t workspace_bytes, intel_stream_t stream);
/* autograd of the above: the incoming gradient is d_intents + d_intents_extra (f32 [B,I] each; the
 * second, nullable, is the part that intel_ensemble_bwd produced); accumulates into `grads`. */
int intel_intent_bwd(const intel_dims_t* d, const intel_tensors_t* params, const intel_batch_t* batch,
                     const float* intents, const float* d_intents, const float* d_intents_extra,
                     intel_tensors_t* grads,
                     void* workspace, size_t workspace_bytes, intel_stream_t stream);

/* IntEL.predict_ensemble (IntEL.py:158-217): weights_out f32 [B,L,K], ens_out f32 [B,L]. */
size_t intel_ensemble_workspace_bytes(const intel_dims_t* d);
int intel_ensemble_fwd(const intel_dims_t* d, const intel_tensors_t* params, const intel_batch_t* batch,
                       const float* intents, float* weights_out, float* ens_out,
                       void* workspace, size_t workspace_bytes, intel_stream_t stream);
/* d_weights [B,L,K] / d_ens [B,L] may be NULL (treated as zero); d_intents_out f32 [B,I] is overwritten. */
int intel_ensemble_bwd(const intel_dims_t* d, const intel_tensors_t* params, const intel_batch_t* batch,
                       const float* intents, const float* d_weights, const float* d_ens,
                       intel_tensors_t* grads, float* d_intents_out,
                       void* workspace, size_t workspace_bytes, intel_stream_t stream);

/* The same backward pass in phases, for data-parallel callers that want to exchange gradients while the tail of the
 * pass still runs (no counterpart in the reference, which is single process: helpers/BaseRunner.py:268-291).
 * HEAD: weight head + both pooled cross attentions; d_intents_out is final afterwards.  ITEM / SCORE: the self-attention
 * stack of one stream plus the gradients of its inputs (item / class embedding rows; score_embeddings).  HEAD must come
 * first; intel_ensemble_bwd == all three in the order HEAD, ITEM, SCORE. */
#define INTEL_ENS_BWD_HEAD 1
#define INTEL_ENS_BWD_ITEM 2
#define INTEL_ENS_BWD_SCORE 4
int intel_ensemble_bwd_phase(const intel_dims_t* d, const intel_tensors_t* params, const intel_batch_t* batch,
                             const float* intents, const float* d_weights, const float* d_ens,
                             intel_tensors_t* grads, float* d_intents_out,
                             void* workspace, size_t workspace_bytes, intel_stream_t stream, int phases);
/* ---- sparse table gradients (IntEL sparse_grad = 1) ----------------------------------------------------
 * Row set of one table for one step: the ascending unique ids in [0, table_rows) of ids_a [n_a] and ids_b [n_b] (either may
 * be empty; other ids are skipped, as the dense scatter skips them).  row_slot: caller-owned device int32 [table_rows],
 * zero-filled once before the first call; every call leaves all entries >= 0 and sets row_slot[id] = the position of id
 * in the set for each id of the set.  rows_out: device int64 [>= min(table_rows, n_a + n_b)]; count_out: device int64 [1]
 * receives U, the size of the set.  Deterministic.  Data-parallel callers pass the ids of all ranks. */
size_t intel_rowset_workspace_bytes(int64_t table_rows);
int intel_rowset_build(int64_t table_rows, const int64_t* ids_a, int64_t n_a, const int64_t* ids_b, int64_t n_b,
                       int32_t* row_slot, int64_t* rows_out, int64_t* count_out, void* workspace, size_t workspace_bytes,
                       intel_stream_t stream);
/* The row_slot maps of the four embedding tables (any may be NULL: that table's gradient stays dense).  With a map, the
 * table's gradient buffer in `grads` is the compact [U, d] block of its row set: row j holds the gradient of row
 * rows_out[j].  Every id the batch feeds to that table must be in the set. */
typedef struct {
    const int32_t *iid, *item, *uid, *ctx;
} intel_row_maps_t;
/* intel_ensemble_bwd_phase / intel_intent_bwd writing the table gradients through the maps (maps NULL: the plain calls) */
int intel_ensemble_bwd_phase_rows(const intel_dims_t* d, const intel_tensors_t* params, const intel_batch_t* batch,
                                  const float* intents, const float* d_weights, const float* d_ens,
                                  intel_tensors_t* grads, float* d_intents_out,
                                  void* workspace, size_t workspace_bytes, intel_stream_t stream, int phases,
                                  const intel_row_maps_t* maps);
int intel_intent_bwd_rows(const intel_dims_t* d, const intel_tensors_t* params, const intel_batch_t* batch,
                          const float* intents, const float* d_intents, const float* d_intents_extra,
                          intel_tensors_t* grads, void* workspace, size_t workspace_bytes, intel_stream_t stream,
                          const intel_row_maps_t* maps);
/* Number of SMs (0..64) the persistent backward kernel of the self-attention stack leaves free when the SCORE phase is
 * called on its own, so that a collective launched on another stream finds room to run beside it.  Default 0. */
int intel_reserve_sms(int n);

/* ---- losses with fused gradients ------------------------------------------------------ */
/* Each writes the scalar loss (batch mean, diversity term folded in like the reference's in-place
 * `loss +=`) to loss_out[0] (float64 accumulator) and the gradient of that scalar w.r.t. ens_score / weights to
 * d_ens [B,L] / d_weights [B,L,K] (overwritten; d_weights may be NULL when cal_diversity == 0). */
/* Listloss.forward (Listloss.py:12-43) */
int intel_loss_pl_fwd_bwd(int64_t B, int64_t L, int64_t K, const float* ens, const float* weights,
                          const double* scores, const int64_t* ranking, const int64_t* session_len,
                          int cal_diversity, double alpha, double* loss_out, float* d_ens, float* d_weights,
                          intel_stream_t stream);
/* BPRloss.forward (BPRloss.py:12-56).  noise f32 [B,L,L] replays torch.rand_like (BPRloss.py:26);
 * NULL -> counter-based in-kernel RNG keyed by `seed`. */
int intel_loss_bpr_fwd_bwd(int64_t B, int64_t L, int64_t K, const float* ens, const float* weights,
                           const double* scores, const int64_t* ranking, const int64_t* session_len,
                           const float* noise, uint64_t seed, int cal_diversity, double alpha,
                           double* loss_out, float* d_ens, float* d_weights, intel_stream_t stream);
/* MSEloss.forward (MSEloss.py:12-30) */
int intel_loss_mse_fwd_bwd(int64_t B, int64_t L, int64_t K, const float* ens, const float* weights,
                           const double* scores, const int64_t* ranking, const int64_t* session_len,
                           int cal_diversity, double alpha, double* loss_out, float* d_ens, float* d_weights,
                           intel_stream_t stream);
/* BaseIntloss.get_intloss (BaseIntloss.py:30-67): out[0]=intent_loss, out[1]=ce, out[2]=kl*T^2 (f64);
 * d_pred f32 [B,I] = d intent_loss / d pred.  scratch: >= 16 bytes of device memory. */
int intel_intent_loss_fwd_bwd(int64_t B, int64_t I, const float* pred, const double* true_intents,
                              double kl_weight, double kl_temp, double* out, float* d_pred,
                              void* scratch, intel_stream_t stream);
/* y[i] = x[i] * (ca * *a + cb * *b) with device scalars a, b (either may be NULL): chains the upstream
 * autograd scalar into the fused gradients without a host sync. */
int intel_scale_by_device_scalar(int64_t n, const float* x, const double* a, double ca, const double* b,
                                 double cb, float* y, intel_stream_t stream);

/* ---- evaluation ------------------------------------------------------------------------ */
/* BaseRunner.evaluate_method (BaseRunner.py:57-131), per-session terms then a deterministic reduction.
 * pred f32 [N, ld], ranking i64 [N, ld] (rows padded as the batches were), session_len / pay / fav /
 * click i64 [N]; max_len = max(max session_len over the whole eval set, max topk); topk[n_topk] host ints.
 * sums f64 [n_topk * 7]: per k -> {ndcg_sum, pay_hr, pay_ndcg, fav_hr, fav_ndcg, click_hr, click_ndcg};
 * counts f64 [4]: {N, #pay sessions, #fav sessions, #click sessions}.  Tie rule: see DESIGN.md. */
size_t intel_ndcg_workspace_bytes(int64_t N, int n_topk);
int intel_ndcg_topk(int64_t N, int64_t ld, const float* pred, const int64_t* ranking,
                    const int64_t* session_len, const int64_t* pay, const int64_t* fav, const int64_t* click,
                    int64_t max_len, const int32_t* topk, int n_topk, double* sums, double* counts,
                    void* workspace, size_t workspace_bytes, intel_stream_t stream);
/* BaseRunner.evaluate_intents (BaseRunner.py:133-150): sums f64 [n_topk*2] = {Int-NDCG, Int-HR} per k. */
size_t intel_intent_topk_workspace_bytes(int64_t N, int n_topk);
int intel_intent_topk(int64_t N, int64_t I, const double* true_intents, const float* pred_intents,
                      const int32_t* topk, int n_topk, double* sums,
                      void* workspace, size_t workspace_bytes, intel_stream_t stream);

/* ---- fixed-weight list fusion (script/baselines.sh) ------------------------------------- */
/* ens[b,l] = sum_k weights[b,l,k] * float(scores[b,l,k])   (GeneralSeq.py:23-32, IntEL.py:215) */
int intel_fuse_fwd(int64_t B, int64_t L, int64_t K, const float* weights, const double* scores,
                   float* ens_out, intel_stream_t stream);
/* SingleSort.forward (SingleSort.py:23-32): ens = float(scores[:,:,column]) */
int intel_select_list(int64_t B, int64_t L, int64_t K, const double* scores, int column, float* ens_out,
                      intel_stream_t stream);
/* Borda.forward (Borda.py:23-30): mean over lists of the ascending rank inside the padded list. */
int intel_rank_lists(int64_t B, int64_t L, int64_t K, const double* scores, float* ens_out,
                     intel_stream_t stream);

/* ---- device-side batch construction ----------------------------------------------------------
 * A columnar corpus resident in device memory replaces the per-session `_get_feed_dict` + `collate_batch` of the reference
 * (models/BaseModel.py:121-197, models/GeneralSeq.py:35-54, models/IntEL/IntEL.py:220-239).  All arrays are device pointers
 * owned by the caller.  Per-row columns have N entries (one per session of the phase, reference row order); the item lists
 * are CSR (item_off [N+1]) with precomputed in-session rankings (BaseModel.py:177-185) and min-max normalised float64
 * scores [nnz, K] (BaseModel.py:173); uhis_* / uitem_* are the per-user session / item histories of SeqReader
 * (helpers/SeqReader.py:18-60), CSR by user id; int_* is the CSR of the intent vectors, row 0 = the all-zero vector. */
typedef struct {
    int64_t N, K, I, max_his;     /* sessions, basic lists, intents, --history_max (0: unlimited) */
    int32_t nz1;                  /* entries per history row in the compact his_intents output (>= longest intent row) */
    const int64_t *u_id, *c_id, *context_mh, *user_mh, *pay, *fav, *click, *session_len, *position, *item_position, *intent_row;
    const int64_t *item_off, *item_id, *item_class, *ranking;
    const double  *scores;
    const int64_t *uhis_off, *uhis_row, *uhis_ctx;       /* [users+1], intent-row and context_mh of each history session */
    const int64_t *uitem_off, *uitem_id;                 /* [users+1], item ids of the user's positive items */
    const int32_t *uitem_int;                            /* behaviour * I / K + class of each of them (IntEL.py:226) */
    const int64_t *int_off;                              /* [rows+1] */
    const int32_t *int_idx;
    const double  *int_val;
} intel_corpus_t;
/* the batch in the layout intel_batch_t reads (compact history intents) + the fields the losses / evaluation need */
typedef struct {
    int64_t *u_id, *c_id, *context_mh, *user_mh, *pay, *fav, *click, *session_len, *position, *history_len, *history_item_len; /* [B] */
    int64_t *i_id, *i_class, *ranking;    /* [B,L], right-padded with 0 */
    double  *scores;                      /* [B,L,K] */
    double  *intents;                     /* [B,I] dense */
    int64_t *his_context;                 /* [B,H1] */
    int32_t *his_intents_idx;             /* [B,H1,nz1] */
    float   *his_intents_val;
    int64_t *his_item_id;                 /* [B,H2] */
    int32_t *his_item_int_idx;            /* [B,H2,1] */
    float   *his_item_int_val;
} intel_built_batch_t;
/* rows: device int64 [B] indices into the phase; perm: device int32 [B,L] or NULL - slot l of session b takes slot
 * perm[b,l] of its stored list (the per-fetch shuffle of BaseModel.py:194-196); L, H1, H2: padded widths of this batch. */
int intel_batch_build(const intel_corpus_t* corpus, int64_t B, const int64_t* rows, const int32_t* perm, int64_t L,
                      int64_t H1, int64_t H2, const intel_built_batch_t* out, intel_stream_t stream);

/* ---- optional per-kernel device timing (used by bench.py for the live roofline numbers) ------ */
/* While enabled every kernel launch is bracketed by CUDA events on its stream. */
int intel_profile_enable(int on);
/* Synchronises the device, then writes one text line per kernel name: "name launches total_ms
 * algorithmic_bytes flops" and clears the records. */
int intel_profile_report(char* buf, size_t cap);

/* ---- aWELv baseline (models/supervise/aWELv.py:28-39; script/baselines.sh:33) -----------------------------
 * w[b,:] = softmax_k <user_table[u_id[b]], model_table[k]>, weights[b,l,:] = w[b,:], ens[b,l] = sum_k w[b,k] scores[b,l,k].
 * user_table [users, h], model_table [K, h] (K <= 16), scores float64 [B,L,K]; w_user [B,K] is kept for the backward call,
 * which accumulates (+=) into the dense g_user_table / g_model_table; d_weights (nullable) [B,L,K], d_ens [B,L]. */
int intel_awelv_fwd(int64_t B, int64_t L, int K, int h, const float* user_table, const float* model_table, const int64_t* u_id,
                    const double* scores, float* weights, float* ens_score, float* w_user, intel_stream_t stream);
int intel_awelv_bwd(int64_t B, int64_t L, int K, int h, const float* user_table, const float* model_table, const int64_t* u_id,
                    const double* scores, const float* w_user, const float* d_weights, const float* d_ens, float* g_user_table,
                    float* g_model_table, intel_stream_t stream);

/* ---- aWELv_IntEL head (models/supervise/aWELv_IntEL.py:190-201) ------------------------------------------
 * The reference feeds the weight head the mean over all L list slots of the gated item / score streams; the head is
 * affine, so that equals the mean over the slots of the per-slot head output of the cross_attention = 0 path
 * (slot_weights [B,L,K] = the `weights` output of intel_ensemble_fwd with dims.cross_attention = 0):
 * p = softmax_k(mean_l slot_weights), w = softmax_k(p) (softmax twice, :197-198), weights[b,l,:] = w, ens = sum_k w_k scores.
 * p_sess, w_sess [B,K] are kept for the backward call, which writes d_slot_weights[b,l,k] = dlogits_k / L (every slot);
 * d_weights / d_ens nullable.  K <= 16. */
int intel_pool_head_fwd(int64_t B, int64_t L, int K, const float* slot_weights, const double* scores, float* weights,
                        float* ens_score, float* p_sess, float* w_sess, intel_stream_t stream);
int intel_pool_head_bwd(int64_t B, int64_t L, int K, const double* scores, const float* p_sess, const float* w_sess,
                        const float* d_weights, const float* d_ens, float* d_slot_weights, intel_stream_t stream);

/* ---- LambdaRank lambdas (helpers/LambdaRankRunner.py:315-344 compute_lambda_new, called at :246) ----------
 * lambdas[b,i] = sum_{j: t_i>t_j} Delta_ij Rho_ij - sum_{j: t_i<t_j} Delta_ji Rho_ji over the valid slots of session b, with
 * t = clamp(ranking, 0), Delta_ij = |g_i d_j + g_j d_i - g_i d_i - g_j d_j| / IDCG (g = 2^t - 1, d_j = 1/log2(j+2) of the list
 * SLOT j), Rho_ij = 1/(1+exp(s_i - s_j)).  ranking int64 [B,L] (raw or already clamped), scores float32 [B,L] (the
 * detached ens_score), session_len int64 [B] -> lambdas float32 [B,L]; pad slots get 0; a session without a positive
 * item gets NaN in all L slots, like the reference's 0/0. */
int intel_lambdarank_lambdas(int64_t B, int64_t L, const int64_t* ranking, const float* scores, const int64_t* session_len,
                             float* lambdas, intel_stream_t stream);

/* ---- optimizer step ------------------------------------------------------------------------------
 * torch.optim.Adam (BaseRunner._build_optimizer, BaseRunner.py:182-188) over `count` parameter tensors in one launch
 * per 48 tensors.  params / grads / exp_avg / exp_avg_sq / numel / weight_decay are HOST arrays of `count` entries
 * (device pointers, element counts, per-tensor L2 coefficient: BaseModel.customize_parameters gives the weights
 * `weight_decay` and the biases 0, BaseModel.py:53-62); step is the 1-based step number of this update. */
int intel_adam_step(int count, float* const* params, const float* const* grads, float* const* exp_avg,
                    float* const* exp_avg_sq, const int64_t* numel, const float* weight_decay, double lr, double beta1,
                    double beta2, double eps, int64_t step, intel_stream_t stream);

/* Row-wise form for sparse gradients: tensor i updates rows[i][0..nrows[i]) (distinct) of params / exp_avg / exp_avg_sq
 * ([*, dim[i]] row-major) with the compact gradient grads[i] [nrows[i], dim[i]], element by element as intel_adam_step
 * would with that gradient; all other rows are left untouched.  rows / grads are device pointers in HOST arrays. */
int intel_adam_rows_step(int count, float* const* params, float* const* exp_avg, float* const* exp_avg_sq,
                         const int64_t* const* rows, const float* const* grads, const int64_t* nrows, const int32_t* dim,
                         const float* weight_decay, double lr, double beta1, double beta2, double eps, int64_t step,
                         intel_stream_t stream);

/* Exact row-wise form (IntEL sparse_grad = 2): the zero-gradient updates that dense Adam gives the rows a step does not
 * name are deferred, and replayed in order through the same per-element arithmetic when the row is next updated or read,
 * so the result is bitwise intel_adam_step's.  Per tensor the caller owns (the library allocates nothing):
 *   n_updates[i]  the number of updates recorded since the bookkeeping was last reset, this step's included;
 *   hist[i]       device float [>= n, 8]: entry k holds the scalars of update k + 1 (lr / (1 - beta1^step),
 *                 sqrt(1 - beta2^step), beta2, eps, 1 - beta1, 1 - beta2, weight decay, 0);
 *   done[i]       device int32 [table rows], zero-filled before the first update: how many of the n updates row r has
 *                 received.  Invariant: row r of params / exp_avg / exp_avg_sq equals dense Adam after done[r] updates.
 * The step replays updates done[r] + 1 .. n - 1 on each listed row with a +0.0 gradient, applies update n with the row's
 * gradient, sets done[r] = n and stores update n's scalars to hist[n - 1].  A tensor with nrows[i] = 0 still records its
 * update.  rows / grads / done / hist are device pointers in HOST arrays. */
int intel_adam_deferred_rows_step(int count, float* const* params, float* const* exp_avg, float* const* exp_avg_sq,
                                  const int64_t* const* rows, const float* const* grads, const int64_t* nrows, const int32_t* dim,
                                  const float* weight_decay, int32_t* const* done, float* const* hist, const int32_t* n_updates,
                                  double lr, double beta1, double beta2, double eps, int64_t step, intel_stream_t stream);
/* Brings rows up to date (all n_updates[i] updates) without a new update.  rows[i] non-NULL: the first *row_count[i]
 * (a device int64, at most nrows[i]) distinct rows of rows[i], each left with done[r] = n.  rows[i] NULL: every one of the
 * nrows[i] rows of the table (a flush); done is then reset to 0 everywhere, and the caller restarts its count at 0. */
int intel_adam_deferred_catch_up(int count, float* const* params, float* const* exp_avg, float* const* exp_avg_sq,
                                 const int64_t* const* rows, const int64_t* const* row_count, const int64_t* nrows,
                                 const int32_t* dim, int32_t* const* done, const float* const* hist, const int32_t* n_updates,
                                 intel_stream_t stream);

/* ---- host-side input packing (no GPU work) ---------------------------------------------------
 * dense float64 [rows, I] host tensor (the reference's his_intents / his_item_int rows, collate_batch) -> the compact
 * form of intel_batch_t: idx int32 [rows, nz], val float32 [rows, nz], zero padded, both in host memory (pinned for
 * an asynchronous copy).  Scans with `threads` host threads (<= 0: all cores).  Returns the largest number of
 * non-zeros of any row: if it exceeds nz the rows were truncated and the caller retries with a larger nz or keeps the
 * dense layout; negative on error.  row_nnz (nullable) receives the per-row counts.
 * group > 0: rows come in groups of `group` (the H history slots of a session) and only the first group_len[g] rows of
 * group g are real (history_len / history_item_len); the padding rows behind them are emitted empty without being read. */
int64_t intel_host_pack_rows(int64_t rows, int64_t I, const double* dense, int32_t nz, int32_t* idx, float* val,
                             int32_t* row_nnz, int threads, int64_t group, const int64_t* group_len);

/* test hook: 0 routes the self-attention stacks through the staged kernels even where the fused per-session
 * kernel applies (both implement the same math; tests compare them). Default 1. */
int intel_debug_use_fused_stack(int on);
/* test hook: 0 keeps large GEMMs on the mma.sync kernels instead of the tcgen05 / TMEM kernel. Default 1. */
int intel_debug_use_tcgen05_gemm(int on);
/* test hook: 0 keeps the fused stack forward pass on the mma.sync kernel instead of the tcgen05 / TMEM kernel. Default 1. */
int intel_debug_use_tcgen05_stack(int on);
/* test hook: 0 keeps the GRU forward recurrence on the mma.sync kernel instead of the tcgen05 cluster kernel. Default 1. */
int intel_debug_use_tcgen05_gru(int on);
/* test hook: 0 keeps the tall resident-weight products and the tall weight gradients on the generic tcgen05 GEMM instead of the
 * persistent kernels (gemm_rows_tc.cu, gemm_wgrad_tc.cu). Default 1. */
int intel_debug_use_rows_gemm(int on);
/* test hook: 0 keeps the BERT4Rec encoder forward on the staged path instead of the fused kernel (bert_fused.cu). Default 1. */
int intel_debug_use_fused_bert(int on);
/* test hook: the index kernels behind the packed GRU path (pack_padded_sequence of GeneralSeq.py:64-71), for one encoder.
 * lens: device int64 [B]; T <= 63.  order: device int32 [B + 1], sessions by decreasing (clamped) length, stable, order[B] = 0;
 * rows_t / rows_t1: device int32 [B * T], the live (session, step) pairs in (b, t) order as row numbers b T + t / b (T + 1) + t;
 * count: device int32 [1] = number of live rows. */
int intel_debug_gru_prep(int64_t B, int64_t T, const int64_t* lens, int32_t* order, int32_t* rows_t, int32_t* rows_t1,
                         int32_t* count, intel_stream_t stream);
/* tuning / test hook: sessions that share one CTA (and one staged copy of the weights) in the fused stack
 * kernels, 1..4 (default 4).  The mma.sync forward kernel takes n as given; the backward kernel runs three sessions
 * for n >= 3 where their tiles fit in shared memory (L <= 56) and two otherwise. */
int intel_debug_stack_sessions_per_cta(int n);

/* ---- building blocks exposed for unit tests --------------------------------------------- */
/* out[r, :] = table[idx[r], :]  (nn.Embedding forward) */
int intel_gather_fwd(int64_t rows, int d, const float* table, const int64_t* idx, float* out, int ld_out,
                     int relu, intel_stream_t stream);
/* grad_table[idx[r], :] += d_out[r, :]  (embedding_dense_backward; dense grad) */
int intel_scatter_add_bwd(int64_t rows, int d, const float* d_out, int ld, const int64_t* idx,
                          float* grad_table, intel_stream_t stream);
/* C[M,N] = A[M,K] * W[N,K]^T + bias  (nn.Linear) - fp32 FFMA tiles */
int intel_linear_fwd(int64_t M, int64_t N, int64_t K, const float* A, const float* W, const float* bias,
                     float* C, intel_stream_t stream);

/* dX[M,K] = dY[M,N] * W[N,K] (optionally * (relu_mask[M,K] > 0));  dW[N,K] += dY^T X, db[N] += colsum(dY) */
int intel_linear_dx(int64_t M, int64_t N, int64_t K, const float* dY, const float* W, float* dX, const float* relu_mask,
                    intel_stream_t stream);
int intel_linear_dw(int64_t M, int64_t N, int64_t K, const float* dY, const float* X, float* dW, float* db,
                    intel_stream_t stream);
/* the same three passes with leading dimensions and the ReLU of an MLP folded in (nn.Sequential(Linear, ReLU, ...), e.g.
 * models/supervise/LambdaRank.py:30-37): relu_a applies max(.,0) to A on load, relu_mask [M,K] (pre-activations, leading
 * dimension ldmask) gates dX, relu_x applies max(.,0) to X on load.  W is [N,K] dense, dY is [M,N] dense. */
int intel_linear_fwd_ex(int64_t M, int64_t N, int64_t K, const float* A, int64_t lda, const float* W, const float* bias,
                        float* C, int64_t ldc, int relu_a, intel_stream_t stream);
int intel_linear_dx_ex(int64_t M, int64_t N, int64_t K, const float* dY, const float* W, float* dX, int64_t lddx,
                       const float* relu_mask, int64_t ldmask, intel_stream_t stream);
int intel_linear_dw_ex(int64_t M, int64_t N, int64_t K, const float* dY, const float* X, int64_t ldx, float* dW, float* db,
                       int relu_x, intel_stream_t stream);
/* P = softmax over each row of Z [R,N] (Tensor.softmax(dim=-1)); dZ = P * (dP - sum(P dP)) */
int intel_softmax_rows_fwd(int64_t R, int64_t N, const float* Z, float* P, intel_stream_t stream);
int intel_softmax_rows_bwd(int64_t R, int64_t N, const float* P, const float* dP, float* dZ, intel_stream_t stream);
/* layers.py MultiHeadAttention core on packed qkv [B,T,3d] -> out [B,T,d]; lens nullable (key mask) */
int intel_mha_fwd(int64_t B, int64_t T, int d, int heads, const float* qkv, const int64_t* lens, float* out,
                  intel_stream_t stream);
int intel_mha_bwd(int64_t B, int64_t T, int d, int heads, const float* qkv, const int64_t* lens, const float* d_out,
                  float* d_qkv, intel_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* INTEL_B200_H */
