// C-ABI orchestration of IntEL.predict_intent / predict_ensemble and their backward passes.
// Each entry point is a fixed sequence of kernel launches on the caller's stream; activations that
// the backward pass needs are left in the caller's workspace at offsets that depend only on dims.
#include "kernels.h"
#include "../../include/intel_b200.h"

using namespace intel;

namespace {

const int NZ_CAP = 16;   // compacted non-zeros kept per dense history row
inline int64_t pad4(int64_t n) { return (n + 3) & ~(int64_t)3; }
inline bool al16(const void* p) { return ((uintptr_t)p & 15) == 0; }

inline cudaStream_t S(intel_stream_t s) { return (cudaStream_t)s; }

int check_dims(const intel_dims_t* d) {
    INTEL_REQUIRE(d, INTEL_ERR_ARG, "dims is null");
    INTEL_REQUIRE(d->B > 0 && d->L > 0 && d->K > 0 && d->I > 0, INTEL_ERR_ARG, "bad batch dims B=%lld L=%lld K=%lld I=%lld",
                  (long long)d->B, (long long)d->L, (long long)d->K, (long long)d->I);
    INTEL_REQUIRE(d->heads > 0 && d->layers > 0, INTEL_ERR_ARG, "heads/layers must be positive");
    INTEL_REQUIRE((d->d_iid + d->d_im) % d->heads == 0 && d->d_s % d->heads == 0, INTEL_ERR_ARG,
                  "stream widths not divisible by num_heads");
    INTEL_REQUIRE(d->encoder == INTEL_ENCODER_BERT4REC || d->encoder == INTEL_ENCODER_GRU4REC, INTEL_ERR_ARG,
                  "Invalid sequence encoder.");
    INTEL_REQUIRE(d->encoder != INTEL_ENCODER_GRU4REC || d->gru_hidden == 128, INTEL_ERR_UNSUPPORTED,
                  "GRU4Rec needs gru_hidden = 128, the reference's GRU4RecEncoder(hidden_size=128)");
    INTEL_REQUIRE(d->bert_layers <= INTEL_MAX_BERT_LAYERS, INTEL_ERR_UNSUPPORTED, "too many BERT4Rec layers");
    return INTEL_OK;
}

// ================================================================================================
// self-attention stack (IntEL.py:182-197): N iterations sharing one set of weights
// ================================================================================================
int g_use_fused_stack = 1;

int stack_fwd(int64_t B, int64_t L, int d, int heads, int layers, const intel_selfatt_t& p, const StackWs& w, float drop_p,
              uint64_t drop_seed, int stream_id, cudaStream_t s, bool save = true) {
    const int64_t R = B * L;
    // whole stack of a session on chip: tcgen05 kernel (trunk_tc.cu, L <= 128) or the mma.sync kernel (trunk.cu, L <= 64);
    // both leave the same activations behind, which the fused and the staged backward passes read alike
    if (g_use_fused_stack && d == TD && trunk_fwd_supported(L, heads, layers))
        return trunk_fwd(B, L, heads, layers, p, w, drop_p, drop_seed, stream_id, s, save);
    for (int l = 0; l < layers; ++l) {
        INTEL_TRY(linear(R, d, d, w.X[l], d, p.wq, d, nullptr, w.QKV[l], 3 * d, s));
        INTEL_TRY(linear(R, d, d, w.X[l], d, p.wk, d, nullptr, w.QKV[l] + d, 3 * d, s));
        INTEL_TRY(linear(R, d, d, w.X[l], d, p.wv, d, nullptr, w.QKV[l] + 2 * d, 3 * d, s));
        INTEL_TRY(mha_fwd(B, L, d, heads, w.QKV[l], nullptr, w.A[l], s));
        INTEL_TRY(linear(R, d, d, w.A[l], d, p.w1, d, p.b1, w.U[l], d, s));
        if (drop_p > 0.f) {      // Z = dropout(relu(U) W2^T + b2) + X
            INTEL_TRY(linear(R, d, d, w.U[l], d, p.w2, d, p.b2, w.Z[l], d, s, /*relu_a=*/true));
            INTEL_TRY(dropout_apply(R, d, w.Z[l], w.X[l], w.Z[l], make_dropout(drop_p, drop_seed, stream_id, l), s));
        } else {
            INTEL_TRY(linear(R, d, d, w.U[l], d, p.w2, d, p.b2, w.Z[l], d, s, /*relu_a=*/true, false, w.X[l], d));
        }
        INTEL_TRY(layernorm_fwd(R, d, w.Z[l], p.lnw, p.lnb, w.X[l + 1], w.st[l], s));
    }
    return INTEL_OK;
}

// dX holds d(loss)/d X[layers] on entry and d(loss)/d X[0] on return.  t1, t2: [R,d] scratch; dqkv: [R,3d].
int stack_bwd(int64_t B, int64_t L, int d, int heads, int layers, const intel_selfatt_t& p, const intel_selfatt_t& g,
              const StackWs& w, float* dX, float* t1, float* t2, float* dqkv, float drop_p, uint64_t drop_seed, int stream_id,
              cudaStream_t s) {
    const int64_t R = B * L;
    if (g_use_fused_stack && trunk_supported(L, d, heads, layers))
        return trunk_bwd(B, L, heads, layers, p, g, w, dX, drop_p, drop_seed, stream_id, s);
    for (int l = layers - 1; l >= 0; --l) {
        float* dZ = t1;
        INTEL_TRY(layernorm_bwd(R, d, dX, w.Z[l], w.st[l], p.lnw, dZ, g.lnw, g.lnb, s));
        const float* dF = dZ;        // gradient of the FFN branch: dZ through the dropout mask (scratch: dqkv)
        if (drop_p > 0.f) {
            INTEL_TRY(dropout_apply(R, d, dZ, nullptr, dqkv, make_dropout(drop_p, drop_seed, stream_id, l), s));
            dF = dqkv;
        }
        INTEL_TRY(linear_dw(R, d, d, dF, d, w.U[l], d, g.w2, d, g.b2, s, /*relu_x=*/true));
        float* dU = t2;
        INTEL_TRY(linear_dx(R, d, d, dF, d, p.w2, d, dU, d, s, 0, w.U[l], d));
        INTEL_TRY(linear_dw(R, d, d, dU, d, w.A[l], d, g.w1, d, g.b1, s));
        float* dA = dX;   // dX is consumed
        INTEL_TRY(linear_dx(R, d, d, dU, d, p.w1, d, dA, d, s));
        INTEL_TRY(mha_bwd(B, L, d, heads, w.QKV[l], nullptr, dA, dqkv, s));
        INTEL_TRY(linear_dw(R, d, d, dqkv, 3 * d, w.X[l], d, g.wq, d, nullptr, s));
        INTEL_TRY(linear_dw(R, d, d, dqkv + d, 3 * d, w.X[l], d, g.wk, d, nullptr, s));
        INTEL_TRY(linear_dw(R, d, d, dqkv + 2 * d, 3 * d, w.X[l], d, g.wv, d, nullptr, s));
        INTEL_TRY(linear_dx(R, d, d, dqkv, 3 * d, p.wq, d, dX, d, s, 0));
        INTEL_TRY(linear_dx(R, d, d, dqkv + d, 3 * d, p.wk, d, dX, d, s, 1));
        INTEL_TRY(linear_dx(R, d, d, dqkv + 2 * d, 3 * d, p.wv, d, dX, d, s, 1));
        INTEL_TRY(add_inplace(R * d, dX, dZ, s));   // residual branch
    }
    return INTEL_OK;
}

// ================================================================================================
// ensemble workspace
// ================================================================================================
// The two self-attention streams of predict_ensemble, 0 = item and 1 = score: each has its width d, its column block
// [off, off + d) of the head input, and its own tensors in the parameters (or the gradients).
struct Stream {
    int d, off;
    const intel_selfatt_t* stack;
    float *xk, *xv;              // intent_*_attention.{key,value}_layer (cross_attention = 1)
    float *w0, *b0, *w2;         // intent_*_embeddings.{0,2} (cross_attention = 0)
};
void streams_of(const intel_dims_t* d, const intel_tensors_t* T, Stream (&st)[2]) {
    const int di = d->d_iid + d->d_im;
    st[0] = {di, 0, &T->item, T->xk_item, T->xv_item, T->gate_item_w0, T->gate_item_b0, T->gate_item_w2};
    st[1] = {d->d_s, di, &T->score, T->xk_score, T->xv_score, T->gate_score_w0, T->gate_score_b0, T->gate_score_w2};
}

// The three weights that read the predicted intents (query_layer of each stream, intent_embeddings) already back to back,
// as the [di + ds + dint, I] matrix Wcat of the one product against the intents
bool intent_weights_stacked(const intel_tensors_t* T, int di, int ds, int64_t I) {
    return T->xq_score == T->xq_item + (int64_t)di * I && T->intent_w == T->xq_score + (int64_t)ds * I;
}

struct EnsWs {
    StackWs stack[2];             // per stream
    float* xs;                    // float copy of the scores [R,K]
    float *q[2], *qk[2], *p[2], *xbar[2];   // cross attention, per stream
    // the three products that read the predicted intents ([B, I] x {query_layer (item), query_layer (score),
    // intent_embeddings}) run as one: Wcat [di + ds + dint, I] = the three weights stacked, qcat / dcat [B, di + ds + dint]
    float *Wcat, *qcat, *dcat;
    float* all;                   // [B, D] head input of the valid rows
    float *w_valid, *w_pad;       // [B,K]
    float *t[2], *m[2], *hu, *hint, *all_item;                      // cross_attention = 0
    // backward scratch
    float *dall, *dwv, *dwp, *dxbar, *dqk, *dq, *dX[2], *t1, *t2, *dqkv;   // dX: d(stack output) of each stream
    float *g, *dall_item, *dm, *dt, *dvec;
};

void ens_layout(const intel_dims_t* d, Arena& a, EnsWs& w) {
    const int64_t B = d->B, L = d->L, R = B * L;
    const int di = d->d_iid + d->d_im, ds = d->d_s, D = di + ds + d->d_u + d->d_int;
    const int dmax = di > ds ? di : ds, dst[2] = {di, ds};
    for (int st = 0; st < 2; ++st) stack_layout(a, R, dst[st], d->layers, w.stack[st]);
    w.xs = a.take<float>(R * d->K);
    w.all = a.take<float>(B * D);
    w.w_valid = a.take<float>(B * d->K);
    w.w_pad = a.take<float>(B * d->K);
    w.dall = a.take<float>(B * D);
    w.dwv = a.take<float>(B * d->K);
    w.dwp = a.take<float>(B * d->K);
    for (float*& x : w.dX) x = a.take<float>(R * dmax);
    w.t1 = a.take<float>(R * dmax);
    w.t2 = a.take<float>(R * dmax);
    w.dqkv = a.take<float>(R * 3 * dmax);
    if (d->cross_attention) {
        const int dc = di + ds + d->d_int;
        w.Wcat = a.take<float>((int64_t)dc * d->I);
        w.qcat = a.take<float>(B * dc);
        w.dcat = a.take<float>(B * dc);
        w.q[0] = w.qcat; w.q[1] = w.qcat + di;                  // column blocks of qcat (row stride dc)
        for (int st = 0; st < 2; ++st) w.qk[st] = a.take<float>(B * dst[st]);
        for (float*& x : w.p) x = a.take<float>(B * L);
        for (int st = 0; st < 2; ++st) w.xbar[st] = a.take<float>(B * dst[st]);
        w.dxbar = a.take<float>(B * dmax);
        w.dqk = a.take<float>(B * dmax);
        w.dq = a.take<float>(B * dmax);
    } else {
        for (float*& x : w.t) x = a.take<float>(B * d->qsize);
        for (int st = 0; st < 2; ++st) w.m[st] = a.take<float>(B * dst[st]);
        w.hu = a.take<float>(B * d->d_u); w.hint = a.take<float>(B * d->d_int);
        w.all_item = a.take<float>(R * D);
        w.g = a.take<float>(R * d->K);
        w.dall_item = a.take<float>(R * D);
        w.dm = a.take<float>(B * dmax);
        w.dt = a.take<float>(B * d->qsize);
        w.dvec = a.take<float>(B * (d->d_u > d->d_int ? d->d_u : d->d_int));
    }
}

// ================================================================================================
// intent predictor workspace
// ================================================================================================
struct BertWs {
    float* X[INTEL_MAX_BERT_LAYERS + 1];
    float *QKV[INTEL_MAX_BERT_LAYERS], *Z1[INTEL_MAX_BERT_LAYERS], *st1[INTEL_MAX_BERT_LAYERS], *C[INTEL_MAX_BERT_LAYERS],
        *F[INTEL_MAX_BERT_LAYERS], *Z2[INTEL_MAX_BERT_LAYERS], *st2[INTEL_MAX_BERT_LAYERS];
};
// rows_t / rows_t1 / nlive: the live-row lists (gru_prep), null when int32 cannot address every row of [B, T + 1, .];
// order: the length-sorted sessions, null when T > 63
struct GruWs { float *gi, *h_all, *gates, *dh, *dgi, *dgh_all; int32_t *order, *rows_t, *rows_t1, *nlive; };
struct EncWs {
    int64_t T; int d;
    float* seq;          // [B*T, d] token embeddings (BERT: positions added in place)
    int32_t* nz_idx; float* nz_val; int32_t* nz_cnt;
    BertWs bert; GruWs gru;
    float* dseq;
};
struct IntWs {
    float* Wt;           // [I, d_int] transpose of intent_embeddings.weight
    float* dWt;
    EncWs e[2];          // per history
    float *feat, *logits, *dlogits, *dfeat;
    float *t1, *t2, *dqkv;   // bert backward scratch
};

// The two histories of predict_intent, 0 = session history (encoder), 1 = item history (item_encoder).  A token of a
// history is [table row of its id | intent embedding of its intents], split at column dtok; the intents are dense float64
// rows [B*T, I] or, when idx is set, nz compact entries per row.  The encoded history goes to columns [off, off + d) of feat.
struct History {
    const float* table; float* gtable; const int64_t* ids; int64_t table_rows; const int32_t* map; int dtok;
    const double* dense; const char* dense_name; const int32_t* idx; const float* val; int nz;
    const int64_t* lens;
    int off;
    const intel_encoder_t* p; intel_encoder_t* g;
};
// G and M may be null (the forward pass)
void histories_of(const intel_dims_t* d, const intel_tensors_t* P, intel_tensors_t* G, const intel_row_maps_t* M,
                  const intel_batch_t* bt, History (&h)[2]) {
    const int off2 = d->d_ctx + d->d_u, off1 = off2 + d->d_iid + d->d_int;   // pred_layer input = [ctx | user | item-history | history]
    h[0] = {P->ctx_emb, G ? G->ctx_emb : nullptr, bt->his_context, d->ctx_rows, M ? M->ctx : nullptr, d->d_ctx,
            bt->his_intents, "his_intents", bt->his_intents_idx, bt->his_intents_val, bt->nz1,
            bt->history_len, off1, &P->enc, G ? &G->enc : nullptr};
    h[1] = {P->iid_emb, G ? G->iid_emb : nullptr, bt->his_item_id, d->item_rows, M ? M->iid : nullptr, d->d_iid,
            bt->his_item_int, "his_item_int", bt->his_item_int_idx, bt->his_item_int_val, bt->nz2,
            bt->history_item_len, off2, &P->item_enc, G ? &G->item_enc : nullptr};
}

void enc_layout(const intel_dims_t* d, Arena& a, EncWs& e, int64_t T, int dd) {
    const int64_t B = d->B, R = B * T;
    e.T = T; e.d = dd;
    e.seq = a.take<float>(R * dd);
    e.nz_idx = a.take<int32_t>(R * NZ_CAP);
    e.nz_val = a.take<float>(R * NZ_CAP);
    e.nz_cnt = a.take<int32_t>(R);
    e.dseq = a.take<float>(R * dd);
    if (d->encoder == INTEL_ENCODER_BERT4REC) {
        e.bert.X[0] = e.seq;
        for (int l = 0; l < d->bert_layers; ++l) {
            e.bert.QKV[l] = a.take<float>(R * 3 * dd);
            e.bert.Z1[l] = a.take<float>(R * dd);
            e.bert.st1[l] = a.take<float>(R * 2);
            e.bert.C[l] = a.take<float>(R * dd);
            e.bert.F[l] = a.take<float>(R * dd);
            e.bert.Z2[l] = a.take<float>(R * dd);
            e.bert.st2[l] = a.take<float>(R * 2);
            e.bert.X[l + 1] = a.take<float>(R * dd);
        }
    } else {
        const int h = d->gru_hidden;
        e.gru.gi = a.take<float>(R * 3 * h);
        e.gru.h_all = a.take<float>(B * (T + 1) * h);
        e.gru.gates = a.take<float>(R * 4 * h);
        e.gru.dh = a.take<float>(B * h);
        e.gru.dgi = a.take<float>(R * 3 * h);
        e.gru.dgh_all = a.take<float>(B * (T + 1) * 3 * h);
        e.gru.order = T <= 63 ? a.take<int32_t>(B + 1) : nullptr;
        const bool packed = B * (T + 1) < (1LL << 31);
        e.gru.rows_t = packed ? a.take<int32_t>(R) : nullptr;
        e.gru.rows_t1 = packed ? a.take<int32_t>(R) : nullptr;
        e.gru.nlive = packed ? a.take<int32_t>(4) : nullptr;
    }
}

void int_layout(const intel_dims_t* d, Arena& a, IntWs& w) {
    const int d1 = d->d_ctx + d->d_int, d2 = d->d_iid + d->d_int;
    const int Dp = d1 + d2 + d->d_ctx + d->d_u;
    w.Wt = a.take<float>(d->I * d->d_int);
    w.dWt = a.take<float>(d->I * d->d_int);
    enc_layout(d, a, w.e[0], d->H1, d1);
    enc_layout(d, a, w.e[1], d->H2, d2);
    w.feat = a.take<float>(d->B * Dp);
    w.logits = a.take<float>(d->B * pad4(d->I));       // rows padded to 16 bytes: intent_num is odd in every config
    w.dlogits = a.take<float>(d->B * pad4(d->I));
    w.dfeat = a.take<float>(d->B * Dp);
    const int64_t r1 = d->B * d->H1 * d1, r2 = d->B * d->H2 * d2;
    const int64_t rm = r1 > r2 ? r1 : r2;
    w.t1 = a.take<float>(rm);
    w.t2 = a.take<float>(rm);
    w.dqkv = a.take<float>(3 * rm);
}

// ---- BERT4RecEncoder (GeneralSeq.py:80-106, layers.py:62-88) --------------------------------------
int bert_fwd(const intel_dims_t* d, const intel_encoder_t& p, EncWs& e, const int64_t* lens, float* out, int64_t ld_out,
             cudaStream_t s) {
    const int64_t B = d->B, T = e.T, R = B * T;
    const int dd = e.d;
    INTEL_REQUIRE(T <= d->history_max + 1, INTEL_ERR_ARG, "history length %lld exceeds history_max+1", (long long)T);
    if (bert_fused_ok(T, dd, d->bert_heads, d->bert_layers)) {       // the whole encoder in one kernel (bert_fused.cu)
        BertWs& w = e.bert;
        return bert_fused_fwd(B, T, d->bert_heads, d->bert_layers, lens, p, e.seq, w.X, w.QKV, w.Z1, w.st1, w.C, w.F, w.Z2, w.st2,
                              d->inference == 0, out, ld_out, s);
    }
    INTEL_TRY(add_positions(B, T, dd, lens, p.pos, e.seq, s));
    for (int l = 0; l < d->bert_layers; ++l) {
        const intel_bert_layer_t& q = p.layer[l];
        BertWs& w = e.bert;
        INTEL_TRY(linear(R, dd, dd, w.X[l], dd, q.qw, dd, q.qb, w.QKV[l], 3 * dd, s));
        INTEL_TRY(linear(R, dd, dd, w.X[l], dd, q.kw, dd, q.kb, w.QKV[l] + dd, 3 * dd, s));
        INTEL_TRY(linear(R, dd, dd, w.X[l], dd, q.vw, dd, q.vb, w.QKV[l] + 2 * dd, 3 * dd, s));
        INTEL_TRY(mha_fwd(B, T, dd, d->bert_heads, w.QKV[l], lens, w.Z1[l], s));
        INTEL_TRY(add_inplace(R * dd, w.Z1[l], w.X[l], s));
        INTEL_TRY(layernorm_fwd(R, dd, w.Z1[l], q.ln1w, q.ln1b, w.C[l], w.st1[l], s));
        INTEL_TRY(linear(R, dd, dd, w.C[l], dd, q.l1w, dd, q.l1b, w.F[l], dd, s));
        INTEL_TRY(linear(R, dd, dd, w.F[l], dd, q.l2w, dd, q.l2b, w.Z2[l], dd, s, true, false, w.C[l], dd));
        INTEL_TRY(layernorm_fwd(R, dd, w.Z2[l], q.ln2w, q.ln2b, w.X[l + 1], w.st2[l], s));
    }
    return take_last(B, T, dd, lens, e.bert.X[d->bert_layers], out, ld_out, s);
}

int bert_bwd(const intel_dims_t* d, const intel_encoder_t& p, intel_encoder_t& g, EncWs& e, const int64_t* lens,
             const float* dout, int64_t ld, float* t1, float* t2, float* dqkv, cudaStream_t s) {
    const int64_t B = d->B, T = e.T, R = B * T;
    const int dd = e.d;
    float* dX = e.dseq;
    INTEL_TRY(fill_zero(dX, (size_t)R * dd * 4, s));
    INTEL_TRY(take_last_bwd(B, T, dd, lens, dout, ld, dX, s));
    for (int l = d->bert_layers - 1; l >= 0; --l) {
        const intel_bert_layer_t& q = p.layer[l];
        intel_bert_layer_t& gq = g.layer[l];
        BertWs& w = e.bert;
        float* dZ2 = t1;
        INTEL_TRY(layernorm_bwd(R, dd, dX, w.Z2[l], w.st2[l], q.ln2w, dZ2, gq.ln2w, gq.ln2b, s));
        INTEL_TRY(linear_dw(R, dd, dd, dZ2, dd, w.F[l], dd, gq.l2w, dd, gq.l2b, s, true));
        float* dF = t2;
        INTEL_TRY(linear_dx(R, dd, dd, dZ2, dd, q.l2w, dd, dF, dd, s, 0, w.F[l], dd));
        INTEL_TRY(linear_dw(R, dd, dd, dF, dd, w.C[l], dd, gq.l1w, dd, gq.l1b, s));
        float* dC = dX;
        INTEL_TRY(linear_dx(R, dd, dd, dF, dd, q.l1w, dd, dC, dd, s));
        INTEL_TRY(add_inplace(R * dd, dC, dZ2, s));
        float* dZ1 = t1;
        INTEL_TRY(layernorm_bwd(R, dd, dC, w.Z1[l], w.st1[l], q.ln1w, dZ1, gq.ln1w, gq.ln1b, s));
        INTEL_TRY(mha_bwd(B, T, dd, d->bert_heads, w.QKV[l], lens, dZ1, dqkv, s));
        INTEL_TRY(linear_dw(R, dd, dd, dqkv, 3 * dd, w.X[l], dd, gq.qw, dd, gq.qb, s));
        INTEL_TRY(linear_dw(R, dd, dd, dqkv + dd, 3 * dd, w.X[l], dd, gq.kw, dd, gq.kb, s));
        INTEL_TRY(linear_dw(R, dd, dd, dqkv + 2 * dd, 3 * dd, w.X[l], dd, gq.vw, dd, gq.vb, s));
        INTEL_TRY(linear_dx(R, dd, dd, dqkv, 3 * dd, q.qw, dd, dX, dd, s, 0));
        INTEL_TRY(linear_dx(R, dd, dd, dqkv + dd, 3 * dd, q.kw, dd, dX, dd, s, 1));
        INTEL_TRY(linear_dx(R, dd, dd, dqkv + 2 * dd, 3 * dd, q.vw, dd, dX, dd, s, 1));
        INTEL_TRY(add_inplace(R * dd, dX, dZ1, s));
    }
    return add_positions_bwd(B, T, dd, lens, dX, g.pos, s);
}

// ---- GRU4RecEncoder (GeneralSeq.py:58-78) ----------------------------------------------------------
// Both GRU encoders of predict_intent (session history, item history) in three stages: input projections, recurrences,
// output projections.  The recurrences of the two encoders share one launch (gru_tc.cu): each is a chain of T dependent steps
// that leaves the tensor pipe idle most of the time, so they are overlapped instead of run back to back.
int gru_fwd_pair(const intel_dims_t* d, const History (&hs)[2], EncWs (&e)[2], float* feat, int64_t ld_out, cudaStream_t s) {
    const int64_t B = d->B;
    const int h = d->gru_hidden;
    GruPrepOne prep[2];         // live rows and length order of both encoders: one launch
    for (int i = 0; i < 2; ++i) {
        const GruWs& w = e[i].gru;
        prep[i] = GruPrepOne{B, (int)e[i].T, hs[i].lens, w.rows_t, w.rows_t1, w.nlive, w.order};
    }
    INTEL_TRY(gru_prep(2, prep, s));
    for (int i = 0; i < 2; ++i) {
        const int64_t T = e[i].T, R = B * T;
        const int dd = e[i].d;
        GruWs& w = e[i].gru;
        // the products over the [B, T] history rows walk the live rows only (about half of them are padding behind a
        // session's length; the reference packs the sequences: GeneralSeq.py:64-71).  gi rows of padding slots stay
        // unwritten: nobody reads them.
        INTEL_TRY(linear(R, 3 * h, dd, e[i].seq, dd, hs[i].p->w_ih, dd, hs[i].p->b_ih, w.gi, 3 * h, s, false, false, nullptr, 0,
                         w.rows_t, w.nlive));
        // the recurrence kernels write h_all[:, 1..T] of every session themselves: only the initial state h_0 needs clearing
        cudaError_t ce = cudaMemset2DAsync(w.h_all, (size_t)(T + 1) * h * 4, 0, (size_t)h * 4, (size_t)B, s);
        INTEL_REQUIRE(ce == cudaSuccess, INTEL_ERR_CUDA, "cudaMemset2DAsync: %s", cudaGetErrorString(ce));
    }
    if (gru_tc_supported()) {
        GruTcPair pr;
        pr.n = 2;
        pr.save_gates = d->inference == 0;
        for (int i = 0; i < 2; ++i) {
            GruWs& w = e[i].gru;
            pr.e[i] = GruTcOne{B, e[i].T, hs[i].lens, w.gi, hs[i].p->w_hh, hs[i].p->b_hh, w.h_all, w.gates, w.order};
        }
        INTEL_TRY(gru_tc_fwd_pair(pr, s));
    } else {
        for (int i = 0; i < 2; ++i) {
            GruWs& w = e[i].gru;
            INTEL_TRY(gru_seq_fwd(B, e[i].T, hs[i].lens, w.gi, hs[i].p->w_hh, hs[i].p->b_hh, w.h_all, w.gates, s));
        }
    }
    if (gru_outproj_pair_ok(e[0].d, e[1].d)) {          // both output projections in one launch
        const int n[2] = {e[0].d, e[1].d};
        const float* W[2] = {hs[0].p->w_out, hs[1].p->w_out};
        const float* hl[2] = {e[0].gru.h_all + e[0].T * h, e[1].gru.h_all + e[1].T * h};
        float* const out[2] = {feat + hs[0].off, feat + hs[1].off};
        const int64_t ldh[2] = {(e[0].T + 1) * h, (e[1].T + 1) * h}, ldo[2] = {ld_out, ld_out};
        return gru_outproj_pair_fwd(B, n, W, hl, ldh, out, ldo, s);
    }
    for (int i = 0; i < 2; ++i) {
        const int64_t T = e[i].T;
        GruWs& w = e[i].gru;
        INTEL_TRY(linear(B, e[i].d, h, w.h_all + T * h, (T + 1) * h, hs[i].p->w_out, h, nullptr, feat + hs[i].off, ld_out, s));
    }
    return INTEL_OK;
}

// Backward pass of both GRU encoders; w.dh holds d(last state) on entry (intel_intent_bwd_rows forms it for both).
// The products of each encoder after the recurrence: dW_hh += dgh_all^T h_all over the [B, T+1] rows, dW_ih += dgi^T seq
// and d(seq) = dgi W_ih over the [B, T] rows, each over the live rows alone when the encoder has the live-row lists.
struct GruBwdProducts { Gemm whh, wih, dseq; };
int gru_bwd_pair(const intel_dims_t* d, const History (&hs)[2], EncWs (&e)[2], const float* dfeat, int64_t ld, cudaStream_t s) {
    const int64_t B = d->B;
    const int h = d->gru_hidden;
    GruBwdProducts pr[2];
    GruBwdPair rec;
    for (int i = 0; i < 2; ++i) {
        const int64_t T = e[i].T, R = B * T;
        const int dd = e[i].d;
        GruWs& w = e[i].gru;
        const intel_encoder_t &p = *hs[i].p, &g = *hs[i].g;
        INTEL_TRY(linear_dw(B, dd, h, dfeat + hs[i].off, ld, w.h_all + T * h, (T + 1) * h, g.w_out, h, nullptr, s));
        pr[i].whh = wgrad_gemm(B * (T + 1), 3 * h, h, w.dgh_all, 3 * h, w.h_all, h, g.w_hh, h, w.rows_t1, w.nlive);
        pr[i].wih = wgrad_gemm(R, 3 * h, dd, w.dgi, 3 * h, e[i].seq, dd, g.w_ih, dd, w.rows_t, w.nlive);
        pr[i].dseq = dgrad_gemm(R, 3 * h, dd, w.dgi, 3 * h, p.w_ih, dd, e[i].dseq, dd, w.rows_t, w.nlive);
        // when all three products read the live rows alone, the recurrence writes nothing for the padding slots (about half
        // of the [B, T] rows); otherwise it writes their gradient rows as zeros, and slot T of dgh_all, which pairs with the
        // final state in the dW_hh product, is cleared here
        const bool live_only = gemm_rows_only(pr[i].whh) && gemm_rows_only(pr[i].wih) && gemm_rows_only(pr[i].dseq);
        if (!live_only) {
            cudaError_t ce = cudaMemset2DAsync(w.dgh_all + T * 3 * h, (size_t)(T + 1) * 3 * h * 4, 0, (size_t)3 * h * 4, (size_t)B, s);
            INTEL_REQUIRE(ce == cudaSuccess, INTEL_ERR_CUDA, "cudaMemset2DAsync: %s", cudaGetErrorString(ce));
        }
        // with the length order, tiles of equally long sessions stop at their own last step; the order is the forward call's,
        // its tile counter (order[B]) is reset here
        if (w.order) INTEL_TRY(fill_zero(w.order + B, sizeof(int32_t), s));
        // the recurrence also sums the bias gradients (column sums of dgi / dgh) on its way
        rec.e[i] = GruBwdOne{B, T, hs[i].lens, p.w_hh, w.h_all, w.gates, w.dh, w.dgi, w.dgh_all, g.b_ih, g.b_hh, w.order,
                             w.order ? w.order + B : nullptr, live_only ? 1 : 0};
    }
    // one launch for both recurrences when both have the length order (their tiles are drawn from its counters), else one each
    if (rec.e[0].counter && rec.e[1].counter) {
        rec.n = 2;
        INTEL_TRY(gru_seq_bwd_pair(rec, s));
    } else {
        for (int i = 0; i < 2; ++i) {
            GruBwdPair one;
            one.e[0] = rec.e[i];
            one.n = 1;
            INTEL_TRY(gru_seq_bwd_pair(one, s));
        }
    }
    for (int i = 0; i < 2; ++i) {
        INTEL_TRY(gemm(pr[i].whh, s));
        INTEL_TRY(gemm(pr[i].wih, s));
        // d(seq) of the padding slots is cleared for the scatters that read every row
        if (e[i].gru.rows_t) INTEL_TRY(fill_zero(e[i].dseq, (size_t)B * e[i].T * e[i].d * 4, s));
        INTEL_TRY(gemm(pr[i].dseq, s));
    }
    return INTEL_OK;
}

}  // namespace

extern "C" {

int intel_debug_use_fused_stack(int on) {
    g_use_fused_stack = on ? 1 : 0;
    return INTEL_OK;
}

int intel_debug_use_tcgen05_gemm(int on) {
    gemm_debug_use_tcgen05(on);
    return INTEL_OK;
}

int intel_debug_use_rows_gemm(int on) {
    gemm_debug_use_rows_gemm(on);
    return INTEL_OK;
}

int intel_debug_gru_prep(int64_t B, int64_t T, const int64_t* lens, int32_t* order, int32_t* rows_t, int32_t* rows_t1,
                         int32_t* count, intel_stream_t stream) {
    INTEL_REQUIRE(lens && order && rows_t && rows_t1 && count, INTEL_ERR_ARG, "gru_prep: null argument");
    INTEL_REQUIRE(T >= 0 && T < (1LL << 31), INTEL_ERR_ARG, "gru_prep: bad history length %lld", (long long)T);
    const GruPrepOne one{B, (int)T, lens, rows_t, rows_t1, count, order};
    return gru_prep(1, &one, S(stream));
}

int intel_debug_use_fused_bert(int on) {
    bert_debug_use_fused(on);
    return INTEL_OK;
}

int intel_debug_use_tcgen05_gru(int on) {
    gru_debug_use_tcgen05(on);
    return INTEL_OK;
}

int intel_debug_use_tcgen05_stack(int on) {
    trunk_debug_use_tcgen05(on);
    return INTEL_OK;
}

int intel_reserve_sms(int n) {
    INTEL_REQUIRE(n >= 0 && n <= 64, INTEL_ERR_ARG, "reserve_sms: n must be in [0, 64]");
    trunk_reserve_sms(n);
    return INTEL_OK;
}

int intel_debug_stack_sessions_per_cta(int n) {
    trunk_debug_sessions_per_cta(n);
    return INTEL_OK;
}

// ================================================================================================
size_t intel_ensemble_workspace_bytes(const intel_dims_t* d) {
    if (check_dims(d) != INTEL_OK) return 0;
    Arena a(nullptr, 0);
    EnsWs w;
    ens_layout(d, a, w);
    return a.off + 256;
}

int intel_ensemble_fwd(const intel_dims_t* d, const intel_tensors_t* P, const intel_batch_t* bt, const float* intents,
                       float* weights_out, float* ens_out, void* workspace, size_t workspace_bytes,
                       intel_stream_t stream) {
    INTEL_TRY(check_dims(d));
    INTEL_REQUIRE(P && bt && intents && weights_out && ens_out, INTEL_ERR_ARG, "ensemble_fwd: null argument");
    INTEL_REQUIRE(d->layers <= 8, INTEL_ERR_UNSUPPORTED, "num_layers > 8");
    INTEL_REQUIRE((d->d_im > 0) == (bt->i_class != nullptr), INTEL_ERR_ARG, "i_class / im_emb_size mismatch");
    Arena a(workspace, workspace_bytes);
    EnsWs w;
    ens_layout(d, a, w);
    INTEL_REQUIRE(workspace && a.ok(), INTEL_ERR_WORKSPACE, "ensemble workspace too small: need %zu", a.off);
    cudaStream_t s = S(stream);
    const int64_t B = d->B, L = d->L, R = B * L, I = d->I;
    const int K = (int)d->K, di = d->d_iid + d->d_im, ds = d->d_s, du = d->d_u, dint = d->d_int;
    const int D = di + ds + du + dint, off_u = di + ds, off_h = di + ds + du;
    Stream ps[2];
    streams_of(d, P, ps);

    // embedding gathers straight into the concatenated item-stream rows (IntEL.py:170-175)
    INTEL_TRY(gather_rows(R, d->d_iid, P->iid_emb, bt->i_id, w.stack[0].X[0], di, 0, s, d->item_rows));
    if (d->d_im > 0) INTEL_TRY(gather_rows(R, d->d_im, P->item_emb, bt->i_class, w.stack[0].X[0] + d->d_iid, di, 0, s, d->class_rows));
    INTEL_TRY(score_embed_fwd(R, K, ds, bt->scores, P->score_w, P->score_b, w.stack[1].X[0], w.xs, s));
    for (int st = 0; st < 2; ++st)     // stream_id st: the two stacks draw different dropout masks
        INTEL_TRY(stack_fwd(B, L, ps[st].d, d->heads, d->layers, *ps[st].stack, w.stack[st], d->dropout_p, d->dropout_seed, st, s,
                            d->inference == 0));

    if (d->cross_attention) {
        const float scale = 1.0f / sqrtf((float)d->qsize);
        // q_item | q_score | intent_embeddings(intent): one product over the predicted intents (read once instead of
        // three times); the weights are stacked into Wcat unless the caller already keeps them back to back
        const int dc = di + ds + dint;
        const float* Wc = P->xq_item;
        if (!intent_weights_stacked(P, di, ds, I)) {
            INTEL_TRY(copy_d2d(w.Wcat, P->xq_item, (size_t)di * I * 4, s));
            INTEL_TRY(copy_d2d(w.Wcat + (int64_t)di * I, P->xq_score, (size_t)ds * I * 4, s));
            INTEL_TRY(copy_d2d(w.Wcat + (int64_t)(di + ds) * I, P->intent_w, (size_t)dint * I * 4, s));
            Wc = w.Wcat;
        }
        INTEL_TRY(linear(B, dc, I, intents, I, Wc, I, nullptr, w.qcat, dc, s));
        // per stream: qk = W_k^T q, the pooling, the value projection into the head input
        for (int st = 0; st < 2; ++st) {
            const Stream& c = ps[st];
            const float* X = w.stack[st].X[d->layers];
            if (cross_full_ok(c.d, L) && al16(c.xk) && al16(c.xv)) {
                INTEL_TRY(cross_full_fwd(B, L, X, w.q[st], dc, c.xk, c.xv, bt->session_len, scale, w.p[st], w.qk[st], w.xbar[st],
                                         w.all + c.off, D, s));
            } else {
                INTEL_TRY(linear_dx(B, c.d, c.d, w.q[st], dc, c.xk, c.d, w.qk[st], c.d, s));            // qk = W_k^T q
                INTEL_TRY(cross_pool_fwd(B, L, c.d, X, w.qk[st], bt->session_len, scale, w.p[st], w.xbar[st], s));
                INTEL_TRY(linear(B, c.d, c.d, w.xbar[st], c.d, c.xv, c.d, nullptr, w.all + c.off, D, s));
            }
        }
        // user + intent parts of the head input
        INTEL_TRY(gather_rows(B, du, P->uid_emb, bt->u_id, w.all + off_u, D, 1, s, d->user_rows));
        INTEL_TRY(bias_relu_rows(B, dint, w.qcat + di + ds, dc, P->intent_b, w.all + off_h, D, s));
        // weights of the valid rows and of the pad rows (whose pooled inputs are zero), then the fusion
        if (head_full_ok(K, D)) {
            INTEL_TRY(head_full_fwd(B, L, K, D, off_u, w.all, P->head_w, P->head_b, bt->scores, bt->session_len, weights_out, ens_out, s));
        } else {
            INTEL_TRY(linear(B, K, D, w.all, D, P->head_w, D, P->head_b, w.w_valid, K, s));
            INTEL_TRY(linear(B, K, du + dint, w.all + off_u, D, P->head_w + off_u, D, P->head_b, w.w_pad, K, s));
            INTEL_TRY(head_fuse_fwd(B, L, K, w.w_valid, w.w_pad, bt->scores, bt->session_len, weights_out, ens_out, s));
        }
    } else {
        const int q = d->qsize;
        for (int st = 0; st < 2; ++st) {
            const Stream& c = ps[st];
            INTEL_TRY(linear(B, q, I, intents, I, c.w0, I, c.b0, w.t[st], q, s, false, true));
            INTEL_TRY(linear(B, c.d, q, w.t[st], q, c.w2, q, nullptr, w.m[st], c.d, s));
        }
        for (int st = 0; st < 2; ++st)
            INTEL_TRY(gate_fwd(B, L, ps[st].d, w.stack[st].X[d->layers], w.m[st], w.all_item + ps[st].off, D, s));
        INTEL_TRY(gather_rows(B, du, P->uid_emb, bt->u_id, w.hu, du, 1, s, d->user_rows));
        INTEL_TRY(bcast_rows(B, L, du, w.hu, du, w.all_item + off_u, D, s));
        INTEL_TRY(linear(B, dint, I, intents, I, P->intent_w, I, P->intent_b, w.hint, dint, s, false, true));
        INTEL_TRY(bcast_rows(B, L, dint, w.hint, dint, w.all_item + off_h, D, s));
        INTEL_TRY(linear(R, K, D, w.all_item, D, P->head_w, D, P->head_b, weights_out, K, s));
        INTEL_TRY(item_fuse_fwd(R, K, weights_out, bt->scores, ens_out, s));
    }
    return INTEL_OK;
}

// The backward pass in three phases (INTEL_ENS_BWD_*): HEAD = weight head + both pooled cross attentions (d_intents_out is
// final afterwards, d(stack output) of each stream is left in the workspace), ITEM / SCORE = the self-attention stack of
// one stream and the gradients of its inputs.  A data-parallel caller runs HEAD, intel_intent_bwd, ITEM - after which every
// gradient except the score stream's is final and can be exchanged - and hides that exchange behind SCORE.
int intel_ensemble_bwd_phase_rows(const intel_dims_t* d, const intel_tensors_t* P, const intel_batch_t* bt, const float* intents,
                                  const float* d_weights, const float* d_ens, intel_tensors_t* G, float* d_intents_out,
                                  void* workspace, size_t workspace_bytes, intel_stream_t stream, int phases,
                                  const intel_row_maps_t* maps) {
    INTEL_TRY(check_dims(d));
    const intel_row_maps_t M = maps ? *maps : intel_row_maps_t{};
    INTEL_REQUIRE(phases > 0 && phases < 8, INTEL_ERR_ARG, "ensemble_bwd: phases must be a combination of INTEL_ENS_BWD_*");
    const bool do_head = phases & INTEL_ENS_BWD_HEAD, do_item = phases & INTEL_ENS_BWD_ITEM, do_score = phases & INTEL_ENS_BWD_SCORE;
    INTEL_REQUIRE(P && bt && intents && G && d_intents_out, INTEL_ERR_ARG, "ensemble_bwd: null argument");
    Arena a(workspace, workspace_bytes);
    EnsWs w;
    ens_layout(d, a, w);
    INTEL_REQUIRE(workspace && a.ok(), INTEL_ERR_WORKSPACE, "ensemble workspace too small: need %zu", a.off);
    cudaStream_t s = S(stream);
    const int64_t B = d->B, L = d->L, R = B * L, I = d->I;
    const int K = (int)d->K, di = d->d_iid + d->d_im, ds = d->d_s, du = d->d_u, dint = d->d_int;
    const int D = di + ds + du + dint, off_u = di + ds, off_h = di + ds + du;
    Stream ps[2], gs[2];
    streams_of(d, P, ps);
    streams_of(d, G, gs);

    if (d->cross_attention) {
        const float scale = 1.0f / sqrtf((float)d->qsize);
        if (do_head) {
        if (head_full_ok(K, D)) {
            INTEL_TRY(head_full_bwd(B, L, K, D, off_u, w.all, P->head_w, d_weights, d_ens, bt->scores, bt->session_len, w.dall,
                                    G->head_w, G->head_b, s));
        } else {
            INTEL_TRY(head_fuse_bwd(B, L, K, d_weights, d_ens, bt->scores, bt->session_len, w.dwv, w.dwp, s));
            INTEL_TRY(linear_dw(B, K, D, w.dwv, K, w.all, D, G->head_w, D, G->head_b, s));
            INTEL_TRY(linear_dw(B, K, du + dint, w.dwp, K, w.all + off_u, D, G->head_w + off_u, D, G->head_b, s));
            INTEL_TRY(linear_dx(B, K, D, w.dwv, K, P->head_w, D, w.dall, D, s));
            INTEL_TRY(linear_dx(B, K, du + dint, w.dwp, K, P->head_w + off_u, D, w.dall + off_u, D, s, 1));
        }
        // h_intent = relu(intent_embeddings(intent)): its gradient is the third column block of dcat
        const int dc = di + ds + dint;
        INTEL_TRY(relu_bwd(B, dint, w.dall + off_h, D, w.all + off_h, D, w.dcat + di + ds, dc, s));
        // h_u = relu(uid_embeddings[u])
        INTEL_TRY(scatter_add_rows(B, du, w.dall + off_u, D, bt->u_id, G->uid_emb, P->uid_emb, s, d->user_rows, M.uid));
        // the two pooled cross attentions
        for (int st = 0; st < 2; ++st) {
            const int dd = ps[st].d, off = ps[st].off;
            const float* X = w.stack[st].X[d->layers];
            const float *xk = ps[st].xk, *xv = ps[st].xv;
            if (cross_full_ok(dd, L) && al16(xk) && al16(xv)) {
                INTEL_TRY(cross_full_bwd(B, L, X, w.q[st], dc, w.qk[st], xk, xv, bt->session_len, scale, w.p[st], w.xbar[st],
                                         w.dall + off, D, w.dX[st], w.dcat + off, dc, gs[st].xk, gs[st].xv, s));
            } else {
                INTEL_TRY(linear_dw(B, dd, dd, w.dall + off, D, w.xbar[st], dd, gs[st].xv, dd, nullptr, s));
                INTEL_TRY(linear_dx(B, dd, dd, w.dall + off, D, xv, dd, w.dxbar, dd, s));
                INTEL_TRY(cross_pool_bwd(B, L, dd, X, w.qk[st], bt->session_len, scale, w.p[st], w.dxbar, w.dX[st], w.dqk, s));
                INTEL_TRY(linear_dw(B, dd, dd, w.q[st], dc, w.dqk, dd, gs[st].xk, dd, nullptr, s));      // dW_k[a,c] = sum q_a dqk_c
                INTEL_TRY(linear(B, dd, dd, w.dqk, dd, xk, dd, nullptr, w.dcat + off, dc, s));      // dq = W_k dqk -> its block of dcat
            }
        }
        // the three products against the predicted intents as one: d_intents = dcat Wcat, dWcat += dcat^T intents
        {
            const float* Wc = P->xq_item;
            if (!intent_weights_stacked(P, di, ds, I)) Wc = w.Wcat;   // stacked by the forward call
            INTEL_TRY(linear_dx(B, dc, I, w.dcat, dc, Wc, I, d_intents_out, I, s, 0));
            if (intent_weights_stacked(G, di, ds, I)) {
                INTEL_TRY(linear_dw(B, dc, I, w.dcat, dc, intents, I, G->xq_item, I, nullptr, s));
            } else {
                INTEL_TRY(linear_dw(B, di, I, w.dcat, dc, intents, I, G->xq_item, I, nullptr, s));
                INTEL_TRY(linear_dw(B, ds, I, w.dcat + di, dc, intents, I, G->xq_score, I, nullptr, s));
                INTEL_TRY(linear_dw(B, dint, I, w.dcat + di + ds, dc, intents, I, G->intent_w, I, nullptr, s));
            }
            INTEL_TRY(colsum(B, dint, w.dcat + di + ds, dc, G->intent_b, s));
        }
        }
    } else {
        const int q = d->qsize;
        if (do_head) {
        INTEL_TRY(item_fuse_bwd(R, K, d_weights, d_ens, bt->scores, w.g, s));
        INTEL_TRY(linear_dw(R, K, D, w.g, K, w.all_item, D, G->head_w, D, G->head_b, s));
        INTEL_TRY(linear_dx(R, K, D, w.g, K, P->head_w, D, w.dall_item, D, s));
        // h_intent / h_u broadcast over the list
        INTEL_TRY(bcast_rows_bwd(B, L, dint, w.dall_item + off_h, D, w.dvec, dint, 0, s));
        INTEL_TRY(relu_bwd(B, dint, w.dvec, dint, w.hint, dint, w.dvec, dint, s));
        INTEL_TRY(linear_dw(B, dint, I, w.dvec, dint, intents, I, G->intent_w, I, G->intent_b, s));
        INTEL_TRY(linear_dx(B, dint, I, w.dvec, dint, P->intent_w, I, d_intents_out, I, s, 0));
        INTEL_TRY(bcast_rows_bwd(B, L, du, w.dall_item + off_u, D, w.dvec, du, 0, s));
        INTEL_TRY(scatter_add_rows(B, du, w.dvec, du, bt->u_id, G->uid_emb, P->uid_emb, s, d->user_rows, M.uid));
        for (int st = 0; st < 2; ++st) {
            const int dd = ps[st].d;
            const float* t = w.t[st];
            INTEL_TRY(gate_bwd(B, L, dd, w.stack[st].X[d->layers], w.m[st], w.dall_item + ps[st].off, D, w.dX[st], w.dm, s));
            INTEL_TRY(linear_dw(B, dd, q, w.dm, dd, t, q, gs[st].w2, q, nullptr, s));
            INTEL_TRY(linear_dx(B, dd, q, w.dm, dd, ps[st].w2, q, w.dt, q, s, 0, t, q));       // relu mask (t = relu(.) > 0)
            INTEL_TRY(linear_dw(B, q, I, w.dt, q, intents, I, gs[st].w0, I, gs[st].b0, s));
            INTEL_TRY(linear_dx(B, q, I, w.dt, q, ps[st].w0, I, d_intents_out, I, s, 1));
        }
        }
    }
    // the self-attention stacks (IntEL.py:182-197) and what feeds them: phase ITEM, then phase SCORE
    const bool do_stream[2] = {do_item, do_score};
    for (int st = 0; st < 2; ++st) {
        if (!do_stream[st]) continue;
        // run on its own, the score phase is the one a caller overlaps with its gradient exchange: leave the reserved SMs free
        const bool reserve = st == 1 && phases == INTEL_ENS_BWD_SCORE;
        if (reserve) trunk_reserve_apply(true);
        const int r = stack_bwd(B, L, ps[st].d, d->heads, d->layers, *ps[st].stack, *gs[st].stack, w.stack[st], w.dX[st], w.t1, w.t2,
                                w.dqkv, d->dropout_p, d->dropout_seed, st, s);
        if (reserve) trunk_reserve_apply(false);
        INTEL_TRY(r);
        if (st == 0) {           // item id / class embedding rows
            INTEL_TRY(scatter_add_rows(R, d->d_iid, w.dX[0], di, bt->i_id, G->iid_emb, nullptr, s, d->item_rows, M.iid));
            if (d->d_im > 0)
                INTEL_TRY(scatter_add_rows(R, d->d_im, w.dX[0] + d->d_iid, di, bt->i_class, G->item_emb, nullptr, s, d->class_rows, M.item));
        } else {                 // score_embeddings
            if (score_embed_bwd_ok(K, ds)) INTEL_TRY(score_embed_bwd(R, K, ds, w.dX[1], ds, w.xs, G->score_w, G->score_b, s));
            else INTEL_TRY(linear_dw(R, ds, K, w.dX[1], ds, w.xs, K, G->score_w, K, G->score_b, s));
        }
    }
    return INTEL_OK;
}

int intel_ensemble_bwd_phase(const intel_dims_t* d, const intel_tensors_t* P, const intel_batch_t* bt, const float* intents,
                             const float* d_weights, const float* d_ens, intel_tensors_t* G, float* d_intents_out,
                             void* workspace, size_t workspace_bytes, intel_stream_t stream, int phases) {
    return intel_ensemble_bwd_phase_rows(d, P, bt, intents, d_weights, d_ens, G, d_intents_out, workspace, workspace_bytes, stream,
                                         phases, nullptr);
}

int intel_ensemble_bwd(const intel_dims_t* d, const intel_tensors_t* P, const intel_batch_t* bt, const float* intents,
                       const float* d_weights, const float* d_ens, intel_tensors_t* G, float* d_intents_out,
                       void* workspace, size_t workspace_bytes, intel_stream_t stream) {
    return intel_ensemble_bwd_phase(d, P, bt, intents, d_weights, d_ens, G, d_intents_out, workspace, workspace_bytes, stream,
                                    INTEL_ENS_BWD_HEAD | INTEL_ENS_BWD_ITEM | INTEL_ENS_BWD_SCORE);
}


// ================================================================================================
size_t intel_intent_workspace_bytes(const intel_dims_t* d) {
    if (check_dims(d) != INTEL_OK) return 0;
    Arena a(nullptr, 0);
    IntWs w;
    int_layout(d, a, w);
    return a.off + 256;
}

int intel_intent_fwd(const intel_dims_t* d, const intel_tensors_t* P, const intel_batch_t* bt, float* intents_out,
                     void* workspace, size_t workspace_bytes, intel_stream_t stream) {
    INTEL_TRY(check_dims(d));
    INTEL_REQUIRE(P && bt && intents_out, INTEL_ERR_ARG, "intent_fwd: null argument");
    INTEL_REQUIRE(d->H1 > 0 && d->H2 > 0, INTEL_ERR_ARG, "empty history tensors");
    Arena a(workspace, workspace_bytes);
    IntWs w;
    int_layout(d, a, w);
    INTEL_REQUIRE(workspace && a.ok(), INTEL_ERR_WORKSPACE, "intent workspace too small: need %zu", a.off);
    cudaStream_t s = S(stream);
    const int64_t B = d->B, I = d->I;
    const int dint = d->d_int, dctx = d->d_ctx, du = d->d_u;
    const int Dp = dctx + dint + d->d_iid + dint + dctx + du;
    History hs[2];
    histories_of(d, P, nullptr, nullptr, bt, hs);

    INTEL_TRY(transpose(dint, I, P->intent_w, w.Wt, 0, s));
    // history tokens: [context embedding | intent embedding of the dense history intents] of the session history,
    // [item id embedding | intent embedding of the one-hot item intents] of the item history
    for (int i = 0; i < 2; ++i) {
        const History& h = hs[i];
        EncWs& e = w.e[i];
        const int64_t R = B * e.T;
        INTEL_TRY(gather_rows(R, h.dtok, h.table, h.ids, e.seq, e.d, 0, s, h.table_rows));
        if (h.idx) {
            INTEL_TRY(sparse_rows_linear_fwd(R, h.nz, dint, h.idx, h.val, w.Wt, P->intent_b, e.seq + h.dtok, e.d, s));
        } else {
            INTEL_REQUIRE(h.dense, INTEL_ERR_ARG, "%s is null", h.dense_name);
            INTEL_TRY(dense_rows_linear_fwd(R, I, dint, h.dense, w.Wt, P->intent_b, e.seq + h.dtok, e.d, e.nz_idx, e.nz_val, e.nz_cnt,
                                            NZ_CAP, s, e.T, h.lens));
        }
    }
    if (d->encoder == INTEL_ENCODER_BERT4REC) {
        for (int i = 0; i < 2; ++i) INTEL_TRY(bert_fwd(d, *hs[i].p, w.e[i], hs[i].lens, w.feat + hs[i].off, Dp, s));
    } else {
        INTEL_TRY(gru_fwd_pair(d, hs, w.e, w.feat, Dp, s));
    }
    INTEL_TRY(gather_rows(B, dctx, P->ctx_emb, bt->context_mh, w.feat, Dp, 0, s, d->ctx_rows));
    INTEL_TRY(gather_rows(B, du, P->uid_emb, bt->u_id, w.feat + dctx, Dp, 0, s, d->user_rows));
    INTEL_TRY(linear(B, I, Dp, w.feat, Dp, P->pred_w, Dp, P->pred_b, w.logits, pad4(I), s));
    return softmax_rows(B, I, w.logits, intents_out, s, pad4(I));
}

int intel_intent_bwd_rows(const intel_dims_t* d, const intel_tensors_t* P, const intel_batch_t* bt, const float* intents,
                          const float* d_intents, const float* d_intents_extra, intel_tensors_t* G, void* workspace,
                          size_t workspace_bytes, intel_stream_t stream, const intel_row_maps_t* maps) {
    INTEL_TRY(check_dims(d));
    const intel_row_maps_t M = maps ? *maps : intel_row_maps_t{};
    INTEL_REQUIRE(P && bt && intents && d_intents && G, INTEL_ERR_ARG, "intent_bwd: null argument");
    Arena a(workspace, workspace_bytes);
    IntWs w;
    int_layout(d, a, w);
    INTEL_REQUIRE(workspace && a.ok(), INTEL_ERR_WORKSPACE, "intent workspace too small: need %zu", a.off);
    cudaStream_t s = S(stream);
    const int64_t B = d->B, I = d->I;
    const int dint = d->d_int, dctx = d->d_ctx, du = d->d_u;
    const int Dp = dctx + dint + d->d_iid + dint + dctx + du;
    History hs[2];
    histories_of(d, P, G, &M, bt, hs);

    INTEL_TRY(softmax_rows_bwd(B, I, intents, d_intents, d_intents_extra, w.dlogits, s, pad4(I)));
    INTEL_TRY(linear_dw(B, I, Dp, w.dlogits, pad4(I), w.feat, Dp, G->pred_w, Dp, G->pred_b, s));
    INTEL_TRY(linear_dx(B, I, Dp, w.dlogits, pad4(I), P->pred_w, Dp, w.dfeat, Dp, s));
    INTEL_TRY(scatter_add_rows(B, dctx, w.dfeat, Dp, bt->context_mh, G->ctx_emb, nullptr, s, d->ctx_rows, M.ctx));
    INTEL_TRY(scatter_add_rows(B, du, w.dfeat + dctx, Dp, bt->u_id, G->uid_emb, nullptr, s, d->user_rows, M.uid));
    if (d->encoder == INTEL_ENCODER_BERT4REC) {
        for (int i = 0; i < 2; ++i)
            INTEL_TRY(bert_bwd(d, *hs[i].p, *hs[i].g, w.e[i], hs[i].lens, w.dfeat + hs[i].off, Dp, w.t1, w.t2, w.dqkv, s));
    } else {
        const int h = d->gru_hidden;
        if (gru_outproj_pair_ok(w.e[0].d, w.e[1].d)) {      // d(last state) of both encoders in one launch
            const int n[2] = {w.e[0].d, w.e[1].d};
            const float* W[2] = {hs[0].p->w_out, hs[1].p->w_out};
            const float* dv[2] = {w.dfeat + hs[0].off, w.dfeat + hs[1].off};
            float* dh[2] = {w.e[0].gru.dh, w.e[1].gru.dh};
            const int64_t ldd[2] = {Dp, Dp}, ldh[2] = {h, h};
            INTEL_TRY(gru_outproj_pair_dx(B, n, W, dv, ldd, dh, ldh, s));
        } else {
            for (int i = 0; i < 2; ++i)
                INTEL_TRY(linear_dx(B, w.e[i].d, h, w.dfeat + hs[i].off, Dp, hs[i].p->w_out, h, w.e[i].gru.dh, h, s));
        }
        INTEL_TRY(gru_bwd_pair(d, hs, w.e, w.dfeat, Dp, s));
    }
    INTEL_TRY(fill_zero(w.dWt, (size_t)I * dint * 4, s));
    for (int i = 0; i < 2; ++i) {
        const History& h = hs[i];
        const EncWs& e = w.e[i];
        const int64_t R = B * e.T;
        INTEL_TRY(scatter_add_rows(R, h.dtok, e.dseq, e.d, h.ids, h.gtable, nullptr, s, h.table_rows, h.map));
        // the intent part, with the bias gradient (column sums)
        if (h.idx) {
            INTEL_TRY(dense_rows_linear_bwd(R, I, dint, nullptr, e.dseq + h.dtok, e.d, h.idx, h.val, nullptr, h.nz, w.dWt, s, G->intent_b));
        } else {
            INTEL_TRY(dense_rows_linear_bwd(R, I, dint, h.dense, e.dseq + h.dtok, e.d, e.nz_idx, e.nz_val, e.nz_cnt, NZ_CAP, w.dWt, s,
                                            G->intent_b));
        }
    }
    return transpose(I, dint, w.dWt, G->intent_w, 1, s);
}

int intel_intent_bwd(const intel_dims_t* d, const intel_tensors_t* P, const intel_batch_t* bt, const float* intents,
                     const float* d_intents, const float* d_intents_extra, intel_tensors_t* G, void* workspace,
                     size_t workspace_bytes, intel_stream_t stream) {
    return intel_intent_bwd_rows(d, P, bt, intents, d_intents, d_intents_extra, G, workspace, workspace_bytes, stream, nullptr);
}

}  // extern "C"
